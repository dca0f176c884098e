"""GPU tests of the verifiers that name the bad items: verify_cell_kzg_proof_batch_groups (a verdict per caller-defined group
of openings) and verify_blob_kzg_proof_batch_items (a verdict per blob).  Verdicts: 0 verifies, 1 does not, 2 malformed.
Every verdict is checked against the plain batch call on the same items."""
import importlib
import random
import threading

import pytest

from tests import vectors

pytestmark = pytest.mark.gpu


def _cases(fn):
    return [pytest.param(n, i, o, id=n) for n, i, o in vectors.load(fn)]


def _plain(pkg, f, *a):
    try:
        return f(*a)
    except pkg.KzgError:
        return None


def _sizes_ok(items, size):
    return all(len(x) == size for x in items)


def _flip(cell, byte=31):
    """a canonical cell that differs from `cell` (the low bit of a big-endian element)"""
    return cell[:byte] + bytes([cell[byte] ^ 1]) + cell[byte + 1:]


def _sub(seq, idx):
    return [seq[i] for i in idx]


def _members(groups, n_groups):
    m = [[] for _ in range(n_groups)]
    for k, g in enumerate(groups):
        m[g].append(k)
    return m


def _row_groups(commitments):
    first = {}
    return [first.setdefault(bytes(c), len(first)) for c in commitments]


def _check_against_plain(ctx, pkg, C, I, CL, PR, groups, st, which=None):
    """every group that is not malformed has the verdict of the plain call on its openings (an empty group: 0)"""
    members = _members(groups, len(st))
    for g in (range(len(st)) if which is None else which):
        if st[g] == 2:
            continue
        idx = members[g]
        want = _plain(pkg, ctx.verify_cell_kzg_proof_batch, _sub(C, idx), _sub(I, idx), _sub(CL, idx), _sub(PR, idx)) if idx else True
        assert want is not None, g
        assert st[g] == (0 if want else 1), g


@pytest.mark.parametrize("name,inp,expected", _cases("verify_cell_kzg_proof_batch"))
def test_cell_vectors_grouped(vec_ctx, pkg, name, inp, expected):
    """every consensus vector as one group, as one group per opening and with groups = commitment rows"""
    C, I, CL, PR = inp["commitments"], inp["cell_indices"], inp["cells"], inp["proofs"]
    n = len(C)
    structural = not (n == len(I) == len(CL) == len(PR)) or not (_sizes_ok(C, 48) and _sizes_ok(PR, 48) and _sizes_ok(CL, 2048))
    if structural:
        with pytest.raises(pkg.KzgError):
            vec_ctx.verify_cell_kzg_proof_batch_groups(C, I, CL, PR, [0] * n, n_groups=1)
        return
    for groups in ([0] * n, list(range(n)), _row_groups(C)):
        ok, st = vec_ctx.verify_cell_kzg_proof_batch_groups(C, I, CL, PR, groups)
        assert len(st) == (max(groups) + 1 if groups else 0)
        if expected is True:
            assert ok and st == [0] * len(st)
        elif expected is False:
            assert not ok and 2 not in st and 1 in st
        else:
            assert not ok and 2 in st
            _check_against_plain(vec_ctx, pkg, C, I, CL, PR, groups, st)


@pytest.mark.parametrize("name,inp,expected", _cases("verify_blob_kzg_proof_batch"))
def test_blob_vectors_items(vec_ctx, pkg, name, inp, expected):
    B, C, P = inp["blobs"], inp["commitments"], inp["proofs"]
    if not (len(B) == len(C) == len(P)) or not (_sizes_ok(B, 131072) and _sizes_ok(C, 48) and _sizes_ok(P, 48)):
        with pytest.raises(pkg.KzgError):
            vec_ctx.verify_blob_kzg_proof_batch_items(B, C, P)
        return
    ok, st = vec_ctx.verify_blob_kzg_proof_batch_items(B, C, P)
    assert len(st) == len(B)
    if expected is True:
        assert ok and st == [0] * len(B)
    elif expected is False:
        assert not ok and 2 not in st and 1 in st
    else:
        assert not ok and 2 in st
    for i, s in enumerate(st):
        if s != 2:
            want = vec_ctx.verify_blob_kzg_proof_batch([B[i]], [C[i]], [P[i]])
            assert s == (0 if want else 1), i


def _openings(ctx, nb, first):
    syn = importlib.import_module("eth_kzg_b200.synthetic")
    flat = b"".join(syn.blob(first + i) for i in range(nb))
    cms, st = ctx.blob_to_kzg_commitment_batch(flat, nb)
    cells, proofs, st2 = ctx.compute_cells_and_kzg_proofs_batch(flat, nb)
    assert not any(st) and not any(st2)
    C = [cms[48 * (k // 128):48 * (k // 128) + 48] for k in range(nb * 128)]
    I = [k % 128 for k in range(nb * 128)]
    CL = [cells[k * 2048:(k + 1) * 2048] for k in range(nb * 128)]
    PR = [proofs[k * 48:(k + 1) * 48] for k in range(nb * 128)]
    return C, I, CL, PR


@pytest.fixture(scope="module")
def full(das_ctx):
    return _openings(das_ctx, 128, 8100)


def test_config5_groups_agree_with_plain(das_ctx, pkg, full):
    """128 x 128 openings, groups = columns: honest data, one flipped cell byte, two swapped proofs, one whole column replaced
    by the column of other blobs.  all_ok equals the plain call; every flagged group and 8 clean ones agree with the plain call
    on the group's openings; the oracle agrees on the 128-opening slice that holds a corruption."""
    from oracle import cref
    C, I, CL, PR = full
    groups = list(I)
    ok, st = das_ctx.verify_cell_kzg_proof_batch_groups(C, I, CL, PR, groups)
    assert ok and st == [0] * 128 and das_ctx.verify_cell_kzg_proof_batch(C, I, CL, PR) is True

    bad_cell = list(CL)
    bad_cell[5000] = _flip(CL[5000])
    bad_proof = list(PR)
    bad_proof[300], bad_proof[301] = PR[301], PR[300]
    col = 77   # every blob's cell and proof of column 77 replaced by the next blob's
    bad_col_cells, bad_col_proofs = list(CL), list(PR)
    for b in range(128):
        k, src = b * 128 + col, ((b + 1) % 128) * 128 + col
        bad_col_cells[k], bad_col_proofs[k] = CL[src], PR[src]
    for cells, proofs, bad_k in ((bad_cell, PR, 5000), (CL, bad_proof, 300), (bad_col_cells, bad_col_proofs, col)):
        ok, st = das_ctx.verify_cell_kzg_proof_batch_groups(C, I, cells, proofs, groups)
        assert ok is das_ctx.verify_cell_kzg_proof_batch(C, I, cells, proofs) is False
        flagged = [g for g in range(128) if st[g]]
        assert flagged and 2 not in st
        clean = [g for g in range(128) if not st[g]][::15][:8]
        _check_against_plain(das_ctx, pkg, C, I, cells, proofs, groups, st, which=flagged + clean)
        assert I[bad_k] in flagged
        lo = bad_k - bad_k % 128
        sl = slice(lo, lo + 128)
        assert cref.verify_cell_kzg_proof_batch(C[sl], I[sl], cells[sl], proofs[sl]) is False
    ok, st = das_ctx.verify_cell_kzg_proof_batch_groups(C, I, bad_col_cells, bad_col_proofs, groups)
    assert [g for g in range(128) if st[g]] == [col]
    # uneven groups: all 16 384 openings in one group next to 16 383 empty ones
    ok, st = das_ctx.verify_cell_kzg_proof_batch_groups(C, I, bad_cell, PR, [0] * len(C), n_groups=16384)
    assert not ok and st == [1] + [0] * 16383


def _localise(ctx, nb, first, group_size, seed):
    """one flipped cell in each of 16 random groups of `group_size` consecutive openings: exactly those groups are 1"""
    C, I, CL, PR = _openings(ctx, nb, first)
    rng = random.Random(seed)
    n_groups = len(C) // group_size
    groups = [k // group_size for k in range(len(C))]
    bad = [g * group_size + rng.randrange(group_size) for g in rng.sample(range(n_groups), min(16, n_groups))]
    cells = list(CL)
    for k in bad:
        cells[k] = _flip(cells[k], 32 * rng.randrange(64) + 31)
    ok, st = ctx.verify_cell_kzg_proof_batch_groups(C, I, cells, PR, groups)
    assert not ok
    assert sorted(g for g, s in enumerate(st) if s) == sorted(groups[k] for k in bad)
    assert set(st) <= {0, 1}


def test_exact_localisation_per_opening(das_ctx):
    _localise(das_ctx, 16, 8300, 1, 1)


def test_exact_localisation_rows_above_32768(das_ctx):
    """264 blobs x 128 = 33 792 openings: the aggregate takes the per-column sums there"""
    _localise(das_ctx, 264, 8400, 128, 2)


def test_exact_localisation_bucket_msm(das_ctx, monkeypatch):
    monkeypatch.setenv("EKZG_VERIFY_MSM", "bucket")
    _localise(das_ctx, 16, 8300, 1, 3)
    _localise(das_ctx, 40, 8700, 512, 4)   # groups of four rows: a CTA per group


def _invalid_proofs():
    return [i["proofs"][0] for n, i, o in vectors.load("verify_cell_kzg_proof_batch") if "_invalid_proof_" in n and len(i["proofs"][0]) == 48]


def test_malformed_items_do_not_sink_the_batch(das_ctx, pkg):
    """groups = rows of 16 blobs: an invalid proof (row 1), a non-canonical cell (row 3), a cell index of 128 (row 5), an
    invalid commitment for all of row 7 and one ordinary bad cell (row 9).  Rows 1, 3, 5, 7 are 2, row 9 is 1, the rest 0;
    the plain call still fails with Err.  The same with one group per opening names exactly those openings."""
    C, I, CL, PR = _openings(das_ctx, 16, 8900)
    C, I, CL, PR = list(C), list(I), list(CL), list(PR)
    PR[1 * 128 + 4] = _invalid_proofs()[0]
    CL[3 * 128 + 9] = b"\xff" * 32 + CL[3 * 128 + 9][32:]
    I[5 * 128 + 2] = 128
    for k in range(7 * 128, 8 * 128):
        C[k] = bytes(48)   # no compression flag: not a valid encoding
    CL[9 * 128 + 100] = _flip(CL[9 * 128 + 100])
    groups = [k // 128 for k in range(len(C))]
    ok, st = das_ctx.verify_cell_kzg_proof_batch_groups(C, I, CL, PR, groups)
    assert not ok
    assert st == [2 if g in (1, 3, 5, 7) else 1 if g == 9 else 0 for g in range(16)]
    with pytest.raises(pkg.KzgError):
        das_ctx.verify_cell_kzg_proof_batch(C, I, CL, PR)
    ok, st = das_ctx.verify_cell_kzg_proof_batch_groups(C, I, CL, PR, list(range(len(C))))
    want = [0] * len(C)
    for k in (1 * 128 + 4, 3 * 128 + 9, 5 * 128 + 2, *range(7 * 128, 8 * 128)):
        want[k] = 2
    want[9 * 128 + 100] = 1
    assert not ok and st == want
    # without the ordinary bad cell every well-formed group verifies
    CL[9 * 128 + 100] = _flip(CL[9 * 128 + 100])
    ok, st = das_ctx.verify_cell_kzg_proof_batch_groups(C, I, CL, PR, groups)
    assert not ok and st == [2 if g in (1, 3, 5, 7) else 0 for g in range(16)]


def test_structural_errors(das_ctx, pkg):
    C, I, CL, PR = _openings(das_ctx, 1, 9100)
    groups = [k % 4 for k in range(128)]
    with pytest.raises(pkg.KzgError):
        das_ctx.verify_cell_kzg_proof_batch_groups(C, I[:-1], CL, PR, groups)
    with pytest.raises(pkg.KzgError):
        das_ctx.verify_cell_kzg_proof_batch_groups(C, I, CL, PR, groups[:-1])
    with pytest.raises(pkg.KzgError):
        das_ctx.verify_cell_kzg_proof_batch_groups(C, I, CL, PR, groups, n_groups=3)
    with pytest.raises(pkg.KzgError):
        das_ctx.verify_cell_kzg_proof_batch_groups(C, I, CL, PR, groups, n_groups=(1 << 20) + 1)
    with pytest.raises(pkg.KzgError):
        das_ctx.verify_blob_kzg_proof_batch_items([bytes(131072)], [], [])
    assert das_ctx.verify_cell_kzg_proof_batch_groups([], [], [], [], [], n_groups=3) == (True, [0, 0, 0])
    assert das_ctx.verify_cell_kzg_proof_batch_groups([], [], [], [], []) == (True, [])
    assert das_ctx.verify_blob_kzg_proof_batch_items([], [], []) == (True, [])
    # the largest group count is accepted; the groups without openings are 0
    ok, st = das_ctx.verify_cell_kzg_proof_batch_groups(C, I, CL, PR, groups, n_groups=1 << 20)
    assert ok and len(st) == 1 << 20 and not any(st)


@pytest.mark.parametrize("chunk,nb", [(None, 9), ("4", 9), (None, 20), ("4", 20)],
                         ids=["host_challenges", "host_challenges_chunks_of_4", "device_challenges", "device_challenges_chunks_of_4"])
def test_blob_items(das_ctx, pkg, chunk, nb, monkeypatch):
    if chunk:
        monkeypatch.setenv("EKZG_CHUNK", chunk)
    syn = importlib.import_module("eth_kzg_b200.synthetic")
    blobs = [syn.blob(9200 + i) for i in range(nb)]
    flat = b"".join(blobs)
    cms, _ = das_ctx.blob_to_kzg_commitment_batch(flat, nb)
    prs, _ = das_ctx.compute_blob_kzg_proof_batch(flat, cms, nb)
    cl = [cms[48 * i:48 * i + 48] for i in range(nb)]
    pl = [prs[48 * i:48 * i + 48] for i in range(nb)]
    assert das_ctx.verify_blob_kzg_proof_batch_items(blobs, cl, pl) == (True, [0] * nb)
    swapped = list(pl)
    swapped[4], swapped[5] = pl[5], pl[4]
    ok, st = das_ctx.verify_blob_kzg_proof_batch_items(blobs, cl, swapped)
    assert ok is das_ctx.verify_blob_kzg_proof_batch(blobs, cl, swapped) is False
    assert st == [1 if i in (4, 5) else 0 for i in range(nb)]
    nc = list(blobs)
    nc[2] = b"\xff" * 32 + blobs[2][32:]
    ok, st = das_ctx.verify_blob_kzg_proof_batch_items(nc, cl, swapped)
    assert not ok and st == [2 if i == 2 else 1 if i in (4, 5) else 0 for i in range(nb)]
    badc = list(cl)
    badc[nb - 1] = bytes(48)
    ok, st = das_ctx.verify_blob_kzg_proof_batch_items(blobs, badc, pl)
    assert not ok and st == [2 if i == nb - 1 else 0 for i in range(nb)]


def test_concurrent_grouped_callers(das_ctx):
    """8 host threads at once, each with a bad cell in a different row, each gets its own verdicts"""
    C, I, CL, PR = _openings(das_ctx, 16, 9300)
    groups = [k // 128 for k in range(len(C))]
    out = [None] * 8

    def worker(t):
        cells = list(CL)
        k = (2 * t) * 128 + 11 * t
        cells[k] = _flip(cells[k])
        out[t] = das_ctx.verify_cell_kzg_proof_batch_groups(C, I, cells, PR, groups)

    th = [threading.Thread(target=worker, args=(t,)) for t in range(8)]
    for x in th:
        x.start()
    for x in th:
        x.join()
    for t in range(8):
        assert out[t] == (False, [1 if g == 2 * t else 0 for g in range(16)]), t
