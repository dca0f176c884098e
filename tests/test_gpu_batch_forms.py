"""GPU tests of the kernel forms that only large or ragged batches select.  Every batch entry point picks its kernels by batch
size (launch_fixed_msm: wide / 16-slice / one-point-per-thread; launch_sum_positions: tree / linear; launch_g1_compress: batched
inversion or not; launch_g1_ntt_phases: cooperative radix-4 / radix-4 / register form; the FK20 piece split; host or device blob
challenges).  Each case below
  - proves with torch.profiler that the form it targets ran and the form on the other side of the threshold did not,
  - puts blobs with chosen polynomial coefficients (monomials, low-degree polynomials, Booth-digit edges of every window width the
    contexts use) and the edge blobs at the positions where the work is split,
  - compares every item with the single-item entry point and a sample of at least 64 items (all boundary and chosen-coefficient
    blobs among them) with the C oracle.  Byte equality throughout: this is integer arithmetic."""
import concurrent.futures
import hashlib
import importlib
import json
import os
import random
import tempfile

import pytest

from oracle import pyref

R = pyref.R
BLOB = 131072
IDENTITY = b"\xc0" + bytes(47)


# ---------------------------------------------------------------- helpers
def launched(fn):
    """names of the kernels one call of fn launches (torch.profiler, as tools/launch_sequence.py records them)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            names = [e["name"] for e in json.load(f)["traceEvents"] if e.get("cat") == "kernel"]
    assert names, "the profiler recorded no kernel launches"
    return names


def count(names, form):
    return sum(form in n for n in names)


def assert_forms(names, want):
    """want: {form: expected launch count, or True for 'at least one'}; a form with 0 must not have run"""
    got = {f: count(names, f) for f in want}
    bad = {f: (got[f], w) for f, w in want.items() if (got[f] == 0 if w is True else got[f] != w)}
    assert not bad, "kernel forms (launched, expected): %r; kernels: %r" % (bad, sorted(set(names)))


MSM_FORMS = ("k_fk20_msm_vm<4>", "k_fk20_msm_vm<16>", "k_fk20_msm_vm<64>")
SUM_FORMS = ("k_sum_positions(", "k_sum_positions_tree(")
COMPRESS_FORMS = ("k_g1_compress(", "k_g1_compress_batched(")
NTT_FORMS = ("k_fk20_g1_ntts<", "k_fk20_g1_ntts_r4<32>", "k_fk20_g1_ntts_r4<8>")


def merge_group(w):
    """points per merged top-window lookup of a table of window w (MsmTable::set_window)"""
    nw = 255 // w + 1
    rtop = (1 << (255 - w * (nw - 1))) + 1
    for m in (4, 2):
        if rtop ** m - 1 <= 1 << (w - 1):
            return m
    return 1


def msm_form(B, cnt, ngroups, w):
    """the launch_fixed_msm form for blobs [b0, b0 + cnt) of a batch of B: wide by the whole batch, tiny by the piece"""
    mg = merge_group(w)
    if B * ngroups >= 512 * 128:
        return "k_fk20_msm_vm<4>"
    if mg <= 4 and cnt * ngroups <= (8 * 64 if mg == 1 else 16 * 128):
        return "k_fk20_msm_vm<64>"
    return "k_fk20_msm_vm<16>"


def fk20_pieces(n):
    """(offset, length) of the FK20 pieces of one chunk (compute_cells_and_kzg_proofs_batch)"""
    q = (n // 4 + 31) & ~31 if n >= 512 else n
    return [(0, q)] + ([(q, n - q)] if q < n else [])


def blob_from_coeffs(c):
    """the blob (evaluations in bit-reversed order, big-endian) of the polynomial with coefficients c: the inverse of
    pyref.blob_to_coeffs"""
    return b"".join((x % R).to_bytes(32, "big") for x in pyref.brp(pyref.ntt([x % R for x in c])))


def booth_carry_scalar(w):
    """every w-bit window 2^(w-1), so that every signed digit carries; the windows that keep it below r"""
    s = 0
    for k in range(256 // w + 1):
        t = s | (1 << (w - 1)) << (k * w)
        if t >= R:
            break
        s = t
    return s


def chosen_coeffs(widths):
    """coefficient vectors that put the commitment MSM (whose scalars are the coefficients) at its edges"""
    rng = random.Random(4096)
    out = []
    for d in (0, 1, 63, 64, 4095):   # one SRS point: one non-identity partial sum out of 64
        c = [0] * 4096
        c[d] = 1
        out.append(c)
    out.append([rng.randrange(R) for _ in range(64)] + [0] * 4032)   # every cell proof is the identity, 63 of 64 partial sums too
    c = [rng.randrange(R) for _ in range(4096)]
    c[64:128] = [0] * 64                                             # one identity partial sum mid-chain
    out.append(c)
    out.append([R - 1] * 4096)                                       # the largest top-window digit
    for w in widths:
        s = booth_carry_scalar(w)
        out += [[s] * 4096, [s + 1] * 4096, [s - 1] * 4096]
    return out


_SPECIALS = {}


def special_blobs(ctx):
    """the chosen-coefficient blobs for the window widths of ctx (and of the default layouts), then the edge blobs"""
    widths = tuple(sorted({8, 13, 14, ctx.window, ctx.srs_window}))
    if widths not in _SPECIALS:
        syn = importlib.import_module("eth_kzg_b200.synthetic")
        _SPECIALS[widths] = [blob_from_coeffs(c) for c in chosen_coeffs(widths)] + list(syn.edge_blobs())
    return _SPECIALS[widths]


_RANDOM = []


def random_blob(i):
    """blob i of one seeded sequence: the same blob at the same position in every case, so that references are reused"""
    import numpy as np
    if not _RANDOM:
        a = np.random.default_rng(0xB200).integers(0, 256, size=(1100, 4096, 32), dtype=np.uint8)
        a[:, :, 0] &= 0x3F
        _RANDOM.append(a)
    return _RANDOM[0][i].tobytes()


def case_rounds(n, specials, boundaries):
    """batches of n distinct blobs that together hold every special blob: in each, the specials sit at the boundary positions
    first, then spread over the batch; the other positions hold random blobs.  -> [(blobs, special positions)]"""
    bset = sorted({p for p in boundaries if 0 <= p < n} | {0, n - 1})
    per = min(len(specials), n - n // 4)
    others = [p for p in range(n) if p not in bset]
    spread = others[::max(1, len(others) // max(1, per - len(bset)))] if per > len(bset) else []
    pos = (bset + spread)[:per]
    rot = n % len(specials)
    order = specials[rot:] + specials[:rot]
    # the zero blob goes last, off the boundaries: its outputs (zero cells, identity proofs) are what an item the kernels
    # skipped reads from zeroed memory
    order = [b for b in order if b != bytes(BLOB)] + [b for b in order if b == bytes(BLOB)]
    rounds = []
    for r in range(0, len(order), per):
        blobs = [random_blob(i) for i in range(n)]
        for p, b in zip(pos, order[r:r + per]):
            blobs[p] = b
        rounds.append((blobs, pos[:len(order[r:r + per])]))
    return rounds


_ORDER = random.Random(7).sample(range(2048), 2048)


def sample_positions(n, must):
    """the positions checked against the oracle: `must`, and the first 64 of one fixed random order that fall below n"""
    return sorted(set(p for p in must if 0 <= p < n) | set([p for p in _ORDER if p < n][:64]))


def key(b):
    return hashlib.sha256(b).digest()


_ORACLE = {}


def oracle_all(kind, items):
    """oracle results for [(cache key, thunk)], in parallel: ctypes releases the GIL, one call takes ~0.15-0.45 s of one core"""
    from oracle import cref
    cref.lib()
    todo = {k: f for k, f in items if (kind, k) not in _ORACLE}
    with concurrent.futures.ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        for k, v in zip(todo, ex.map(lambda f: f(), todo.values())):
            _ORACLE[kind, k] = v
    return [_ORACLE[kind, k] for k, _ in items]


_SINGLE = {}


def single(ctx, kind, b, fn):
    """the single-item entry point's result for input b, once per table layout"""
    k = (ctx.window, ctx.srs_window, kind, key(b))
    if k not in _SINGLE:
        _SINGLE[k] = fn()
    return _SINGLE[k]


# ---------------------------------------------------------------- CPU self-check
def test_blob_from_coeffs_self_check():
    """blob_from_coeffs inverts pyref.blob_to_coeffs on every chosen coefficient vector, and the oracle commits to X^0 as the
    G1 generator"""
    from oracle import cref
    cs = chosen_coeffs((8, 13, 14))
    for c in cs:
        assert pyref.blob_to_coeffs(blob_from_coeffs(c)) == c
    for w in (8, 13, 14):
        s = booth_carry_scalar(w)
        assert s < R and all((s >> (k * w)) & ((1 << w) - 1) == 1 << (w - 1) for k in range(s.bit_length() // w))
    assert cref.blob_to_kzg_commitment(blob_from_coeffs(cs[0])) == pyref.g1_compress(pyref.G1_GEN)


# ---------------------------------------------------------------- EIP-4844 provers
def check_4844_round(ctx, blobs, must, n):
    """commitments and blob proofs of one batch against the single-item calls (every item) and the oracle (sampled)"""
    from oracle import cref
    flat = b"".join(blobs)
    res = {}
    names_c = launched(lambda: res.setdefault("c", ctx.blob_to_kzg_commitment_batch(flat, n)))
    cms, st = res["c"]
    assert st == [0] * n
    names_p = launched(lambda: res.setdefault("p", ctx.compute_blob_kzg_proof_batch(flat, cms, n)))
    prs, st = res["p"]
    assert st == [0] * n
    for i, b in enumerate(blobs):
        c1 = single(ctx, "commitment", b, lambda: ctx.blob_to_kzg_commitment(b))
        assert cms[48 * i:48 * i + 48] == c1, "commitment %d differs from the single-blob call" % i
        p1 = single(ctx, "blob_proof", b, lambda: ctx.compute_blob_kzg_proof(b, c1))
        assert prs[48 * i:48 * i + 48] == p1, "blob proof %d differs from the single-blob call" % i
    pos = sample_positions(n, must)
    oc = oracle_all("commitment", [(key(blobs[i]), lambda b=blobs[i]: cref.blob_to_kzg_commitment(b)) for i in pos])
    for i, c in zip(pos, oc):
        assert cms[48 * i:48 * i + 48] == c, "commitment %d differs from the oracle" % i
    op = oracle_all("blob_proof", [(key(blobs[i]), lambda b=blobs[i], c=c: cref.compute_blob_kzg_proof(b, c)) for i, c in zip(pos, oc)])
    for i, p in zip(pos, op):
        assert prs[48 * i:48 * i + 48] == p, "blob proof %d differs from the oracle" % i
    return names_c, names_p


@pytest.mark.gpu
@pytest.mark.parametrize("n,chunk", [(8, None), (9, None), (16, None), (17, None), (256, None), (257, None), (1024, None),
                                     (1031, None), (1100, 2048)])
def test_4844_provers(vec_ctx, n, chunk, monkeypatch):
    """blob_to_kzg_commitment_batch and compute_blob_kzg_proof_batch across the MSM, tree-sum and challenge thresholds.  1031
    is two chunks (wide, then tiny, in one call); 1100 with EKZG_CHUNK=2048 is a ragged wide launch"""
    if chunk:
        monkeypatch.setenv("EKZG_CHUNK", str(chunk))
    cap = chunk or 1024
    chunks = [min(cap, n - o) for o in range(0, n, cap)]
    bounds = [0, 7, 8, 15, 16, 31, 32, 255, 256] + [o + d for o in range(cap, n, cap) for d in (-1, 0)]
    want = {f: 0 for f in MSM_FORMS + SUM_FORMS}
    for c in chunks:
        want[msm_form(c, c, 64, vec_ctx.srs_window)] = True
        want[SUM_FORMS[1] if c <= 256 else SUM_FORMS[0]] = True
    for blobs, pos in case_rounds(n, special_blobs(vec_ctx), bounds):
        names_c, names_p = check_4844_round(vec_ctx, blobs, set(bounds) | set(pos), n)
        assert_forms(names_c, want)
        assert_forms(names_p, dict(want, **{"k_quotient": True, "k_blob_challenge": True if n > 16 else 0}))


# ---------------------------------------------------------------- compute_kzg_proof
@pytest.mark.gpu
def test_compute_kzg_proof_edge_points(vec_ctx, pkg):
    """every chosen-coefficient and edge blob at z = 0, 1, r-1 and the domain points w^0, w^1, w^4095 (where y is the blob's
    element at the bit-reversed position), against the oracle; a non-canonical z is an error"""
    from oracle import cref
    w = pyref.root_of_unity(4096)
    zs = [(0, None), (1, None), (R - 1, None)] + [(pow(w, j, R), j) for j in (0, 1, 4095)]
    blobs = special_blobs(vec_ctx)
    got = {}
    names = launched(lambda: got.setdefault((0, 1), vec_ctx.compute_kzg_proof(blobs[0], (1).to_bytes(32, "big"))))
    assert_forms(names, {"k_quotient": True, "k_fk20_msm_vm<64>": True, "k_fk20_msm_vm<16>": 0, "k_fk20_msm_vm<4>": 0,
                         "k_sum_positions_tree(": True, "k_sum_positions(": 0})
    items = []
    for bi, b in enumerate(blobs):
        for z, j in zs:
            z32 = z.to_bytes(32, "big")
            proof, y = got[bi, z] if (bi, z) in got else vec_ctx.compute_kzg_proof(b, z32)
            if j is not None:
                e = pyref.bit_reverse(j, 12)
                assert y == b[32 * e:32 * e + 32], "blob %d: y at w^%d is not the blob element %d" % (bi, j, e)
            items.append(((bi, z), (proof, y), (key(b) + z32, lambda b=b, z32=z32: cref.compute_kzg_proof(b, z32))))
    want = oracle_all("kzg_proof", [t for _, _, t in items])
    for (where, g, _), o in zip(items, want):
        assert g == o, "compute_kzg_proof of blob %d at z = %#x differs from the oracle" % where
    with pytest.raises(pkg.KzgError):
        vec_ctx.compute_kzg_proof(blobs[0], R.to_bytes(32, "big"))
    with pytest.raises(cref.OracleError):
        cref.compute_kzg_proof(blobs[0], R.to_bytes(32, "big"))


# ---------------------------------------------------------------- cell proofs
def check_cells_round(ctx, blobs, must, n):
    """cells and proofs of one batch against the single-blob call (every blob: the direct route) and the oracle (sampled)"""
    from oracle import cref
    flat = b"".join(blobs)
    res = []
    names = launched(lambda: res.append(ctx.compute_cells_and_kzg_proofs_batch(flat, n)))
    cells, proofs, st = res[0]
    assert st == [0] * n
    for i, b in enumerate(blobs):
        c1, p1 = single(ctx, "cells", b, lambda: tuple(b"".join(x) for x in ctx.compute_cells_and_kzg_proofs(b)))
        assert cells[i * 262144:(i + 1) * 262144] == c1, "cells of blob %d differ from the single-blob call" % i
        assert proofs[i * 6144:(i + 1) * 6144] == p1, "proofs of blob %d differ from the single-blob call" % i
    pos = sample_positions(n, must)
    want = oracle_all("cells", [(key(blobs[i]), lambda b=blobs[i]: tuple(b"".join(x) for x in cref.compute_cells_and_kzg_proofs(b)))
                                for i in pos])
    for i, (c, p) in zip(pos, want):
        assert cells[i * 262144:(i + 1) * 262144] == c, "cells of blob %d differ from the oracle" % i
        assert proofs[i * 6144:(i + 1) * 6144] == p, "proofs of blob %d differ from the oracle" % i
    return names, cells, proofs


@pytest.mark.gpu
@pytest.mark.parametrize("n", [255, 256, 257, 511, 512, 777])
def test_fk20_batch(vec_ctx, n):
    """compression unbatched then batched (255/256), radix-4 then the register-form G1 NTTs with a last group of one blob (256/257),
    the 16-slice then the wide MSM (511/512), and at 777 a first piece of 224 blobs and a last NTT group of 9"""
    pieces = fk20_pieces(n)
    want = {f: 0 for f in MSM_FORMS + COMPRESS_FORMS + NTT_FORMS}
    for _, c in pieces:
        want[msm_form(n, c, 128, vec_ctx.window)] = True
    want[COMPRESS_FORMS[1] if n * 128 >= 32768 else COMPRESS_FORMS[0]] = True
    want[NTT_FORMS[2] if n <= 80 else NTT_FORMS[1] if n <= 256 else NTT_FORMS[0]] = True
    bounds = [0, 7, 8, 31, 32, 255, 256] + [o + d for o, _ in pieces[1:] for d in (-1, 0)]
    for blobs, pos in case_rounds(n, special_blobs(vec_ctx), bounds):
        names = check_cells_round(vec_ctx, blobs, set(bounds) | set(pos), n)[0]
        assert_forms(names, want)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 8])
def test_direct_route_batches(vec_ctx, n, monkeypatch):
    """the direct proof route (128 SRS MSMs per blob) at its largest batches: n = 3 sums 384 virtual blobs linearly, n = 8
    launches the wide MSM on the SRS tables -- against FK20 (EKZG_DIRECT_MAX=0) on the same blobs, the single-blob call and the
    oracle on every blob"""
    Bv = 128 * n
    want = {f: 0 for f in MSM_FORMS + SUM_FORMS + NTT_FORMS}
    want.update({msm_form(Bv, Bv, 64, vec_ctx.srs_window): True, SUM_FORMS[0]: True, "k_coset_quotients": True})
    for blobs, pos in case_rounds(n, special_blobs(vec_ctx), []) + [([random_blob(i) for i in range(n)], [])]:
        monkeypatch.setenv("EKZG_DIRECT_MAX", str(n))
        names, cells, proofs = check_cells_round(vec_ctx, blobs, range(n), n)
        assert_forms(names, want)
        monkeypatch.setenv("EKZG_DIRECT_MAX", "0")
        fk = vec_ctx.compute_cells_and_kzg_proofs_batch(b"".join(blobs), n)
        assert fk == (cells, proofs, [0] * n), "the direct route differs from FK20"


# ---------------------------------------------------------------- verifiers
def _flip(cell, byte=31):
    return cell[:byte] + bytes([cell[byte] ^ 1]) + cell[byte + 1:]


@pytest.mark.gpu
def test_blob_verifiers_1024(vec_ctx):
    """verify_blob_kzg_proof_batch(_items) on 1024 blobs: honest, and one bad proof at 0, 1023 and 513 (another blob's proof);
    then the first 16 and 17 blobs (challenges on the host, then on the device).  Every verdict against the single-blob call,
    sampled ones against the oracle"""
    from oracle import cref
    n = 1024
    blobs, pos = case_rounds(n, special_blobs(vec_ctx), [0, 255, 256, 512, 513, 1023])[0]
    flat = b"".join(blobs)
    cms, _ = vec_ctx.blob_to_kzg_commitment_batch(flat, n)
    prs, _ = vec_ctx.compute_blob_kzg_proof_batch(flat, cms, n)
    cl = [cms[48 * i:48 * i + 48] for i in range(n)]
    pl = [prs[48 * i:48 * i + 48] for i in range(n)]
    for i in range(n):
        assert single(vec_ctx, "verify_blob", blobs[i] + cl[i] + pl[i], lambda: vec_ctx.verify_blob_kzg_proof(blobs[i], cl[i], pl[i])) is True, i
    sample = sample_positions(n, [0, 1, 16, 255, 256, 512, 513, 514, 1023] + list(pos))
    want = oracle_all("verify_blob", [(key(blobs[i] + cl[i] + pl[i]), lambda i=i: cref.verify_blob_kzg_proof(blobs[i], cl[i], pl[i]))
                                      for i in sample])
    assert all(want)
    for m in (n, 16, 17):
        for bad in [[], [0], [m - 1]] + ([[513]] if m > 513 else []):
            p = list(pl[:m])
            for i in bad:
                p[i] = pl[(i + 1) % m]
            res = {}
            names = launched(lambda: res.setdefault("items", vec_ctx.verify_blob_kzg_proof_batch_items(blobs[:m], cl[:m], p)))
            assert_forms(names, {"k_blob_challenge": True if m > 16 else 0})
            ok, st = res["items"]
            assert st == [1 if i in bad else 0 for i in range(m)], (m, bad)
            assert ok is (not bad) is vec_ctx.verify_blob_kzg_proof_batch(blobs[:m], cl[:m], p)
            for i in bad:
                assert vec_ctx.verify_blob_kzg_proof(blobs[i], cl[i], p[i]) is False
                assert cref.verify_blob_kzg_proof(blobs[i], cl[i], p[i]) is False


def _openings(ctx, blobs):
    nb = len(blobs)
    flat = b"".join(blobs)
    cms, st = ctx.blob_to_kzg_commitment_batch(flat, nb)
    cells, proofs, st2 = ctx.compute_cells_and_kzg_proofs_batch(flat, nb)
    assert not any(st) and not any(st2)
    C = [cms[48 * (k // 128):48 * (k // 128) + 48] for k in range(nb * 128)]
    I = [k % 128 for k in range(nb * 128)]
    CL = [cells[k * 2048:(k + 1) * 2048] for k in range(nb * 128)]
    PR = [proofs[k * 48:(k + 1) * 48] for k in range(nb * 128)]
    return C, I, CL, PR


@pytest.mark.gpu
@pytest.mark.parametrize("n_open", [512, 513, 65536])
def test_cell_verifier_one_group_per_opening(vec_ctx, n_open):
    """verify_cell_kzg_proof_batch_groups with a group per opening: 512 groups run the per-group interpolation MSM one point per
    thread, 513 the 16-slice form, 65 536 (512 blobs x 128 cells) the wide form.  The aggregate check always runs one
    single-point MSM (one-point-per-thread form) before.  Exact verdicts; flagged and sampled openings against the plain call and
    the oracle"""
    from oracle import cref
    nb = (n_open + 127) // 128
    blobs = [random_blob(i) for i in range(nb)]
    sp = special_blobs(vec_ctx)
    blobs[0], blobs[-1] = sp[1], sp[-1]
    C, I, CL, PR = (x[:n_open] for x in _openings(vec_ctx, blobs))
    bad = [0, n_open - 1] + ([32767] if n_open > 32768 else [n_open // 2])
    cells = list(CL)
    for k in bad:
        cells[k] = _flip(cells[k], 32 * (k % 64) + 31)
    groups = list(range(n_open))
    res = {}
    names = launched(lambda: res.setdefault("g", vec_ctx.verify_cell_kzg_proof_batch_groups(C, I, cells, PR, groups)))
    want = dict.fromkeys(MSM_FORMS, 0)
    want["k_fk20_msm_vm<64>"] = 1                                      # the aggregate's single-point MSM
    want[msm_form(n_open, n_open, 1, vec_ctx.srs_window)] += 1         # the per-group one
    assert_forms(names, want)
    ok, st = res["g"]
    assert not ok and [k for k in range(n_open) if st[k]] == sorted(bad) and set(st) <= {0, 1}
    check = sorted(set(bad) | set(random.Random(n_open).sample(range(n_open), 64)))
    for k in check:
        assert vec_ctx.verify_cell_kzg_proof_batch([C[k]], [I[k]], [cells[k]], [PR[k]]) is (k not in bad), k
    want = oracle_all("verify_cell", [(key(C[k] + cells[k] + PR[k]) + bytes([I[k]]),
                                       lambda k=k: cref.verify_cell_kzg_proof_batch([C[k]], [I[k]], [cells[k]], [PR[k]])) for k in check])
    assert want == [k not in bad for k in check]
