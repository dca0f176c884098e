"""GPU tests of blob recovery without cell proofs (eth_kzg_b200_recover_blobs_batch / eth_kzg_b200_recover_blob): the same
inputs, statuses and error messages as recover_cells_and_kzg_proofs, and for every valid item cells 0..63 of its output,
byte for byte.  Covers the consensus vectors, round trips over the erasure patterns, parity with the proofs call and the
C oracle, invalid items at every position, chunking with pinned and pageable buffers, a multi-device context, concurrent
single-blob callers, and the kernels the path launches (no FK20 stage)."""
import ctypes as C
import importlib
import json
import os
import random
import threading

import pytest

from tests import vectors

pytestmark = pytest.mark.gpu

BLOB = 131072
CELL = 2048
EXT = 128 * CELL
R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001


def _syn():
    return importlib.import_module("eth_kzg_b200.synthetic")


def _cells_of(ctx, blobs):
    """the 128 cells of every blob (compute_cells, no proofs), as lists of 2048-byte cells"""
    cells, _, st = ctx.compute_cells_and_kzg_proofs_batch(b"".join(blobs), len(blobs), want_proofs=False)
    assert st == [0] * len(blobs)
    return [[cells[b * EXT + k * CELL:b * EXT + (k + 1) * CELL] for k in range(128)] for b in range(len(blobs))]


def _raw_batch(ctx, lib, which, idx_lists, cell_lists):
    """one batch call through the C ABI -> (Err?, message, status list, blobs (n x 131072 B; cells 0..63 for the proofs call))"""
    n = len(idx_lists)
    counts = (C.c_uint64 * max(n, 1))(*[len(x) for x in idx_lists])
    flat_idx = [i for x in idx_lists for i in x]
    idx = (C.c_uint64 * max(len(flat_idx), 1))(*flat_idx)
    cells = b"".join(c for x in cell_lists for c in x)
    status = C.create_string_buffer(max(n, 1))
    h = C.c_void_p(ctx.handle)
    if which == "blobs":
        out = C.create_string_buffer(max(n, 1) * BLOB)
        res = lib.eth_kzg_b200_recover_blobs_batch(h, C.c_uint64(n), counts, idx, cells, out, status)
        blobs = out.raw[:n * BLOB]
    else:
        oc = C.create_string_buffer(max(n, 1) * EXT)
        op = C.create_string_buffer(max(n, 1) * 128 * 48)
        res = lib.eth_kzg_b200_recover_cells_and_kzg_proofs_batch(h, C.c_uint64(n), counts, idx, cells, oc, op, status)
        blobs = b"".join(oc.raw[i * EXT:i * EXT + BLOB] for i in range(n))
    msg = None
    if res.status != 0:
        msg = C.string_at(res.error_msg).decode() if res.error_msg else ""
        lib.eth_kzg_free_error_message(res.error_msg)
    return res.status != 0, msg, list(status.raw[:n]), blobs


def _assert_same_as_proofs_call(ctx, pkg, idx_lists, cell_lists):
    """statuses, Err and message equal to the proofs call; valid items byte-equal to its cells 0..63.  -> the status list"""
    lib = pkg.load_library()
    err_b, msg_b, st_b, blobs_b = _raw_batch(ctx, lib, "blobs", idx_lists, cell_lists)
    err_p, msg_p, st_p, blobs_p = _raw_batch(ctx, lib, "proofs", idx_lists, cell_lists)
    assert st_b == st_p
    assert (err_b, msg_b) == (err_p, msg_p)
    assert err_b == any(st_b)
    for i, s in enumerate(st_b):
        if s == 0:
            assert blobs_b[i * BLOB:(i + 1) * BLOB] == blobs_p[i * BLOB:(i + 1) * BLOB], "item %d" % i
    return st_b


# ---- consensus vectors --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,inp,expected", [pytest.param(n, i, o, id=n) for n, i, o in vectors.load("recover_cells_and_kzg_proofs")])
def test_recover_blob_vectors(vec_ctx, pkg, name, inp, expected):
    idx, cells = inp["cell_indices"], inp["cells"]
    if expected is not None:
        want = b"".join(expected[0][:64])
        assert vec_ctx.recover_blob(idx, cells) == want
        assert vec_ctx.recover_blobs_batch([idx], [cells]) == (want, [0])
        return
    with pytest.raises(pkg.KzgError) as proofs_err:
        vec_ctx.recover_cells_and_kzg_proofs(idx, cells)
    with pytest.raises(pkg.KzgError) as blob_err:
        vec_ctx.recover_blob(idx, cells)
    assert str(blob_err.value) == str(proofs_err.value)
    if len(idx) == len(cells) and all(len(c) == CELL for c in cells):   # expressible as a batch item
        st = _assert_same_as_proofs_call(vec_ctx, pkg, [idx], [cells])
        assert st[0] != 0


# ---- round trips --------------------------------------------------------------------------------------------------------
def _patterns():
    rng = random.Random(7594)
    return {
        "first_half": list(range(64)),
        "second_half": list(range(64, 128)),
        "every_other": list(range(0, 128, 2)),
        "random_64": sorted(rng.sample(range(128), 64)),
        "random_100": sorted(rng.sample(range(128), 100)),
        "all": list(range(128)),
    }


def test_roundtrip_erasure_patterns(das_ctx):
    syn = _syn()
    blobs = [syn.blob(4100 + i) for i in range(5)] + syn.edge_blobs()
    cells = _cells_of(das_ctx, blobs)
    idx_lists, cell_lists, want = [], [], []
    for b, blob in enumerate(blobs):
        assert b"".join(cells[b][:64]) == blob
        for keep in _patterns().values():
            idx_lists.append(keep)
            cell_lists.append([cells[b][k] for k in keep])
            want.append(blob)
    out, st = das_ctx.recover_blobs_batch(idx_lists, cell_lists)
    assert st == [0] * len(want)
    for i, blob in enumerate(want):
        assert out[i * BLOB:(i + 1) * BLOB] == blob, "item %d" % i


def test_roundtrip_same_columns_every_blob(das_ctx):
    """PeerDAS: a node that custodies the same 64 columns holds the same cell indices of every blob"""
    syn = _syn()
    blobs = [syn.blob(4200 + i) for i in range(24)]
    cells = _cells_of(das_ctx, blobs)
    cols = sorted(random.Random(64).sample(range(128), 64))
    out, st = das_ctx.recover_blobs_batch([cols] * len(blobs), [[c[k] for k in cols] for c in cells])
    assert st == [0] * len(blobs)
    assert out == b"".join(blobs)


# ---- parity with the proofs call and the oracle ------------------------------------------------------------------------
def test_parity_with_proofs_call_random_blobs(das_ctx, pkg):
    import numpy as np
    n = 40
    raw = np.random.default_rng(17).integers(0, 256, size=(n, 4096, 32), dtype=np.uint8)
    raw[:, :, 0] &= 0x3F
    blobs = [raw[i].tobytes() for i in range(n)]
    cells = _cells_of(das_ctx, blobs)
    rng = random.Random(5)
    idx = [sorted(rng.sample(range(128), rng.choice([64, 65, 90, 127, 128]))) for _ in range(n)]
    st = _assert_same_as_proofs_call(das_ctx, pkg, idx, [[cells[b][k] for k in idx[b]] for b in range(n)])
    assert st == [0] * n


def test_matches_oracle(das_ctx):
    from oracle import cref
    blob = _syn().blob(4321)
    ocells, _ = cref.compute_cells_and_kzg_proofs(blob)
    keep = _patterns()["random_64"]
    oc, _ = cref.recover_cells_and_kzg_proofs(keep, [ocells[k] for k in keep])
    assert das_ctx.recover_blob(keep, [ocells[k] for k in keep]) == b"".join(oc[:64]) == blob


# ---- invalid items -----------------------------------------------------------------------------------------------------
def _invalid_items(cells_a, cells_b):
    """(class, indices, cells) for every invalid class"""
    good = list(range(0, 128, 2))
    noncanon = [cells_a[k] for k in good]
    noncanon[10] = R.to_bytes(32, "big") + noncanon[10][32:]          # exactly r: the smallest non-canonical scalar
    two = sorted(good + [1, 3, 5, 7, 9, 11])                           # 70 cells: more than 64, so the degree check can fail
    mixed = [cells_a[k] if j < 35 else cells_b[k] for j, k in enumerate(two)]
    return [
        ("too_few", list(range(63)), [cells_a[k] for k in range(63)]),
        ("not_ascending", [2, 0] + list(range(4, 128, 2)), [cells_a[k] for k in [2, 0] + list(range(4, 128, 2))]),
        ("duplicate", [0, 0] + list(range(2, 128, 2)), [cells_a[k] for k in [0, 0] + list(range(2, 128, 2))]),
        ("out_of_range", list(range(0, 126, 2)) + [128], [cells_a[k] for k in range(0, 126, 2)] + [cells_a[0]]),
        ("non_canonical", good, noncanon),
        ("two_blobs", two, mixed),
    ]


def test_invalid_item_at_each_position(das_ctx, pkg):
    syn = _syn()
    blobs = [syn.blob(4400 + i) for i in range(9)]
    cells = _cells_of(das_ctx, blobs)
    rng = random.Random(3)
    valid = []
    for b in range(9):
        keep = sorted(rng.sample(range(128), 64 + b))
        valid.append((keep, [cells[b][k] for k in keep]))
    want_status = {"too_few": 3, "not_ascending": 3, "duplicate": 3, "out_of_range": 3, "non_canonical": 1, "two_blobs": 4}
    for cls, idx, cl in _invalid_items(cells[0], cells[1]):
        for pos in (0, 4, 9):
            items = valid[:pos] + [(idx, cl)] + valid[pos:]
            st = _assert_same_as_proofs_call(das_ctx, pkg, [i[0] for i in items], [i[1] for i in items])
            assert st == [want_status[cls] if i == pos else 0 for i in range(len(items))], (cls, pos)
            out, st2 = das_ctx.recover_blobs_batch([i[0] for i in items], [i[1] for i in items])
            assert st2 == st
            for i in range(len(items)):
                if i != pos:
                    b = i if i < pos else i - 1
                    assert out[i * BLOB:(i + 1) * BLOB] == blobs[b], (cls, pos, i)


def test_error_precedence_in_mixed_batch(das_ctx, pkg):
    """several invalid classes in one batch: an index error is reported before any device-side error, as by the proofs call"""
    syn = _syn()
    blobs = [syn.blob(4500 + i) for i in range(3)]
    cells = _cells_of(das_ctx, blobs)
    bad = {c: (i, cl) for c, i, cl in _invalid_items(cells[0], cells[1])}
    keep = list(range(1, 128, 2))
    ok = (keep, [cells[2][k] for k in keep])
    for order in (["two_blobs", "non_canonical", "too_few"], ["non_canonical", "two_blobs"], ["two_blobs", "out_of_range", "not_ascending"]):
        items = [ok] + [bad[c] for c in order] + [ok]
        st = _assert_same_as_proofs_call(das_ctx, pkg, [i[0] for i in items], [i[1] for i in items])
        assert st[0] == st[-1] == 0 and all(st[1:-1])


def test_all_valid_batch_is_ok(das_ctx, pkg):
    syn = _syn()
    blobs = [syn.blob(4600 + i) for i in range(3)]
    cells = _cells_of(das_ctx, blobs)
    keep = list(range(64, 128))
    err, msg, st, out = _raw_batch(das_ctx, pkg.load_library(), "blobs", [keep] * 3, [[c[k] for k in keep] for c in cells])
    assert (err, msg, st, out) == (False, None, [0, 0, 0], b"".join(blobs))


# ---- chunking and memory -----------------------------------------------------------------------------------------------
@pytest.fixture
def small_chunks():
    old = os.environ.get("EKZG_CHUNK")
    os.environ["EKZG_CHUNK"] = "24"
    yield 24
    if old is None:
        del os.environ["EKZG_CHUNK"]
    else:
        os.environ["EKZG_CHUNK"] = old


def _ragged_batch(ctx, n, first, bad_at):
    """n items over n synthetic blobs with varying patterns; item i in bad_at is made invalid (non-canonical or too few cells)"""
    syn = _syn()
    blobs = [syn.blob(first + i) for i in range(n)]
    cells = _cells_of(ctx, blobs)
    rng = random.Random(first)
    idx, cl = [], []
    for b in range(n):
        keep = sorted(rng.sample(range(128), rng.choice([64, 77, 100, 128])))
        c = [cells[b][k] for k in keep]
        if b in bad_at and b % 2:
            c[0] = b"\xff" * 32 + c[0][32:]
        elif b in bad_at:
            keep, c = keep[:40], c[:40]
        idx.append(keep)
        cl.append(c)
    return blobs, idx, cl


def _pinned_call(ctx, lib, idx, cl):
    import torch
    n = len(idx)
    counts = (C.c_uint64 * n)(*[len(x) for x in idx])
    flat_idx = [i for x in idx for i in x]
    ind = (C.c_uint64 * len(flat_idx))(*flat_idx)
    h_cells = torch.frombuffer(bytearray(b"".join(c for x in cl for c in x)), dtype=torch.uint8).pin_memory()
    h_out = torch.empty(n * BLOB, dtype=torch.uint8).pin_memory()
    h_st = torch.empty(n, dtype=torch.uint8).pin_memory()
    res = lib.eth_kzg_b200_recover_blobs_batch(C.c_void_p(ctx.handle), C.c_uint64(n), counts, ind, C.c_void_p(h_cells.data_ptr()),
                                               C.c_void_p(h_out.data_ptr()), C.c_void_p(h_st.data_ptr()))
    if res.status != 0:
        lib.eth_kzg_free_error_message(res.error_msg)
    return res.status != 0, bytes(h_out.numpy()), list(h_st.numpy())


@pytest.mark.parametrize("with_invalid", [False, True])
def test_chunked_equals_one_chunk(das_ctx, pkg, small_chunks, with_invalid):
    n = 2 * small_chunks + 5                       # 3 chunks over the two workspaces, the last one ragged
    bad = {0, small_chunks - 1, small_chunks, 2 * small_chunks + 1, n - 1} if with_invalid else set()
    blobs, idx, cl = _ragged_batch(das_ctx, n, 4700, bad)
    lib = pkg.load_library()
    chunked = _raw_batch(das_ctx, lib, "blobs", idx, cl)
    pinned = _pinned_call(das_ctx, lib, idx, cl)
    os.environ["EKZG_CHUNK"] = "1024"
    whole = _raw_batch(das_ctx, lib, "blobs", idx, cl)
    whole_pinned = _pinned_call(das_ctx, lib, idx, cl)
    assert chunked[2] == whole[2] == pinned[2] == whole_pinned[2]
    assert chunked[0] == whole[0] == pinned[0] == whole_pinned[0] == bool(bad)
    for i in range(n):
        if i not in bad:
            assert whole[2][i] == 0
            for out in (chunked[3], whole[3], pinned[1], whole_pinned[1]):
                assert out[i * BLOB:(i + 1) * BLOB] == blobs[i], "item %d" % i
    _assert_same_as_proofs_call(das_ctx, pkg, idx, cl)


def test_pieces_of_one_chunk(das_ctx, pkg):
    """300 items in one chunk: three pieces, invalid items on both sides of the piece boundaries"""
    n = 300
    bad = {0, 99, 100, 101, 199, 200, 299}
    blobs, idx, cl = _ragged_batch(das_ctx, n, 5000, bad)
    st = _assert_same_as_proofs_call(das_ctx, pkg, idx, cl)
    out, st2 = das_ctx.recover_blobs_batch(idx, cl)
    assert st2 == st and [i for i in range(n) if st[i]] == sorted(bad)
    for i in range(n):
        if i not in bad:
            assert out[i * BLOB:(i + 1) * BLOB] == blobs[i], "item %d" % i
    _, pinned_out, pinned_st = _pinned_call(das_ctx, pkg.load_library(), idx, cl)
    assert pinned_st == st and all(pinned_out[i * BLOB:(i + 1) * BLOB] == blobs[i] for i in range(n) if i not in bad)


def test_empty_batch(das_ctx, pkg):
    lib = pkg.load_library()
    res = lib.eth_kzg_b200_recover_blobs_batch(C.c_void_p(das_ctx.handle), C.c_uint64(0), None, None, None, None, None)
    assert res.status == 0
    assert das_ctx.recover_blobs_batch([], []) == (b"", [])


# ---- multi-device, threads ---------------------------------------------------------------------------------------------
def test_multi_device_equals_single(das_ctx, pkg):
    old = os.environ.get("EKZG_DEVICES")
    os.environ["EKZG_DEVICES"] = "0,0"
    try:
        multi = pkg.DASContext(use_precomp=False)
    finally:
        if old is None:
            del os.environ["EKZG_DEVICES"]
        else:
            os.environ["EKZG_DEVICES"] = old
    try:
        assert len(multi.devices) == 2
        n = 70
        bad = {3, 40, 69}
        blobs, idx, cl = _ragged_batch(das_ctx, n, 5400, bad)
        lib = pkg.load_library()
        m_err, _, m_st, m_out = _raw_batch(multi, lib, "blobs", idx, cl)
        s_err, _, s_st, s_out = _raw_batch(das_ctx, lib, "blobs", idx, cl)
        assert (m_err, m_st, m_out) == (s_err, s_st, s_out)
        assert [i for i in range(n) if m_st[i]] == sorted(bad)
        # each shard reports its own first error, so the message is compared with the proofs call on the same context
        _assert_same_as_proofs_call(multi, pkg, idx, cl)
        keep = list(range(0, 128, 2))
        cells0 = _cells_of(das_ctx, [blobs[0]])[0]
        assert multi.recover_blob(keep, [cells0[k] for k in keep]) == blobs[0]
    finally:
        multi.close()


def test_concurrent_recover_blob(das_ctx):
    syn = _syn()
    blobs = [syn.blob(5600 + i) for i in range(16)]
    cells = _cells_of(das_ctx, blobs)
    pats = list(_patterns().values())
    results, errors = [None] * 16, []

    def run(t):
        try:
            keep = pats[t % len(pats)]
            results[t] = das_ctx.recover_blob(keep, [cells[t][k] for k in keep])
        except Exception as ex:   # noqa: BLE001 -- reported below
            errors.append(ex)

    th = [threading.Thread(target=run, args=(t,)) for t in range(16)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors
    assert results == blobs


# ---- what the path launches --------------------------------------------------------------------------------------------
FK20_STAGES = ("toeplitz", "fk20", "fixed_msm", "g1_ntt", "g1_compress", "coset_quotients", "coeffs_to_cells")
THIS_PATH = ("k_recover_prep", "k_recover_ntt_packed", "k_recover_ntt<2>", "k_recover_ntt<3>", "k_coeffs_to_blob")

# One chunk of 100 blobs (a single piece) in a process of its own, so that no earlier test's profiler or context state can
# bear on what is recorded: the launch-count delta of one call, and the kernel names one torch.profiler run of it records.
_CHILD = r"""
import json, os, sys, tempfile
import torch
from torch.profiler import ProfilerActivity, profile
sys.path.insert(0, sys.argv[1])
import __graft_entry__ as g
pkg = g.load_package()
lib = pkg.load_library()
ctx = pkg.DASContext(use_precomp=False)
syn = __import__("importlib").import_module("eth_kzg_b200.synthetic")
n = 100
blobs = [syn.blob(5800 + i) for i in range(n)]
cells, _, st = ctx.compute_cells_and_kzg_proofs_batch(b"".join(blobs), n, want_proofs=False)
keep = list(range(1, 128, 2))
cl = [[cells[(b * 128 + k) * 2048:(b * 128 + k + 1) * 2048] for k in keep] for b in range(n)]
ctx.recover_blobs_batch([keep] * n, cl)   # first use allocates
torch.cuda.synchronize()
before = lib.eth_kzg_b200_kernel_launch_count()
out, st = ctx.recover_blobs_batch([keep] * n, cl)
launches = lib.eth_kzg_b200_kernel_launch_count() - before
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    ctx.recover_blobs_batch([keep] * n, cl)
    torch.cuda.synchronize()
with tempfile.TemporaryDirectory() as d:
    path = os.path.join(d, "trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        names = [e["name"] for e in json.load(f)["traceEvents"] if e.get("cat") == "kernel"]
ctx.close()
print(json.dumps({"ok": st == [0] * n and out == b"".join(blobs), "launches": launches, "kernels": names}))
"""


def test_launches_no_fk20(das_ctx):
    """(das_ctx: skipped where there is no device, like the rest of the file)"""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    r = subprocess.run([sys.executable, "-c", _CHILD, root], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    names = res["kernels"]
    assert res["ok"]
    assert res["launches"] == len(THIS_PATH)
    assert sorted(k.split("(")[0].split("::")[-1] for k in names) == sorted(THIS_PATH), names
    assert not [k for k in names if any(s in k for s in FK20_STAGES)], names
