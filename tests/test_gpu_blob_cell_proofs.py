"""GPU tests of verify_blob_cell_proofs_batch: the 128 cell proofs and the commitment of whole blobs, checked by recomputing them
on the device.  Verdicts per blob: 0 verifies, 1 does not, 2 malformed; per cell: 0 the proof of the cell, 1 a valid point but
not that proof, 2 an invalid encoding (all 2 for a non-canonical blob).  Checked against the consensus vectors, the C oracle, the
two-call route (cells, then the grouped cell verifier) and exact expectations for each class of corruption."""
import concurrent.futures
import ctypes as C
import json
import os
import random
import subprocess
import sys

import pytest

from oracle import pyref
from tests import setup_util as su
from tests import vectors
from tests.test_gpu_batch_forms import blob_from_coeffs, launched
from tests.test_gpu_setup import _g1_on_curve_off_subgroup

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = pyref.R
BLOB = 131072
IDENTITY = b"\xc0" + bytes(47)


# ---------------------------------------------------------------- helpers
def rand_blobs(n, seed):
    import numpy as np
    a = np.random.default_rng(seed).integers(0, 256, size=(n, 4096, 32), dtype=np.uint8)
    a[:, :, 0] &= 0x3F
    return [a[i].tobytes() for i in range(n)]


def low_degree_blob(seed):
    """degree < 64: every cell proof is the identity"""
    rng = random.Random(seed)
    return blob_from_coeffs([rng.randrange(R) for _ in range(64)] + [0] * 4032)


def non_canonical(blob):
    return (R + 5).to_bytes(32, "big") + blob[32:]


def honest(ctx, blobs):
    """-> (commitments, [[128 proofs] per blob]) from the library's provers"""
    n = len(blobs)
    flat = b"".join(blobs)
    comm, st = ctx.blob_to_kzg_commitment_batch(flat, n)
    _, proofs, st2 = ctx.compute_cells_and_kzg_proofs_batch(flat, n)
    assert st == [0] * n and st2 == [0] * n
    return [comm[48 * i:48 * i + 48] for i in range(n)], [[proofs[(i * 128 + k) * 48:(i * 128 + k + 1) * 48] for k in range(128)] for i in range(n)]


def run(ctx, blobs, comms, proofs):
    """-> (all_ok, item status, [[128 cell statuses] per blob])"""
    n = len(blobs)
    ok, st, cells = ctx.verify_blob_cell_proofs_batch(b"".join(blobs), b"".join(comms), b"".join(b"".join(p) for p in proofs), n, want_cells=True)
    return ok, st, [list(cells[128 * i:128 * i + 128]) for i in range(n)]


def expect(n, items=None, cells=None):
    """expected (all_ok, item status, cell statuses): items {i: status}, cells {(i, k): status} or {i: status of all 128}"""
    st = [0] * n
    cs = [[0] * 128 for _ in range(n)]
    for i, v in (items or {}).items():
        st[i] = v
    for key, v in (cells or {}).items():
        if isinstance(key, tuple):
            cs[key[0]][key[1]] = v
        else:
            cs[key] = [v] * 128
    return all(s == 0 for s in st), st, cs


def off_curve():
    x = 1
    while su.fp_sqrt((x * x * x + 4) % su.P) is not None:
        x += 1
    enc = bytearray(x.to_bytes(48, "big"))
    enc[0] |= 0x80
    return bytes(enc)


def x_not_below_p():
    enc = bytearray(su.P.to_bytes(48, "big"))
    enc[0] |= 0x80
    return bytes(enc)


def bad_flags(valid):
    return bytes([valid[0] & 0x7F]) + valid[1:]   # the compression bit cleared: not a 48-byte encoding


def off_subgroup():
    return _g1_on_curve_off_subgroup(random.Random(7594))


# ---------------------------------------------------------------- 1. consensus vectors
_CELL_CASES = [pytest.param(n, i, o, id=n) for n, i, o in vectors.load("compute_cells_and_kzg_proofs")]


@pytest.mark.parametrize("name,inp,out", _CELL_CASES)
def test_consensus_vectors(vec_ctx, name, inp, out):
    blob = inp["blob"]
    if len(blob) != BLOB:
        pytest.skip("a blob of the wrong length cannot cross the C ABI")
    if out is None:
        ok, st, cs = run(vec_ctx, [blob], [IDENTITY], [[IDENTITY] * 128])
        assert (ok, st, cs) == expect(1, {0: 2}, {0: 2})
        return
    comm = vec_ctx.blob_to_kzg_commitment(blob)
    assert run(vec_ctx, [blob], [comm], [list(out[1])]) == expect(1)


# ---------------------------------------------------------------- 2. C oracle
_ORACLE = {}


def oracle(blobs):
    from oracle import cref
    cref.lib()
    todo = [b for b in blobs if b not in _ORACLE]
    with concurrent.futures.ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        for b, v in zip(todo, ex.map(lambda b: (cref.blob_to_kzg_commitment(b), cref.compute_cells_and_kzg_proofs(b)[1]), todo)):
            _ORACLE[b] = v
    return [_ORACLE[b] for b in blobs]


def test_against_c_oracle(vec_ctx):
    import importlib
    syn = importlib.import_module("eth_kzg_b200.synthetic")
    blobs = list(syn.edge_blobs()) + [low_degree_blob(1), blob_from_coeffs([0] * 4095 + [1])] + rand_blobs(10, 16)
    assert len(blobs) >= 16
    ref = oracle(blobs)
    assert all(p == IDENTITY for p in ref[4][1]), "a degree < 64 blob has identity proofs"
    assert run(vec_ctx, blobs, [c for c, _ in ref], [p for _, p in ref]) == expect(len(blobs))


# ---------------------------------------------------------------- 3. corruption classes
N3 = 64
_BATCH = {}


def batch64(ctx):
    key = (ctx.window, ctx.srs_window)
    if key not in _BATCH:
        blobs = rand_blobs(N3, 64)
        _BATCH[key] = (blobs,) + honest(ctx, blobs)
    return _BATCH[key]


def coset_value(k):
    """h_k^64: every point x of cell k satisfies x^64 = h_k^64"""
    w = pyref.root_of_unity(8192)
    return pow(w, pyref.bit_reverse(64 * k, 13) * 64, R)


def corrupt(ctx, cls, p):
    """the 64-blob batch with corruption `cls` at position p -> (blobs, commitments, proofs, expected)"""
    blobs, comms, proofs = batch64(ctx)
    blobs, comms, proofs = list(blobs), list(comms), [list(x) for x in proofs]
    q = (p + 1) % N3
    if cls == "swap":
        proofs[p][5], proofs[p][77] = proofs[p][77], proofs[p][5]
        return blobs, comms, proofs, expect(N3, {p: 1}, {(p, 5): 1, (p, 77): 1})
    if cls == "other_blob_proof":
        proofs[p][9] = proofs[q][9]
        return blobs, comms, proofs, expect(N3, {p: 1}, {(p, 9): 1})
    if cls == "identity_for_real":
        assert proofs[p][3] != IDENTITY
        proofs[p][3] = IDENTITY
        return blobs, comms, proofs, expect(N3, {p: 1}, {(p, 3): 1})
    if cls == "real_for_identity":
        blobs[p] = low_degree_blob(p)
        c, pr = honest(ctx, [blobs[p]])
        comms[p], proofs[p] = c[0], pr[0]
        assert proofs[p] == [IDENTITY] * 128
        proofs[p][4] = comms[q]   # a valid point other than the identity
        return blobs, comms, proofs, expect(N3, {p: 1}, {(p, 4): 1})
    if cls.startswith("malformed_proof_"):
        enc = {"x_ge_p": x_not_below_p(), "flags": bad_flags(proofs[p][11]), "off_curve": off_curve(), "off_subgroup": off_subgroup()}[cls[16:]]
        proofs[p][11] = enc
        return blobs, comms, proofs, expect(N3, {p: 2}, {(p, 11): 2})
    if cls == "other_commitment":
        comms[p] = comms[q]
        return blobs, comms, proofs, expect(N3, {p: 1})
    if cls == "malformed_commitment":
        comms[p] = off_curve()
        return blobs, comms, proofs, expect(N3, {p: 2})
    if cls == "non_canonical_blob":
        blobs[p] = non_canonical(blobs[p])
        return blobs, comms, proofs, expect(N3, {p: 2}, {p: 2})
    if cls == "coset_commitment":
        k = 37
        coeffs = pyref.blob_to_coeffs(blobs[p])
        c, a = 123456789, coset_value(k)
        coeffs2 = list(coeffs)
        coeffs2[64] = (coeffs2[64] + c) % R
        coeffs2[0] = (coeffs2[0] - c * a) % R
        blob2 = blob_from_coeffs(coeffs2)
        cells, cells2 = ctx.compute_cells(blobs[p]), ctx.compute_cells(blob2)
        assert cells[k] == cells2[k] and cells[k + 1] != cells2[k + 1], "p and p' agree on cell k only"
        comm2, proofs2 = honest(ctx, [blob2])
        assert ctx.verify_cell_kzg_proof_batch([comm2[0]], [k], [cells[k]], [proofs2[0][k]]), "the plain verifier accepts opening k"
        comms[p] = comm2[0]
        proofs[p][k] = proofs2[0][k]
        return blobs, comms, proofs, expect(N3, {p: 1}, {(p, k): 1})
    raise AssertionError(cls)


CLASSES = ["swap", "other_blob_proof", "identity_for_real", "real_for_identity", "malformed_proof_x_ge_p", "malformed_proof_flags",
           "malformed_proof_off_curve", "malformed_proof_off_subgroup", "other_commitment", "malformed_commitment", "coset_commitment",
           "non_canonical_blob"]


@pytest.mark.parametrize("cls", CLASSES)
def test_corruption_classes(vec_ctx, cls):
    for p in (0, N3 // 2, N3 - 1):
        blobs, comms, proofs, want = corrupt(vec_ctx, cls, p)
        assert run(vec_ctx, blobs, comms, proofs) == want, (cls, p)


# ---------------------------------------------------------------- 4. against the two-call route
def test_against_two_call_route(vec_ctx):
    """one mixed batch (every class but the non-canonical blob, whose cells the two-call route cannot compute) through this call
    and through compute_cells_and_kzg_proofs_batch + verify_cell_kzg_proof_batch_groups"""
    blobs, comms, proofs = batch64(vec_ctx)
    blobs, comms, proofs = list(blobs), list(comms), [list(x) for x in proofs]
    for p, cls in enumerate(CLASSES[:-1]):
        b, c, pr, _ = corrupt(vec_ctx, cls, 5 * p + 2)
        blobs[5 * p + 2], comms[5 * p + 2], proofs[5 * p + 2] = b[5 * p + 2], c[5 * p + 2], pr[5 * p + 2]
    n = len(blobs)
    own, ost = vec_ctx.blob_to_kzg_commitment_batch(b"".join(blobs), n)
    assert ost == [0] * n
    ok, st, cs = run(vec_ctx, blobs, comms, proofs)
    cells, _, cst = vec_ctx.compute_cells_and_kzg_proofs_batch(b"".join(blobs), n, want_proofs=False)
    assert cst == [0] * n
    C_ = [comms[i] for i in range(n) for _ in range(128)]
    I = [k for _ in range(n) for k in range(128)]
    CL = [cells[j * 2048:(j + 1) * 2048] for j in range(n * 128)]
    PR = [proofs[i][k] for i in range(n) for k in range(128)]
    ok_b, per_blob = vec_ctx.verify_cell_kzg_proof_batch_groups(C_, I, CL, PR, [i for i in range(n) for _ in range(128)])
    _, per_open = vec_ctx.verify_cell_kzg_proof_batch_groups(C_, I, CL, PR, list(range(n * 128)))
    assert st == per_blob and ok == ok_b
    assert sorted(set(st)) == [0, 1, 2]
    checked = 0
    for i in range(n):
        if comms[i] == own[48 * i:48 * i + 48]:
            assert cs[i] == per_open[128 * i:128 * i + 128], i
            checked += 1
    assert checked == n - 3   # all but the other, the malformed and the coset-agreeing commitment


# ---------------------------------------------------------------- 5. batch forms
@pytest.mark.parametrize("n", [1, 2, 8, 9, 33, 257])
def test_batch_sizes(vec_ctx, n, monkeypatch):
    blobs = rand_blobs(n, 1000 + n)
    comms, proofs = honest(vec_ctx, blobs)
    assert run(vec_ctx, blobs, comms, proofs) == expect(n)
    items, cells = {n - 1: 1}, {(n - 1, 127): 1}
    proofs[n - 1][127] = proofs[n - 1][126]
    if n > 1:
        proofs[0][0] = off_curve()
        items[0], cells[(0, 0)] = 2, 2
    assert run(vec_ctx, blobs, comms, proofs) == expect(n, items, cells)


_CHUNKED = """
import json, sys
sys.path.insert(0, %r)
import __graft_entry__ as g
pkg = g.load_package()
from tests.test_gpu_blob_cell_proofs import rand_blobs, honest, run, expect, off_curve
ctx = pkg.DASContext(use_precomp=False)
n = 1031
blobs = rand_blobs(n, 1031)
comms, proofs = honest(ctx, blobs)
assert run(ctx, blobs, comms, proofs) == expect(n)
proofs[0][0] = proofs[0][1]
proofs[511][127] = off_curve()
comms[512] = comms[513]
proofs[1030][64] = proofs[1029][64]
assert run(ctx, blobs, comms, proofs) == expect(n, {0: 1, 511: 2, 512: 1, 1030: 1}, {(0, 0): 1, (511, 127): 2, (1030, 64): 1})
ctx.close()
print("chunked ok")
""" % ROOT


def test_two_chunks_of_512():
    env = dict(os.environ, EKZG_CHUNK="512")
    r = subprocess.run([sys.executable, "-c", _CHUNKED], env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0 and "chunked ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_pinned_and_pageable_inputs_agree(das_ctx, pkg):
    import torch
    n = 40
    blobs = rand_blobs(n, 40)
    comms, proofs = honest(das_ctx, blobs)
    proofs[17][3] = off_subgroup()
    comms[30] = comms[31]
    want = run(das_ctx, blobs, comms, proofs)
    assert want == expect(n, {17: 2, 30: 1}, {(17, 3): 2})
    pinned = lambda b: torch.frombuffer(bytearray(b), dtype=torch.uint8).pin_memory()  # noqa: E731
    h_b, h_c, h_p = pinned(b"".join(blobs)), pinned(b"".join(comms)), pinned(b"".join(b"".join(p) for p in proofs))
    h_st = torch.full((n,), 7, dtype=torch.uint8).pin_memory()
    h_cs = torch.full((n * 128,), 7, dtype=torch.uint8).pin_memory()
    ok = C.c_bool(True)
    lib = pkg.load_library()
    res = lib.eth_kzg_b200_verify_blob_cell_proofs_batch(C.c_void_p(das_ctx.handle), C.c_uint64(n), C.c_void_p(h_b.data_ptr()),
                                                         C.c_void_p(h_c.data_ptr()), C.c_void_p(h_p.data_ptr()), C.c_void_p(h_st.data_ptr()),
                                                         C.c_void_p(h_cs.data_ptr()), C.byref(ok))
    assert res.status == 0
    cs = bytes(h_cs.numpy())
    assert (ok.value, list(h_st.numpy()), [list(cs[128 * i:128 * i + 128]) for i in range(n)]) == want


def test_empty_batch(das_ctx):
    assert das_ctx.verify_blob_cell_proofs_batch(b"", b"", b"", 0) == (True, [], None)
    ok, st, cells = das_ctx.verify_blob_cell_proofs_batch(b"", b"", b"", 0, want_cells=True)
    assert (ok, st, cells) == (True, [], b"")


def test_cell_status_optional(das_ctx):
    blobs = rand_blobs(3, 3)
    comms, proofs = honest(das_ctx, blobs)
    proofs[1][2] = IDENTITY
    flat = (b"".join(blobs), b"".join(comms), b"".join(b"".join(p) for p in proofs))
    assert das_ctx.verify_blob_cell_proofs_batch(*flat, 3) == (False, [0, 1, 0], None)


# ---------------------------------------------------------------- 6. launch shape
def test_launch_shape(vec_ctx):
    blobs, comms, proofs = batch64(vec_ctx)
    flat = (b"".join(blobs), b"".join(comms), b"".join(b"".join(p) for p in proofs))
    names = launched(lambda: vec_ctx.verify_blob_cell_proofs_batch(*flat, N3))
    assert sum("k_compare_blob_proofs" in x for x in names) == 1
    assert not any("k_g1_validate" in x for x in names), sorted(set(names))
    bad = [list(p) for p in proofs]
    bad[10][20] = bad[10][21]
    bad[50][0] = off_curve()
    flat_bad = (flat[0], flat[1], b"".join(b"".join(p) for p in bad))
    names = launched(lambda: vec_ctx.verify_blob_cell_proofs_batch(*flat_bad, N3))
    assert sum("k_compare_blob_proofs" in x for x in names) == 1
    assert sum("k_g1_validate" in x for x in names) == 1


# ---------------------------------------------------------------- 7. concurrency
def test_concurrent_callers(vec_ctx):
    blobs, comms, proofs = batch64(vec_ctx)

    def caller(t):
        lo = 8 * t
        b, c, p = list(blobs[lo:lo + 8]), list(comms[lo:lo + 8]), [list(x) for x in proofs[lo:lo + 8]]
        j = t % 8
        p[j][t] = p[j][(t + 1) % 128]
        items, cells = {j: 1}, {(j, t): 1}
        if t % 2:
            c[(j + 3) % 8] = off_curve()
            items[(j + 3) % 8] = 2
        return run(vec_ctx, b, c, p) == expect(8, items, cells)

    for _ in range(2):
        with concurrent.futures.ThreadPoolExecutor(8) as ex:
            assert all(ex.map(caller, range(8)))


# ---------------------------------------------------------------- 8. multi-device
_MULTI = """
import json, sys
sys.path.insert(0, %r)
import __graft_entry__ as g
pkg = g.load_package()
from tests.test_gpu_blob_cell_proofs import multi_case, run
ctx = pkg.DASContext(use_precomp=False)
print(json.dumps([len(ctx.devices), run(ctx, *multi_case(ctx))]))
ctx.close()
""" % ROOT


def multi_case(ctx):
    from tests.test_gpu_blob_cell_proofs import off_curve
    n = 100
    blobs = rand_blobs(n, 100)
    comms, proofs = honest(ctx, blobs)
    for i in (0, 31, 32, 47, 48, 49, 63, 64, 99):
        proofs[i][i % 128] = proofs[(i + 1) % n][i % 128]
    proofs[50][5] = off_curve()
    comms[64] = comms[65]
    return blobs, comms, proofs


def test_multi_device_shards():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two or more GPUs")
    out = []
    for devices in ("", "all"):
        env = dict(os.environ, EKZG_DEVICES=devices)
        r = subprocess.run([sys.executable, "-c", _MULTI], env=env, capture_output=True, text=True, timeout=1200)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        out.append(json.loads(r.stdout.strip().splitlines()[-1]))
    (d1, single), (dn, multi) = out
    assert d1 == 1 and dn >= 2
    assert multi == single
    assert single[1][50] == 2 and single[1][64] == 1 and single[1][31] == 1
