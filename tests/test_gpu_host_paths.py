"""Host paths of the runtime (csrc/kzg_runtime.cu) that the other suites leave out: single-item calls past the coalescer
(EKZG_NO_COALESCE), whose outputs go out through the C ABI's 128 separate pointers from temporary buffers, and pinned
caller memory on the EIP-4844 batch path across chunk boundaries."""
import ctypes as C
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# EKZG_NO_COALESCE is read once per process: the single-item calls run in a child process, against the batch entry points
_UNCOALESCED = """
import sys
sys.path.insert(0, %r)
import __graft_entry__ as g
pkg = g.load_package()
import importlib
syn = importlib.import_module("eth_kzg_b200.synthetic")
ctx = pkg.DASContext(use_precomp=False)
blobs = [syn.blob(1300 + i) for i in range(3)] + [syn.edge_blobs()[3]]
n = len(blobs)
flat = b"".join(blobs)
cells, proofs, st = ctx.compute_cells_and_kzg_proofs_batch(flat, n)
assert st == [0] * n
idx = [list(range(0, 128, 2)), list(range(64, 128)), list(range(1, 128, 2)) + [0], list(range(128))]
idx[2].sort()
rc, rp, rst = ctx.recover_cells_and_kzg_proofs_batch(idx, [[cells[(b * 128 + j) * 2048:(b * 128 + j + 1) * 2048] for j in idx[b]] for b in range(n)])
assert rst == [0] * n and (rc, rp) == (cells, proofs)
for b in range(n):
    want_c = [cells[(b * 128 + j) * 2048:(b * 128 + j + 1) * 2048] for j in range(128)]
    want_p = [proofs[(b * 128 + j) * 48:(b * 128 + j + 1) * 48] for j in range(128)]
    assert ctx.compute_cells_and_kzg_proofs(blobs[b]) == (want_c, want_p), b
    assert ctx.compute_cells(blobs[b]) == want_c, b
    assert ctx.recover_cells_and_kzg_proofs(idx[b], [want_c[j] for j in idx[b]]) == (want_c, want_p), b
ctx.close()
print("uncoalesced ok")
""" % ROOT


def test_uncoalesced_single_item_calls():
    env = dict(os.environ, EKZG_NO_COALESCE="1")
    r = subprocess.run([sys.executable, "-c", _UNCOALESCED], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "uncoalesced ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.fixture
def small_chunks(monkeypatch):
    monkeypatch.setenv("EKZG_CHUNK", "24")
    return 24


def test_pinned_and_pageable_4844_callers_agree(das_ctx, pkg, small_chunks):
    import importlib

    import torch
    syn = importlib.import_module("eth_kzg_b200.synthetic")
    n = 2 * small_chunks + 5                                        # three chunks, the last one ragged
    flat = b"".join(syn.blob(1400 + i) for i in range(n))
    comm, st = das_ctx.blob_to_kzg_commitment_batch(flat, n)        # ctypes string buffers: pageable
    proofs, st2 = das_ctx.compute_blob_kzg_proof_batch(flat, comm, n)
    assert st == [0] * n and st2 == [0] * n
    lib = pkg.load_library()
    pinned = lambda b: torch.frombuffer(bytearray(b), dtype=torch.uint8).pin_memory()  # noqa: E731
    h_in, h_comm = pinned(flat), pinned(comm)
    h_out = torch.empty(n * 48, dtype=torch.uint8).pin_memory()
    h_st = torch.full((n,), 7, dtype=torch.uint8).pin_memory()
    res = lib.eth_kzg_b200_blob_to_kzg_commitment_batch(C.c_void_p(das_ctx.handle), C.c_uint64(n), C.c_void_p(h_in.data_ptr()),
                                                        C.c_void_p(h_out.data_ptr()), C.c_void_p(h_st.data_ptr()))
    assert res.status == 0
    assert bytes(h_out.numpy()) == comm and list(h_st.numpy()) == [0] * n
    h_st.fill_(7)
    res = lib.eth_kzg_b200_compute_blob_kzg_proof_batch(C.c_void_p(das_ctx.handle), C.c_uint64(n), C.c_void_p(h_in.data_ptr()),
                                                        C.c_void_p(h_comm.data_ptr()), C.c_void_p(h_out.data_ptr()), C.c_void_p(h_st.data_ptr()))
    assert res.status == 0
    assert bytes(h_out.numpy()) == proofs and list(h_st.numpy()) == [0] * n
