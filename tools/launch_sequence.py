"""Kernel launches of the host entry points, to show that two builds of the library (EKZG_LIB picks one) drive the device
the same way: for each call below, the change of eth_kzg_b200_kernel_launch_count over one call, and the kernel names one
torch.profiler run of the call records, in issue order per stream.  Writes one JSON object; two builds launch the same
kernels when their files are equal.

  EKZG_LIB=path/to/libc_eth_kzg_b200.so python tools/launch_sequence.py --out launches.json

Calls: compute_cells_and_kzg_proofs batch (1, 2, 8, 33, 1024 blobs), the device entry point (1, 1024), recovery batch
(1, 40), blob_to_kzg_commitment batch and compute_blob_kzg_proof batch (1, 40), compute_kzg_proof (1 call, 40 calls), the
verifiers verify_cell_kzg_proof_batch (128 and 16 384 openings) and verify_blob_kzg_proof_batch (1, 20 blobs), and, where the
build has them, the grouped cell verifier and the per-blob verifier on the same inputs (honest, and with one bad item), and
verify_blob_cell_proofs_batch on 20 blobs (honest, and with one bad proof), and recover_blobs_batch (1, 40) on the recovery
batch's inputs.
Each call runs once before it is counted, so first-use allocations are not part of it."""
import argparse
import ctypes as C
import importlib
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def blobs(n, seed):
    """n canonical blobs (every 32-byte element below 2^254)"""
    import numpy as np
    a = np.random.default_rng(seed).integers(0, 256, size=(n, 4096, 32), dtype=np.uint8)
    a[:, :, 0] &= 0x3F
    return a.tobytes()


def kernels(trace_path):
    """kernel names of a chrome trace, per stream in start order; the streams sorted by their sequences"""
    with open(trace_path) as f:
        ev = [e for e in json.load(f)["traceEvents"] if e.get("cat") == "kernel"]
    per_stream = {}
    for e in sorted(ev, key=lambda e: e["ts"]):
        per_stream.setdefault(e["args"].get("stream"), []).append(e["name"])
    return sorted(per_stream.values())


def record(lib, fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    before = lib.eth_kzg_b200_kernel_launch_count()
    fn()
    torch.cuda.synchronize()
    launches = lib.eth_kzg_b200_kernel_launch_count() - before
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        names = kernels(path)
    return {"launches": launches, "kernels": names}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    import torch
    import __graft_entry__ as g
    pkg = g.load_package()
    lib = pkg.load_library()
    ctx = pkg.DASContext(use_precomp=False)
    flat = blobs(1024, 1)
    res = {}

    for n in (1, 2, 8, 33, 1024):
        res["compute_batch_%d" % n] = record(lib, lambda n=n: ctx.compute_cells_and_kzg_proofs_batch(flat[:n * 131072], n))

    d_blobs = torch.frombuffer(bytearray(flat), dtype=torch.uint8).cuda()
    d_cells = torch.empty(1024 * 128 * 2048, dtype=torch.uint8, device="cuda")
    d_proofs = torch.empty(1024 * 128 * 48, dtype=torch.uint8, device="cuda")
    d_status = torch.empty(1024, dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    for n in (1, 1024):
        res["device_%d" % n] = record(lib, lambda n=n: ctx.compute_cells_and_kzg_proofs_device(
            n, d_blobs.data_ptr(), d_cells.data_ptr(), d_proofs.data_ptr(), d_status.data_ptr(), stream))

    cells, _, _ = ctx.compute_cells_and_kzg_proofs_batch(flat[:40 * 131072], 40)
    idx = [list(range(b % 2, 128, 2)) for b in range(40)]
    cl = [[cells[(b * 128 + j) * 2048:(b * 128 + j + 1) * 2048] for j in idx[b]] for b in range(40)]
    for n in (1, 40):
        res["recover_batch_%d" % n] = record(lib, lambda n=n: ctx.recover_cells_and_kzg_proofs_batch(idx[:n], cl[:n]))

    comm, _ = ctx.blob_to_kzg_commitment_batch(flat[:40 * 131072], 40)
    z = bytes(31) + b"\x05"
    for n in (1, 40):
        res["commitment_batch_%d" % n] = record(lib, lambda n=n: ctx.blob_to_kzg_commitment_batch(flat[:n * 131072], n))
        res["blob_proof_batch_%d" % n] = record(lib, lambda n=n: ctx.compute_blob_kzg_proof_batch(flat[:n * 131072], comm[:n * 48], n))
        res["kzg_proof_x%d" % n] = record(lib, lambda n=n: [ctx.compute_kzg_proof(flat[i * 131072:(i + 1) * 131072], z) for i in range(n)])

    nb = 128
    cms, _ = ctx.blob_to_kzg_commitment_batch(flat[:nb * 131072], nb)
    cells, proofs, _ = ctx.compute_cells_and_kzg_proofs_batch(flat[:nb * 131072], nb)
    C = [cms[48 * (k // 128):48 * (k // 128) + 48] for k in range(nb * 128)]
    I = [k % 128 for k in range(nb * 128)]
    CL = [cells[k * 2048:(k + 1) * 2048] for k in range(nb * 128)]
    PR = [proofs[k * 48:(k + 1) * 48] for k in range(nb * 128)]
    bad = list(CL)
    bad[100] = bad[100][:31] + bytes([bad[100][31] ^ 1]) + bad[100][32:]
    bl = [flat[i * 131072:(i + 1) * 131072] for i in range(20)]
    bp, _ = ctx.compute_blob_kzg_proof_batch(flat[:20 * 131072], comm[:20 * 48], 20)
    bcl = [comm[48 * i:48 * i + 48] for i in range(20)]
    bpl = [bp[48 * i:48 * i + 48] for i in range(20)]
    for n in (128, 16384):
        res["verify_cells_%d" % n] = record(lib, lambda n=n: ctx.verify_cell_kzg_proof_batch(C[:n], I[:n], CL[:n], PR[:n]))
    for n in (1, 20):
        res["verify_blobs_%d" % n] = record(lib, lambda n=n: ctx.verify_blob_kzg_proof_batch(bl[:n], bcl[:n], bpl[:n]))
    if hasattr(lib, "eth_kzg_b200_verify_cell_kzg_proof_batch_groups"):
        for name, cl in (("honest", CL), ("one_bad", bad)):
            res["verify_cells_groups_16384_%s" % name] = record(lib, lambda cl=cl: ctx.verify_cell_kzg_proof_batch_groups(C, I, cl, PR, I))
        swapped = bpl[:1] + [bpl[2], bpl[1]] + bpl[3:]
        for name, pl in (("honest", bpl), ("one_bad", swapped)):
            res["verify_blobs_items_20_%s" % name] = record(lib, lambda pl=pl: ctx.verify_blob_kzg_proof_batch_items(bl, bcl, pl))
    if hasattr(lib, "eth_kzg_b200_verify_blob_cell_proofs_batch"):
        cp = proofs[:20 * 128 * 48]
        cp_bad = cp[:48] + cp[2 * 48:3 * 48] + cp[2 * 48:]   # blob 0: the proof of cell 2 in place of cell 1
        for name, p in (("honest", cp), ("one_bad", cp_bad)):
            res["verify_blob_cell_proofs_20_%s" % name] = record(
                lib, lambda p=p: ctx.verify_blob_cell_proofs_batch(flat[:20 * 131072], cms[:20 * 48], p, 20, want_cells=True))
    if hasattr(lib, "eth_kzg_b200_recover_blobs_batch"):
        rcl = [[cells[(b * 128 + j) * 2048:(b * 128 + j + 1) * 2048] for j in idx[b]] for b in range(40)]   # (`cl` was reused above)
        for n in (1, 40):
            res["recover_blobs_batch_%d" % n] = record(lib, lambda n=n: ctx.recover_blobs_batch(idx[:n], rcl[:n]))
    ctx.close()

    with open(args.out, "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)
    for k in sorted(res):
        print("%-22s %5d launches  %s" % (k, res[k]["launches"], [len(s) for s in res[k]["kernels"]]))


if __name__ == "__main__":
    main()
