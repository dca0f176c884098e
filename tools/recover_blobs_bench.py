"""Time of recover_blobs_batch (blobs from their cells, no proofs) against recover_cells_and_kzg_proofs_batch (cells and
proofs), the only other way to rebuild blobs from columns.  Both are called through the C ABI with buffers allocated once, so
neither pays for the Python binding's copies.  Seeded random canonical blobs, 64 of 128 cells erased, either a random 64 per
blob or the same 64 columns for every blob (a PeerDAS node's custody); caller buffers either pinned (torch pin_memory) or
pageable (ctypes).  The production table layout (use_precomp=True).  Per case: one warm-up call of each route, then --reps
rounds that time the two routes alternately on the host clock (every call ends in a device synchronise); medians reported,
with the bytes each route moves each way and the GB/s that gives.  The card's name, power limit and SM clock are read in
the same run.  With --profile-n, a separate torch.profiler run of the new call at that size (random erasure, pinned) sums
its kernel times by name.  Prints one JSON object.

  python tools/recover_blobs_bench.py [--reps 5] [--sizes 1,8,128,256,1024,4096] [--profile-n 1024] [--out result.json]"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BLOB, CELL = 131072, 2048


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def check(lib, res):
    if res.status != 0:
        msg = C.string_at(res.error_msg).decode() if res.error_msg else "error"
        lib.eth_kzg_free_error_message(res.error_msg)
        raise RuntimeError(msg)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sizes", default="1,8,128,256,1024,4096")
    ap.add_argument("--profile-n", type=int, default=0)
    ap.add_argument("--out")
    args = ap.parse_args()
    import numpy as np
    import torch
    import __graft_entry__ as g
    pkg = g.load_package()
    lib = pkg.load_library()
    ctx = pkg.DASContext(use_precomp=True)
    h = C.c_void_p(ctx.handle)
    sizes = [int(x) for x in args.sizes.split(",")]
    N = max(sizes + [args.profile_n])

    raw = np.random.default_rng(7594).integers(0, 256, size=(N, 4096, 32), dtype=np.uint8)
    raw[:, :, 0] &= 0x3F   # canonical
    blobs = raw.tobytes()
    all_cells, _, st = ctx.compute_cells_and_kzg_proofs_batch(blobs, N, want_proofs=False)
    assert st == [0] * N
    all_cells = np.frombuffer(all_cells, dtype=np.uint8).reshape(N, 128, CELL)
    rng = np.random.default_rng(64)
    keep = {"random": np.sort(np.stack([rng.permutation(128)[:64] for _ in range(N)]), axis=1),
            "same_columns": np.tile(np.sort(rng.permutation(128)[:64]), (N, 1))}

    def buffers(n, erasure, pinned):
        k = keep[erasure][:n]
        cells = all_cells[np.arange(n)[:, None], k].reshape(-1)
        counts = (C.c_uint64 * n)(*([64] * n))
        idx = (C.c_uint64 * (64 * n))(*k.reshape(-1).tolist())
        if pinned:
            t = {"cells": torch.from_numpy(cells.copy()).pin_memory(), "blobs": torch.empty(n * BLOB, dtype=torch.uint8).pin_memory(),
                 "ocells": torch.empty(n * 128 * CELL, dtype=torch.uint8).pin_memory(), "oproofs": torch.empty(n * 128 * 48, dtype=torch.uint8).pin_memory()}
            ptr = {name: C.c_void_p(x.data_ptr()) for name, x in t.items()}
        else:
            t = {"cells": C.create_string_buffer(cells.tobytes(), len(cells)), "blobs": C.create_string_buffer(n * BLOB),
                 "ocells": C.create_string_buffer(n * 128 * CELL), "oproofs": C.create_string_buffer(n * 128 * 48)}
            ptr = t
        status = C.create_string_buffer(n)
        return t, ptr, counts, idx, status

    res = {"card (name, power limit, SM clock, max SM clock)": card(), "reps": args.reps, "cases": {}}
    for n in sizes:
        for erasure in ("random", "same_columns"):
            for pinned in (True, False):
                t, p, counts, idx, status = buffers(n, erasure, pinned)

                def new():
                    check(lib, lib.eth_kzg_b200_recover_blobs_batch(h, C.c_uint64(n), counts, idx, p["cells"], p["blobs"], status))

                def old():
                    check(lib, lib.eth_kzg_b200_recover_cells_and_kzg_proofs_batch(h, C.c_uint64(n), counts, idx, p["cells"], p["ocells"],
                                                                                   p["oproofs"], status))

                new()
                old()
                got = bytes(t["blobs"].numpy()) if pinned else t["blobs"].raw
                assert got == blobs[:n * BLOB], "recovered blobs differ (%d, %s)" % (n, erasure)
                tn, to = [], []
                for _ in range(args.reps):
                    for fn, ts in ((new, tn), (old, to)):
                        t0 = time.perf_counter()
                        fn()
                        ts.append((time.perf_counter() - t0) * 1e3)
                a, b = statistics.median(tn), statistics.median(to)
                up = n * 64 * (CELL + 8) + n * 8                       # cells, indices, counts
                down_new, down_old = n * BLOB, n * 128 * (CELL + 48)
                res["cases"]["%d_%s_%s" % (n, erasure, "pinned" if pinned else "pageable")] = {
                    "new_ms": round(a, 3), "proofs_call_ms": round(b, 3), "speedup": round(b / a, 2),
                    "new_blobs_per_s": round(n / a * 1e3, 1), "proofs_call_blobs_per_s": round(n / b * 1e3, 1),
                    "bytes_up": up, "bytes_down_new": down_new, "bytes_down_proofs_call": down_old,
                    "new_GB_per_s": round((up + down_new) / a / 1e6, 2), "proofs_call_GB_per_s": round((up + down_old) / b / 1e6, 2)}
                del t
    if args.profile_n:
        from torch.profiler import ProfilerActivity, profile
        n = args.profile_n
        t, p, counts, idx, status = buffers(n, "random", True)
        check(lib, lib.eth_kzg_b200_recover_blobs_batch(h, C.c_uint64(n), counts, idx, p["cells"], p["blobs"], status))
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            check(lib, lib.eth_kzg_b200_recover_blobs_batch(h, C.c_uint64(n), counts, idx, p["cells"], p["blobs"], status))
            torch.cuda.synchronize()
        with tempfile.TemporaryDirectory() as d:
            path = os.path.join(d, "trace.json")
            prof.export_chrome_trace(path)
            with open(path) as f:
                ev = json.load(f)["traceEvents"]
        kern, copies = {}, {}
        for e in ev:
            if e.get("cat") == "kernel":
                name = e["name"].split("(")[0].split("::")[-1]
                kern[name] = kern.get(name, 0.0) + e["dur"] / 1e3
            elif e.get("cat") == "gpu_memcpy":
                copies[e["name"]] = copies.get(e["name"], 0.0) + e["dur"] / 1e3
        res["profile_%d_random_pinned_ms" % n] = {"kernels": {k: round(v, 3) for k, v in sorted(kern.items())},
                                                  "kernel_sum": round(sum(kern.values()), 3),
                                                  "copies": {k: round(v, 3) for k, v in sorted(copies.items())}}
    ctx.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
