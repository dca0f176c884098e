"""Time of verify_blob_cell_proofs_batch (recompute every blob's commitment and cell proofs on the device, compare bytes) against
the two-call route it replaces in a blob-pool check: compute the cells of every blob (cells only), then verify_cell_kzg_proof_batch
over all n x 128 openings.  Both routes are called through the C ABI with buffers allocated once, so neither pays for the Python
binding's copies; the two-call route's openings point straight into its cell buffer, as a native caller's would.  Seeded
synthetic blobs, the production table layout (use_precomp=True).  Per case: one warm-up call of each route, then --reps rounds that
time the two routes alternately on the host clock (every call ends in a device synchronise); the medians are reported.  Prints one
JSON object with the card name and power limit read in the same run.

  python tools/blob_cell_proofs_bench.py [--reps 5] [--out result.json]

Cases: honest batches of 1, 8, 128 and 1024 blobs; 1024 blobs with one bad proof."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
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
    ap.add_argument("--out")
    args = ap.parse_args()
    import numpy as np
    import __graft_entry__ as g
    pkg = g.load_package()
    lib = pkg.load_library()
    ctx = pkg.DASContext(use_precomp=True)
    h = C.c_void_p(ctx.handle)

    N = 1024
    raw = np.random.default_rng(7594).integers(0, 256, size=(N, 4096, 32), dtype=np.uint8)
    raw[:, :, 0] &= 0x3F   # canonical
    blobs = C.create_string_buffer(raw.tobytes(), N * 131072)
    comms, st = ctx.blob_to_kzg_commitment_batch(blobs.raw, N)
    _, proofs, st2 = ctx.compute_cells_and_kzg_proofs_batch(blobs.raw, N)
    assert st == [0] * N and st2 == [0] * N
    bad = bytearray(proofs)
    bad[(700 * 128 + 9) * 48:(700 * 128 + 10) * 48] = proofs[(701 * 128 + 9) * 48:(701 * 128 + 10) * 48]
    comm_buf = C.create_string_buffer(comms, N * 48)
    proof_bufs = {"honest": C.create_string_buffer(proofs, len(proofs)), "one_bad_proof": C.create_string_buffer(bytes(bad), len(bad))}

    # two-call route: cells into one buffer, openings as pointer arrays into it and into the proof / commitment buffers
    cells = C.create_string_buffer(N * 128 * 2048)
    status = C.create_string_buffer(N)
    base_c, base_cl = C.addressof(comm_buf), C.addressof(cells)
    c_ptrs = (C.c_void_p * (N * 128))(*[base_c + 48 * (j // 128) for j in range(N * 128)])
    cl_ptrs = (C.c_void_p * (N * 128))(*[base_cl + 2048 * j for j in range(N * 128)])
    p_ptrs = {k: (C.c_void_p * (N * 128))(*[C.addressof(b) + 48 * j for j in range(N * 128)]) for k, b in proof_bufs.items()}
    idx = (C.c_uint64 * (N * 128))(*[j % 128 for j in range(N * 128)])
    item = C.create_string_buffer(N)
    cell_st = C.create_string_buffer(N * 128)

    def new_route(n, which):
        ok = C.c_bool(False)
        check(lib, lib.eth_kzg_b200_verify_blob_cell_proofs_batch(h, C.c_uint64(n), blobs, comm_buf, proof_bufs[which], item, cell_st, C.byref(ok)))
        return ok.value

    def two_calls(n, which):
        check(lib, lib.eth_kzg_b200_compute_cells_and_kzg_proofs_batch(h, C.c_uint64(n), blobs, cells, None, status))
        ok = C.c_bool(False)
        m = C.c_uint64(n * 128)
        check(lib, lib.eth_kzg_verify_cell_kzg_proof_batch(h, m, c_ptrs, m, idx, m, cl_ptrs, m, p_ptrs[which], C.byref(ok)))
        return ok.value

    res = {"card": card(), "reps": args.reps, "cases": {}}
    for n, which in ((1, "honest"), (8, "honest"), (128, "honest"), (1024, "honest"), (1024, "one_bad_proof")):
        verdicts = (new_route(n, which), two_calls(n, which))   # warm-up
        assert verdicts == ((which == "honest"),) * 2, verdicts
        tn, tt = [], []
        for _ in range(args.reps):
            for fn, ts in ((new_route, tn), (two_calls, tt)):
                t0 = time.perf_counter()
                fn(n, which)
                ts.append((time.perf_counter() - t0) * 1e3)
        a, b = statistics.median(tn), statistics.median(tt)
        res["cases"]["%d_%s" % (n, which)] = {"new_ms": round(a, 2), "two_call_ms": round(b, 2), "speedup": round(b / a, 2),
                                              "new_blobs_per_s": round(n / a * 1e3, 1)}
    ctx.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
