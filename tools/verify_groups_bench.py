"""Time of the verifiers that name the bad items against the plain batch verifiers, on seeded synthetic data: median of
--reps calls after one warm-up call per case, each call timed on the host clock (every call ends in a device synchronise
and returns its verdicts).  Prints one JSON object with the card name and power limit read in the same run.

  python tools/verify_groups_bench.py [--reps 5] [--out result.json]

Cases: 128 blobs x 128 cells (BASELINE config #5) honest through the plain call and through the grouped call with groups =
columns; one corrupted column (groups = columns); 16 scattered bad cells with one group per opening (16 384 groups); every
cell bad (groups = columns); 1024 blobs through verify_blob_kzg_proof_batch and the per-blob call, honest and with one bad
blob."""
import argparse
import json
import os
import random
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


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts), out


def flip(cell, byte=31):
    return cell[:byte] + bytes([cell[byte] ^ 1]) + cell[byte + 1:]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out")
    args = ap.parse_args()
    import __graft_entry__ as g
    import numpy as np
    pkg = g.load_package()
    ctx = pkg.DASContext(use_precomp=True)

    rng = np.random.default_rng(7)
    raw = rng.integers(0, 256, size=(1024, 4096, 32), dtype=np.uint8)
    raw[:, :, 0] &= 0x3F   # canonical
    flat = raw.tobytes()
    nb = 128
    cms, _ = ctx.blob_to_kzg_commitment_batch(flat[:nb * 131072], nb)
    cells, proofs, _ = ctx.compute_cells_and_kzg_proofs_batch(flat[:nb * 131072], nb)
    C = [cms[48 * (k // 128):48 * (k // 128) + 48] for k in range(nb * 128)]
    I = [k % 128 for k in range(nb * 128)]
    CL = [cells[k * 2048:(k + 1) * 2048] for k in range(nb * 128)]
    PR = [proofs[k * 48:(k + 1) * 48] for k in range(nb * 128)]
    cols = list(I)
    res = {"card": card(), "reps": args.reps, "ms": {}}
    ms = res["ms"]

    def cell_case(name, cells_in, groups, plain=False):
        if plain:
            t, out = timed(lambda: ctx.verify_cell_kzg_proof_batch(C, I, cells_in, PR), args.reps)
            ms[name] = {"median_ms": round(t, 2), "verified": out}
        else:
            t, (ok, st) = timed(lambda: ctx.verify_cell_kzg_proof_batch_groups(C, I, cells_in, PR, groups), args.reps)
            ms[name] = {"median_ms": round(t, 2), "all_ok": ok, "groups_1": sum(1 for s in st if s == 1), "groups_2": sum(1 for s in st if s == 2)}

    cell_case("cells_128x128_honest_plain", CL, None, plain=True)
    cell_case("cells_128x128_honest_groups_columns", CL, cols)
    bad_col = list(CL)
    for b in range(nb):
        bad_col[b * 128 + 5] = flip(bad_col[b * 128 + 5])
    cell_case("cells_128x128_one_bad_column_groups_columns", bad_col, cols)
    scattered = list(CL)
    for k in random.Random(3).sample(range(len(CL)), 16):
        scattered[k] = flip(scattered[k])
    cell_case("cells_128x128_16_bad_cells_group_per_opening", scattered, list(range(len(CL))))
    cell_case("cells_128x128_all_bad_groups_columns", [flip(c) for c in CL], cols)

    n = 1024
    bl = [flat[i * 131072:(i + 1) * 131072] for i in range(n)]
    bc, _ = ctx.blob_to_kzg_commitment_batch(flat, n)
    bp, _ = ctx.compute_blob_kzg_proof_batch(flat, bc, n)
    bcl = [bc[48 * i:48 * i + 48] for i in range(n)]
    bpl = [bp[48 * i:48 * i + 48] for i in range(n)]
    bad = list(bpl)
    bad[500] = bpl[501]
    for name, pr in (("honest", bpl), ("one_bad_blob", bad)):
        t, out = timed(lambda: ctx.verify_blob_kzg_proof_batch(bl, bcl, pr), args.reps)
        ms["blobs_1024_%s_plain" % name] = {"median_ms": round(t, 2), "verified": out}
        t, (ok, st) = timed(lambda: ctx.verify_blob_kzg_proof_batch_items(bl, bcl, pr), args.reps)
        ms["blobs_1024_%s_items" % name] = {"median_ms": round(t, 2), "all_ok": ok, "items_1": sum(1 for s in st if s == 1)}
    ctx.close()
    res["honest_groups_over_plain"] = round(ms["cells_128x128_honest_groups_columns"]["median_ms"] / ms["cells_128x128_honest_plain"]["median_ms"], 3)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
