#!/usr/bin/env python3
"""Benchmark of the hot path: compute_cells_and_kzg_proofs, blobs/s (BASELINE.json metric, config #3).

  python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle port on the box's host cores

A step = one pass of the hot path over one batch of 1024 synthetic blobs PER GPU (weak scaling: blobs are
independent, every rank works on its own shard, no data-path collective -- SURVEY.md §8e).
  value    : blobs/s with the batch already resident in HBM (device-pointer entry point), CUDA-event timed, max over ranks.
  e2e      : blobs/s through the public host-buffer C-ABI call (eth_kzg_b200_compute_cells_and_kzg_proofs_batch):
             pinned host input -> H2D -> kernels -> D2H -> host output, all inside the timed region.
  roofline : the BINDING view of the dominant kernel (K4, the FK20 MSMs): wide integer multiply-adds per second against
             the IMAD.WIDE issue rate measured in this process at start-up; roofline_hbm is the secondary (non-binding) view.
  strong   : BASELINE config #3 as written -- 1024 blobs IN TOTAL over the N GPUs: every rank computes its 1024/N shard from
             pinned host memory, the results are gathered to rank 0 over NCCL and land in rank 0's host buffer; and the same
             job through ONE process whose DASContext spans the N devices (EKZG_DEVICES), the way a binding would use the box.
  configs  : (N = 1) BASELINE configs #1, #2, #4, #5 at full size with >= 64 items each checked against the CPU oracle;
  abi_single_blob : (N = 1) tools/abi_load.c, 1024 native threads calling the reference's per-blob symbol.
  --dump-outputs DIR : what the timed path (either arm) returned in its last step, as .npy files (see dump_outputs).
Prints ONE JSON line on rank 0."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True      # the benchmark leaves the tree as the build left it (which may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BLOBS_PER_GPU = 1024
BYTES_PER_BLOB = 131072
CELLS_BYTES = 128 * 2048
PROOFS_BYTES = 128 * 48
METRIC = "blobs/sec compute_cells_and_kzg_proofs"

# Work model of OUR algorithm per blob (DESIGN.md §4), in integer multiply-adds on the fmaheavy pipe (what ncu reports as
# sm__pipe_fmaheavy_cycles_active): one 12-limb Montgomery multiplication = 12*(12+12+1) = 300 IMAD.WIDE, one dedicated
# squaring = 78 + 12*13 = 234.
IMAD_MUL, IMAD_SQR = 300, 234
IMAD_WIDE_PEAK_FALLBACK = 9.13e12   # tools/gpu_probe.cu on this pool's B200 (1965 MHz); only used if the in-process probe fails
IMAD_RED = 156                                      # one Montgomery reduction; a*b + c*d fused (fp_mul2_add) saves one
OP_XYZZ_MADD = 8 * IMAD_MUL + 2 * IMAD_SQR - IMAD_RED          # K4: one table entry into an XYZZ accumulator
OP_JAC_DBL = 2 * IMAD_MUL + 5 * IMAD_SQR
OP_JAC_MADD = 7 * IMAD_MUL + 4 * IMAD_SQR
OP_JAC_ADD = 11 * IMAD_MUL + 5 * IMAD_SQR
OP_MADD_ZR = 8 * IMAD_MUL + 3 * IMAD_SQR
DUMP_BYTES = 64 * 10**6             # --dump-outputs: all files together, .npy headers included
DUMP_SEED = 0xB200


def k5_imad_per_blob():
    """exact multiply-add count of the two G1 NTTs of one blob: walks the same (phase, butterfly) list as
    k_fk20_g1_ntts and the op lists of rust-eth-kzg_b200/csrc/twiddle_ops.inc"""
    rows = []
    for ln in open(os.path.join(ROOT, "rust-eth-kzg_b200", "csrc", "twiddle_ops.inc")):
        ln = ln.strip()
        if ln.startswith("{") and len(ln) > 2:
            v = [int(x) for x in ln.strip("{},").split(",")]
            rows.append(v[1:1 + v[0]])
    assert len(rows) == 128
    table = OP_JAC_DBL + (3 * IMAD_MUL + IMAD_SQR) + 7 * OP_MADD_ZR + (27 * IMAD_MUL + 7 * IMAD_SQR) + 8 * IMAD_MUL + 2 * IMAD_MUL
    ladder = [sum((op >> 8) * OP_JAC_DBL + (OP_JAC_MADD if op & 0x20 else 0) for op in r) for r in rows]
    total = heavy = 0
    for ph in range(14):
        mode, st = (1, 13 - ph) if ph >= 7 else (0, ph)
        for t in range(64):
            e = (t & ((1 << st) - 1)) << (6 - st)
            tw = (128 - e) & 127 if mode == 0 else e
            if e:
                total += table + ladder[tw]
                heavy += 1
            if mode == 0:
                total += OP_JAC_ADD * (1 if st == 6 else 2)
            elif st != 6:
                total += 2 * OP_JAC_ADD
    return total, heavy


def synth_blobs(n, first=0):
    import __graft_entry__
    __graft_entry__.load_package()
    import importlib
    syn = importlib.import_module("eth_kzg_b200.synthetic")
    return syn.blobs(n, first)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)"""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


def host_threads():
    """all host threads this process may use -- NOT omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1"""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def workload_config(n):
    """identical in both arms, so that the driver's same_config holds"""
    return {"workload": "compute_cells_and_kzg_proofs, batch of %d synthetic blobs per GPU per step (BASELINE config #3), mainnet trusted setup" % n,
            "blobs_per_gpu_per_step": n,
            "l2": "inputs (%.0f MB) + tables exceed the 126 MB L2; no explicit flush" % (n * BYTES_PER_BLOB / 1e6),
            "sharding": "independent blobs per rank, tables replicated, no collective"}


def dump_outputs(out_dir, n, d_cells, d_proofs, d_status):
    """What one step of the timed path returned for n blobs, one float32 per output byte (exact: bytes are 0..255),
    so that two builds (or the two arms) can be compared file for file on the same synthetic inputs:
      status.npy [n]                      per-blob status (0 = ok)
      proofs.npy [k, 128, 48]             compressed G1 proofs
      cells.npy [k', 128, 2048]           cells
      proofs_blobs.npy, cells_blobs.npy   which blobs (float64 indices): all n, or a fixed seeded sample (sorted) where the
                                          whole output would not fit in DUMP_BYTES; proofs get up to half of it"""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    status = d_status.to(torch.float32).cpu().numpy()
    left = DUMP_BYTES - status.nbytes - 5 * 128               # 128: one .npy header
    for name, rows, share in (("proofs", d_proofs.view(n, 128, 48), 0.5), ("cells", d_cells.view(n, 128, 2048), 1.0)):
        per_blob = 4 * rows[0].numel() + 8                     # its float32 values and its float64 index
        k = min(n, int(left * share) // per_blob)
        idx = np.arange(n) if k == n else np.sort(np.random.default_rng(DUMP_SEED).choice(n, k, replace=False))
        out = rows[torch.from_numpy(idx).to(rows.device)].to(torch.float32).cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), out)
        np.save(os.path.join(out_dir, name + "_blobs.npy"), idx.astype(np.float64))
        left -= out.nbytes + 8 * k
    np.save(os.path.join(out_dir, "status.npy"), status)


def port_note():
    return ("C restatement of the reference algorithm (oracle/, 64-bit limbs + __int128, no assembly); the Rust/blst reference cannot be built in this "
            "image (no cargo).  fp_mul_ns is this port's measured Montgomery multiplication on one core of this box; blst's assembly is ~25-30 ns "
            "on current x86 cores, so divide the GPU/CPU ratio by about fp_mul_ns/28 to estimate the distance to the real reference")


def cpu_baseline(sample_blobs, threads=0):
    """the oracle port (oracle/src/kzg.c, the reference's algorithm restated in C + OpenMP) on the host cores"""
    from oracle import cref
    cref.build()
    nthreads = threads or host_threads()
    blobs = synth_blobs(sample_blobs)
    cref.compute_cells_and_kzg_proofs_batch(blobs[:BYTES_PER_BLOB * min(2, sample_blobs)], min(2, sample_blobs), nthreads)  # builds tables
    t0 = time.perf_counter()
    cref.compute_cells_and_kzg_proofs_batch(blobs, sample_blobs, nthreads)
    dt = time.perf_counter() - t0
    return {"value": sample_blobs / dt, "unit": "blobs/s", "cores": nthreads, "kind": "port",
            "sample": "%d synthetic blobs of the same generator, one blob per OpenMP thread, %.1f s" % (sample_blobs, dt),
            "fp_mul_ns": cref.time_fp_mul(), "note": port_note()}


def run_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import cref
    cref.build()
    cores = host_threads()
    n = args.blobs                      # the same 1024 blobs per step as the GPU arm
    blobs = synth_blobs(n)
    cref.compute_cells_and_kzg_proofs_batch(blobs[:BYTES_PER_BLOB], 1, cores)   # builds the tables
    # keep the whole run inside the driver's limit whatever K and W are: probe the rate on 2 blobs per thread; if K + W
    # full steps would take more than ~15 minutes, the step shrinks (and the config line says so)
    t0 = time.perf_counter()
    cref.compute_cells_and_kzg_proofs_batch(blobs, min(n, 2 * cores), cores)
    rate = min(n, 2 * cores) / (time.perf_counter() - t0)
    budget_s = float(os.environ.get("EKZG_REF_BUDGET_S", "900"))
    per_step = n
    if (args.steps + args.warmup) * n / rate > budget_s:
        per_step = max(cores, int(budget_s * rate / (args.steps + args.warmup)) // cores * cores)
    blobs = blobs[:per_step * BYTES_PER_BLOB]
    for _ in range(args.warmup):
        cref.compute_cells_and_kzg_proofs_batch(blobs, per_step, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = cref.compute_cells_and_kzg_proofs_batch(blobs, per_step, cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        import torch
        cells, proofs = (torch.frombuffer(bytearray(b), dtype=torch.uint8) for b in out)
        dump_outputs(args.dump_outputs, per_step, cells, proofs, torch.zeros(per_step, dtype=torch.int32))
    v = per_step * args.steps / dt
    cfg = workload_config(n)
    if per_step != n:
        cfg["reference_step_shrunk_to"] = per_step
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "blobs/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64 limbs (Fp 6x64, Fr 4x64 Montgomery)", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": "blobs/s", "cores": cores, "kind": "port", "sample": "%d blobs x %d steps" % (per_step, args.steps),
                             "fp_mul_ns": cref.time_fp_mul(), "note": port_note()},
            "e2e": {"value": v, "unit": "blobs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def strong_scaling(args, ctx, pkg, rank, world, local_rank):
    """BASELINE config #3 as written: args.blobs blobs IN TOTAL over the `world` GPUs, results gathered to rank 0's host memory.
    Returns (ms per step as max over ranks, blobs) -- every rank calls it."""
    import torch
    import torch.distributed as dist
    import importlib
    sh = importlib.import_module("eth_kzg_b200.sharding")
    n = args.blobs
    lo, cnt = sh.shard_bounds(n, world, rank)
    counts = [sh.shard_bounds(n, world, r)[1] for r in range(world)]
    mx = max(counts)
    h_in = torch.frombuffer(bytearray(synth_blobs(cnt, first=lo)), dtype=torch.uint8).pin_memory()   # this rank's shard of THE batch
    d_in = torch.empty(mx * BYTES_PER_BLOB, dtype=torch.uint8, device="cuda")
    d_cells = torch.empty((mx, CELLS_BYTES), dtype=torch.uint8, device="cuda")
    d_proofs = torch.empty((mx, PROOFS_BYTES), dtype=torch.uint8, device="cuda")
    d_status = torch.zeros(mx, dtype=torch.int32, device="cuda")
    h_cells = torch.empty((n, CELLS_BYTES), dtype=torch.uint8).pin_memory() if rank == 0 else None
    h_proofs = torch.empty((n, PROOFS_BYTES), dtype=torch.uint8).pin_memory() if rank == 0 else None
    stream = torch.cuda.current_stream()

    def step():
        d_in[:cnt * BYTES_PER_BLOB].copy_(h_in, non_blocking=True)
        ctx.compute_cells_and_kzg_proofs_device(cnt, d_in.data_ptr(), d_cells.data_ptr(), d_proofs.data_ptr(), d_status.data_ptr(), stream.cuda_stream)
        g_cells = sh.gather_rows(d_cells[:cnt], counts)
        g_proofs = sh.gather_rows(d_proofs[:cnt], counts)
        if rank == 0:
            h_cells.copy_(g_cells, non_blocking=True)
            h_proofs.copy_(g_proofs, non_blocking=True)

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1000 / args.steps
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    check = None
    if rank == 0:
        # the gathered batch equals what one device computes for blobs 0..n-1 (first and last blob of every shard checked)
        probe = sorted({b for r in range(world) for b in (sh.shard_bounds(n, world, r)[0], sum(sh.shard_bounds(n, world, r)) - 1)})
        bad = []
        for b in probe:
            c, p, st = ctx.compute_cells_and_kzg_proofs_batch(synth_blobs(1, first=b), 1)
            if not (bytes(h_cells[b].numpy()) == c and bytes(h_proofs[b].numpy()) == p):
                bad.append(b)
        # a mismatch is reported in the line (shards_checked < 0), not raised: the other ranks are already past their collectives
        check = len(probe) if not bad else -len(bad)
    return float(t[0]), n, check


def one_process_multi_device(args, pkg, world):
    """the whole box behind ONE DASContext (EKZG_DEVICES): what a Go/C#/Nim/JVM binding gets from eth_kzg_das_context_new.
    Rank 0 only, after every rank has released its own context."""
    import torch
    os.environ["EKZG_DEVICES"] = ",".join(str(i) for i in range(world))
    t0 = time.perf_counter()
    ctx = pkg.DASContext(use_precomp=bool(args.precomp))
    t_init = time.perf_counter() - t0
    lib = pkg.load_library()
    out = {"devices": ctx.devices, "context_init_s": t_init, "fk20_window_bits": ctx.window}
    for label, n in (("strong", args.blobs), ("weak", args.blobs * world)):
        h_in = torch.frombuffer(bytearray(synth_blobs(n)), dtype=torch.uint8).pin_memory()
        h_cells = torch.empty(n * CELLS_BYTES, dtype=torch.uint8).pin_memory()
        h_proofs = torch.empty(n * PROOFS_BYTES, dtype=torch.uint8).pin_memory()
        h_status = torch.zeros(n, dtype=torch.uint8).pin_memory()

        def step():
            res = lib.eth_kzg_b200_compute_cells_and_kzg_proofs_batch(ctypes.c_void_p(ctx.handle), ctypes.c_uint64(n), ctypes.c_void_p(h_in.data_ptr()),
                                                                      ctypes.c_void_p(h_cells.data_ptr()), ctypes.c_void_p(h_proofs.data_ptr()),
                                                                      ctypes.c_void_p(h_status.data_ptr()))
            assert res.status == 0
        for _ in range(3):
            step()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step()
        ms = (time.perf_counter() - t0) * 1000 / args.steps
        out[label] = {"blobs_total": n, "ms_per_step": ms, "value": n / (ms / 1000), "unit": "blobs/s"}
        del h_in, h_cells, h_proofs, h_status
    ctx.close()
    del os.environ["EKZG_DEVICES"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--blobs", type=int, default=BLOBS_PER_GPU, help="blobs per GPU per step")
    ap.add_argument("--precomp", type=int, default=1, help="use_precomp flag of the context (window from EKZG_FK20_WINDOW)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline only: skip configs / latency / abi_single_blob / one-process multi-device")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step (rank 0's blobs) to DIR/*.npy, at most 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        # host-side barrier for the one-process measurement at the end: an NCCL barrier would leave a spinning kernel of the
        # waiting ranks' processes on their GPUs, and two processes time-slice a GPU (measured: 2.4x slower shards)
        host_group = dist.new_group(backend="gloo")
    import __graft_entry__
    pkg = __graft_entry__.load_package()
    t_init = time.perf_counter()
    ctx = pkg.DASContext(use_precomp=bool(args.precomp))
    t_init = time.perf_counter() - t_init
    lib0 = pkg.load_library()
    # the roofline denominator, measured here and now on this device at its current clock
    imad_peak = ctx.probe_imad_wide()
    peak_source = "in-process probe at start-up (csrc/kzg_probe.cu: carry-chained IMAD.WIDE.U32.X on every SM)"
    if not imad_peak or imad_peak < 1e12:
        imad_peak, peak_source = IMAD_WIDE_PEAK_FALLBACK, "fallback constant (tools/gpu_probe.cu, profiles/r1_gpu_probe.json): the in-process probe failed"
    n = args.blobs
    # this rank's shard of the job: independent blobs, different on every rank
    host_blobs = synth_blobs(n, first=rank * n)
    h_in = torch.frombuffer(bytearray(host_blobs), dtype=torch.uint8).pin_memory()
    d_in = h_in.cuda()
    d_cells = torch.empty(n * CELLS_BYTES, dtype=torch.uint8, device="cuda")
    d_proofs = torch.empty(n * PROOFS_BYTES, dtype=torch.uint8, device="cuda")
    d_status = torch.zeros(n, dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream()

    def device_step():
        ctx.compute_cells_and_kzg_proofs_device(n, d_in.data_ptr(), d_cells.data_ptr(), d_proofs.data_ptr(), d_status.data_ptr(), stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        device_step()
    barrier()
    assert int(d_status.sum().item()) == 0
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ctx.set_profiling(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    launches0 = lib0.eth_kzg_b200_kernel_launch_count()
    e0.record(stream)
    for _ in range(args.steps):
        device_step()
    e1.record(stream)
    barrier()
    dev_ms = e0.elapsed_time(e1)
    launches = int(lib0.eth_kzg_b200_kernel_launch_count() - launches0)
    nb, stage_ms = ctx.collect_stage_times()
    ctx.set_profiling(False)

    # end to end through the host-buffer ABI call: pinned input, H2D + kernels + D2H inside the timed region
    lib = pkg.load_library()
    h_cells = torch.empty(n * CELLS_BYTES, dtype=torch.uint8).pin_memory()
    h_proofs = torch.empty(n * PROOFS_BYTES, dtype=torch.uint8).pin_memory()
    h_status = torch.zeros(n, dtype=torch.uint8).pin_memory()

    def e2e_step():
        res = lib.eth_kzg_b200_compute_cells_and_kzg_proofs_batch(ctypes.c_void_p(ctx.handle), ctypes.c_uint64(n), ctypes.c_void_p(h_in.data_ptr()),
                                                                  ctypes.c_void_p(h_cells.data_ptr()), ctypes.c_void_p(h_proofs.data_ptr()),
                                                                  ctypes.c_void_p(h_status.data_ptr()))
        assert res.status == 0

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1000
    clocks = sampler.stop() if rank == 0 else None
    # parity spot check inside the bench: device-resident and host paths agree
    assert torch.equal(h_proofs.cuda(), d_proofs) and torch.equal(h_cells.cuda(), d_cells), "device and host paths disagree"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, n, d_cells, d_proofs, d_status)

    t = torch.tensor([dev_ms, e2e_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = float(t[0]), float(t[1])
    del d_cells, d_proofs, h_cells, h_proofs
    strong_ms, strong_n, strong_checked = strong_scaling(args, ctx, pkg, rank, world, local_rank)

    line = None
    if rank == 0:
        total_blobs = n * world * args.steps
        value = total_blobs / (dev_ms / 1000)
        e2e = total_blobs / (e2e_ms / 1000)
        w, nw = ctx.window, 255 // ctx.window + 1
        # merged top window (MsmTable::mg in csrc/msm_table.cuh): nw - 1 + 1/mg table additions per scalar
        rtop = (1 << (255 - w * (nw - 1))) + 1
        mg = next((m for m in (4, 2) if rtop ** m - 1 <= 1 << (w - 1)), 1)
        adds_per_scalar = nw - 1 + 1.0 / mg
        names = ["K1_blob_to_coeffs_cells", "K2_toeplitz_scalars", "K4_fk20_msm", "K5_g1_ntt", "K6_compress"]
        stages = {nm: ms / max(nb, 1) for nm, ms in zip(names, stage_ms)}
        tot = sum(stages.values()) or 1.0
        msm_ms = stages["K4_fk20_msm"]
        # the work model is the XYZZ kernel's (8M + 2S per table addition): a kernel form that needs fewer multiply-adds per addition
        # (EKZG_K4=b, batched affine) shows up as a higher fraction of the same model, i.e. as useful work per second
        msm_imad = int(n * 128 * 64 * adds_per_scalar * OP_XYZZ_MADD)
        k5_imad, k5_heavy = k5_imad_per_blob()
        ntt_imad = n * k5_imad
        ach = msm_imad / (msm_ms / 1000) if msm_ms else 0.0
        ach5 = ntt_imad / (stages["K5_g1_ntt"] / 1000) if stages["K5_g1_ntt"] else 0.0
        roofline = {"bound": "imad", "kernel": "k_fk20_msm (K4, %s form)" % {"r": "register XYZZ", "a": "batched affine, global scratch", "b": "batched affine, shared memory"}.get(os.environ.get("EKZG_K4", "v")[:1], "shared-memory-operand XYZZ"),
                    "achieved": ach / 1e12, "peak": imad_peak / 1e12, "unit": "T IMAD.WIDE/s", "frac": ach / imad_peak,
                    "peak_source": peak_source,
                    # DRAM bytes of that kernel per launch (ncu --set full, profiles/r2_p_prof_k4_k5_raw.csv: 26.97 GB read + 0.15 GB written at
                    # 1024 blobs, w = 14); the HBM view with the algorithmic bytes is in roofline_hbm
                    "traffic": (27.12e9 * n / 1024 if w == 14 else None), "traffic_unit": "bytes per launch",
                    "algorithmic_imad_per_launch": msm_imad, "kernel_ms": msm_ms,
                    "model": "%d blobs x 8192 scalars x %.2f table additions x %d multiply-adds (XYZZ mixed addition 8M+2S, one fused reduction)" % (n, adds_per_scalar, OP_XYZZ_MADD),
                    "k_fk20_g1_ntts": {"imad_per_launch": ntt_imad, "scalar_muls_per_blob": k5_heavy, "achieved": ach5 / 1e12, "frac": ach5 / imad_peak, "kernel_ms": stages["K5_g1_ntt"]},
                    "whole_step": {"imad": msm_imad + ntt_imad, "frac": (msm_imad + ntt_imad) / (dev_ms / args.steps / 1000) / imad_peak}}
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        msm_bytes = int(n * (128 * 64 * adds_per_scalar * 96 + 128 * 64 * 32 + 128 * 144))
        hbm_ach = msm_bytes / (msm_ms / 1000) / 1e9 if msm_ms else 0.0
        traffic = 27.12e9 * n / 1024 if w == 14 else None
        roofline_hbm = {"bound": "hbm (NOT binding)", "kernel": "k_fk20_msm", "achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                        "algorithmic_bytes": msm_bytes, "traffic": traffic, "traffic_over_algorithmic": traffic / msm_bytes if traffic else None,
                        "traffic_source": "ncu --set full, dram__bytes_read+write per launch of k_fk20_msm_vm<4> at 1024 blobs, w=14 (profiles/r2_p_prof_k4_k5_raw.csv)",
                        "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback",
                        "note": "1.8x the algorithmic bytes: 96-byte table entries straddle 64-byte DRAM atoms; at ~8 % of HBM peak it costs nothing -- the kernel is bound by the fmaheavy pipe"}
        line = {
            "metric": METRIC, "value": value, "unit": "blobs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32 limbs (Fp 12x32, Fr 8x32 Montgomery, IMAD.WIDE carry chains)", "data": "synthetic",
            "config": workload_config(n),
            "setup": {"fk20_window_bits": w, "srs_window_bits": ctx.srs_window, "fk20_table_gib": ctx.table_bytes / 2**30, "context_init_s": t_init},
            "e2e": {"value": e2e, "unit": "blobs/s", "h2d_bytes_per_step": n * BYTES_PER_BLOB, "d2h_bytes_per_step": n * (CELLS_BYTES + PROOFS_BYTES + 4),
                    "ms_per_step": e2e_ms / args.steps, "api": "eth_kzg_b200_compute_cells_and_kzg_proofs_batch (host buffers)"},
            "gpu_launches": launches,
            "clocks": clocks, "roofline": roofline, "roofline_hbm": roofline_hbm,
            "stages_ms_per_step": stages, "stage_share": {k: v / tot for k, v in stages.items()},
            "strong": {"blobs_total": strong_n, "n_gpus": world, "ms_per_step": strong_ms, "value": strong_n / (strong_ms / 1000), "unit": "blobs/s",
                       "shards_checked": strong_checked,
                       "path": "per rank: pinned host shard -> H2D -> kernels; NCCL gather of cells and proofs to rank 0 -> D2H into rank 0's pinned buffer; host wall clock, max over ranks",
                       "limiter": "K5's dependency chain of fixed-scalar multiplications (7 deep up to 256 blobs per GPU: 10-15 ms; 12 deep above: 17+ ms) whatever the shard size (DESIGN.md §6)"},
        }
    extras = not args.no_extras
    if extras and world == 1:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_configs as bc
        cfgs = {}
        k4, k5 = int(n * 128 * 64 * adds_per_scalar * OP_XYZZ_MADD) // n, k5_imad
        for key, fn in (("1", lambda: bc.latency(ctx, pkg)), ("2", lambda: bc.config2(ctx, pkg, 3, 64, imad_peak)),
                        ("4", lambda: bc.config4(ctx, pkg, 3, 64, imad_peak, k4 + k5)), ("5", lambda: bc.config5(ctx, pkg, 3, 64))):
            try:
                cfgs[key] = fn()
            except Exception as ex:   # a failing side measurement must not hide the headline; it is reported as failed, not dropped
                cfgs[key] = {"failed": repr(ex)[:300]}
        line["configs"] = cfgs
        if "latency_1blob_ms" in cfgs.get("1", {}):
            line["latency_1blob_ms"] = cfgs["1"]["latency_1blob_ms"]
            line["latency_32blob_ms"] = cfgs["1"]["latency_32blob_ms"]
            if "latency_8blob_batch_ms" in cfgs["1"]:
                line["latency_8blob_batch_ms"] = cfgs["1"]["latency_8blob_batch_ms"]
    ctx.close()
    del d_in
    torch.cuda.empty_cache()
    if extras and world > 1:
        torch.cuda.synchronize()
        dist.barrier(group=host_group)      # every rank has released its tables; the other ranks now wait on the HOST
        if rank == 0:
            try:
                line["strong"]["one_process"] = one_process_multi_device(args, pkg, world)
            except Exception as ex:
                line["strong"]["one_process"] = {"failed": repr(ex)[:300]}
        dist.barrier(group=host_group)
    if rank == 0:
        if extras and world == 1:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_configs as bc
            line["abi_single_blob"] = bc.abi_load(threads=1024, calls=16)
        if not args.no_cpu_baseline and world == 1:
            try:
                # bounded sample: ~20 s of CPU work on a 16-thread host (the oracle port does ~3 blobs/s/thread)
                line["cpu_baseline"] = cpu_baseline(int(os.environ.get("EKZG_CPU_SAMPLE", "0")) or 64 * host_threads())
            except Exception as ex:  # the checker failing must not hide the GPU number
                line["cpu_baseline"] = {"value": None, "unit": "blobs/s", "cores": 0, "kind": "port", "sample": "failed: %r" % (ex,)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
