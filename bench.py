#!/usr/bin/env python
"""bench.py -- the driver-facing benchmark of the fused ABFT-SGEMM hot path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--size n] [--id KERNEL_ID] [--sweep]
                  [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic input: one fused fault-tolerant SGEMM
C = alpha*A*B^T + beta*C (encode pre-pass + tcgen05 kernel with checksum tile-columns, per-tile detect/correct) at
BASELINE.json configs[1]: M=N=K=4096, alpha=1, beta=-1.5 (the reference's timing phase, sgemm.cu:22,234), reference
input distribution (utils/utils.cu:23-31).  Inputs are resident in HBM for `value`; `e2e` runs the same step through
the host-buffer C-ABI call (ftsgemm_run_host) with H2D/D2H inside the timed region.  At N>1 every rank (one process per
GPU, torchrun) owns one C block of a 2-D block-sharded product (A row-panel x B row-panel -> no operand traffic) and the
ranks exchange their device-side fault verdict vectors (ftsgemm_stats_device -> NCCL all-gather, asynchronous, joined
before the timed region ends) every step: weak scaling, value = aggregate GFLOPS over the max-over-ranks time.

The JSON line also carries: `sweep` (N=1: fused ABFT / own plain kernel / cuBLAS-TF32 for M=N=K=1024..16384, the same
number of launches per cell, engines interleaved), `strong` (BASELINE.json configs[4]: ONE 32768^3 product on the P x Q
rank grid, incl. the verdict exchange), `id16` (configs[1] literally: the 128x128x8 tile), `parity` (sampled rows of the
bench's own result against the CPU oracle, outside the timed regions).

--dump-outputs DIR writes C as the last timed step left it, so that two builds can be compared output for output: the inputs
are seeded, so the same arguments give the same inputs on every run.  DIR/C_rows.npy (float32) holds rows of the M x N
result, DIR/C_row_index.npy (float64) which rows: all of them when they fit the budget, else a fixed seeded sample.  All
files together stay within DUMP_BYTES: under torchrun every rank writes C_rows_rank<r>.npy / C_row_index_rank<r>.npy for
its own C block within DUMP_BYTES / world.  (--impl reference has no GPU output to dump and refuses the option.)

--impl reference times the reference's own CPU SGEMM (cpu_gemm, utils/utils.cu:79-89, compiled unmodified into
oracle/_ref/libref_utils.so; falls back to the OpenMP oracle port) on the host cores; rank 0 only.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "fused ABFT SGEMM GFLOPS (2*M*N*K/t) and ABFT overhead % vs cuBLAS-TF32, M=N=K=4096"
README_ABFT_HUGE_4096 = 4005.0  # BASELINE.md section 1 (README.md:53), hardware unspecified
DUMP_BYTES = 32 << 20  # --dump-outputs: at most this much in all ranks' files together (half of C at the default 4096^2)


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"bf16_tflops": float(d["bf16_tflops"]), "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "hbm_gbs": float(d["hbm_gbs"]), "src": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """SM clock, power and throttle reasons DURING the timed region.  The timed region of this benchmark is only a few
    milliseconds, so the sampler polls NVML directly from a thread (~1 kHz) instead of `nvidia-smi -lms` (>= 100 ms
    granularity); it falls back to nvidia-smi if pynvml is unavailable."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index=0):
        self.index, self.samples, self.stop_flag, self.thread, self.nvml = index, [], False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = None
            try:  # NVML enumerates all GPUs of the box, CUDA only the visible ones: match by UUID
                import torch
                uuid = str(torch.cuda.get_device_properties(self.index).uuid)
                uuid = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
                try:
                    self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
                except TypeError:
                    self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
                self.how = "matched by UUID"
            except Exception:
                self.h = None
            if self.h is None:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
                self.how = "NVML index = CUDA index (UUID lookup unavailable)"

            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nvml = None
            return
        self.thread = threading.Thread(target=self._poll, daemon=True)
        self.thread.start()

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)
                pw = n.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                rs = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.time(), sm, pw, rs))
            except Exception:
                pass
            time.sleep(0.0005)

    def stop(self, t0, t1):
        if self.nvml is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        self.stop_flag = True
        self.thread.join(timeout=1.0)
        inside = [x for x in self.samples if t0 <= x[0] <= t1]
        if not inside:  # region shorter than one NVML round trip: nearest samples
            inside = sorted(self.samples, key=lambda x: abs(x[0] - 0.5 * (t0 + t1)))[:3]
        reasons = set()
        for _, _, _, rs in inside:
            for bit, name in self.REASONS.items():
                if rs & bit:
                    reasons.add(name)
        sm = [x[1] for x in inside]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.max_sm,
                "power_w_max": max((x[2] for x in inside), default=None), "samples": len(inside),
                "reasons": sorted(reasons), "how": "pynvml polled from a thread during the timed region; device " + getattr(self, "how", "?")}


def _cpu_port_baseline(n, seconds_target=12.0):
    """OpenMP oracle (port of cpu_gemm's arithmetic) on all host cores, bounded row sample of the n^3 workload."""
    import numpy as np
    from oracle import oracle as O
    A, B, _ = O.make_inputs(min(n, 1024))
    if n > 1024:  # tile the 1024-sized reference-distribution block; content does not affect CPU time
        rng = np.random.default_rng(0)
        A = (rng.integers(-9, 10, n * n) * 0.1).astype(np.float32)
        B = (rng.integers(-9, 10, n * n) * 0.1).astype(np.float32)
    nn = n if n > 1024 else min(n, 1024)
    # chunks of 64 sampled rows (enough for the OpenMP team to reach its steady rate) until the time budget is spent:
    # a one-shot extrapolation from a short probe was off by 2-3x
    chunk = 64
    all_rows = np.linspace(0, nn - 1, min(nn, 4096)).astype(np.int32)
    O.sgemm_nt_rows(nn, nn, nn, 1.0, A, B, 0.0, None, all_rows[:4])  # first touch / thread start-up
    nrows, dt = 0, 0.0
    while dt < seconds_target and nrows < len(all_rows):
        rows = all_rows[nrows:nrows + chunk]
        t0 = time.time()
        O.sgemm_nt_rows(nn, nn, nn, 1.0, A, B, 0.0, None, rows)
        dt += time.time() - t0
        nrows += len(rows)
    gf = 2.0 * nrows * nn * nn / dt / 1e9
    return {"value": round(gf, 3), "unit": "GFLOPS", "cores": O.num_threads(), "kind": "port",
            "sample": f"{nrows} of {nn} rows x {nn} cols x K={nn} (sequential-k fp32, OpenMP over columns), {dt:.1f} s"}


def run_reference_arm(args):
    """The reference's own CPU SGEMM on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    from oracle import oracle as O
    n_ref = 1024  # bounded sample of the 4096^3 workload: cpu_gemm is square, single-threaded, ~4.5 s at n=1024
    r = O.ref_utils()
    A, B, C = O.make_inputs(n_ref)
    X = np.ascontiguousarray(B.reshape(n_ref, n_ref).T).reshape(-1)
    steps, warm = max(1, min(args.steps, 6)), min(args.warmup, 1)
    times = []
    if r is not None:
        # cpu_gemm itself is single-threaded: one independent instance per host thread (ctypes releases the GIL), all on
        # the same inputs, each into its own output; the step's throughput is the aggregate over the instances
        import threading
        cores = max(1, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
        kind = "reference"
        sample = (f"{cores} concurrent instances (one per host thread) of cpu_gemm (utils/utils.cu:79-89, unmodified), n={n_ref} "
                  f"each = {cores}/64 of the 4096^3 flops per step")
        outs = [np.zeros(n_ref * n_ref, np.float32) for _ in range(cores)]

        def one(z):
            r.ref_cpu_gemm(1.0, -1.5, O._p(X), O._p(A), n_ref, O._p(z))

        t_begin = time.time()
        for i in range(warm + steps):
            if times and time.time() - t_begin > 120.0:
                break  # 128 instances take ~38 s per step on the pool's hosts: keep the whole arm within a few minutes
            for z in outs:
                z.fill(0.0)
            ths = [threading.Thread(target=one, args=(z,)) for z in outs]
            t0 = time.time()
            for t in ths:
                t.start()
            for t in ths:
                t.join()
            if i >= warm:
                times.append(time.time() - t0)
    else:
        kind, cores = "port", O.num_threads()
        sample = f"oracle_sgemm_nt (OpenMP port of cpu_gemm) n={n_ref} per step"
        for i in range(warm + steps):
            Z = np.zeros(n_ref * n_ref, np.float32)
            t0 = time.time()
            O.sgemm_nt(n_ref, n_ref, n_ref, 1.0, A, B, -1.5, Z)
            if i >= warm:
                times.append(time.time() - t0)
    dt = sum(times) / len(times)
    instances = cores if kind == "reference" else 1
    gf = instances * 2.0 * n_ref ** 3 / dt / 1e9
    out = {"impl": "reference", "metric": METRIC, "value": round(gf, 4), "unit": "GFLOPS", "n_gpus": args.gpus,
           "steps": len(times), "warmup": warm, "ms_per_step": round(dt * 1e3, 2), "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"reference CPU SGEMM, bounded sample of M=N=K=4096: {sample}", "alpha": 1.0, "beta": -1.5},
           "cpu_baseline": {"value": round(gf, 4), "unit": "GFLOPS", "cores": cores, "kind": kind, "sample": sample},
           "e2e": {"value": round(gf, 4), "unit": "GFLOPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    _emit(out)


_JSON_FD = None


def _claim_stdout():
    """Keep stdout for the ONE JSON line: anything libraries print there (NCCL's version banner under torchrun) goes to
    stderr instead."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    sys.stdout.flush()
    if _JSON_FD is None:
        os.write(1, line)
    else:
        os.write(_JSON_FD, line)


def fill_ref_dist(t, gen):
    """Reference input distribution (utils/utils.cu:23-31: magnitude (rand()%10)*0.1, random sign), in place and chunked
    so that multi-GiB operands need no multi-GiB temporaries."""
    import torch
    n = t.numel()
    step = 1 << 26
    for i in range(0, n, step):
        v = t[i:i + step]
        v.copy_(torch.randint(0, 10, (v.numel(),), generator=gen, device=t.device, dtype=torch.int32))
        v.mul_(0.1)
        sgn = torch.randint(0, 2, (v.numel(),), generator=gen, device=t.device, dtype=torch.int32)
        v.mul_(sgn.float().mul_(2).sub_(1))
    return t


def sample_rows(dC, M, N, budget):
    """Rows of C (column-major M x N on the device) for --dump-outputs: (row index as float64, those rows as float32),
    together at most `budget` bytes."""
    import numpy as np
    import torch
    R = min(M, budget // (4 * N + 8))
    if R < 1:
        raise ValueError(f"--dump-outputs: one row of C ({4 * N} bytes) exceeds the budget of {budget} bytes")
    rows = np.arange(M) if R == M else np.sort(np.random.default_rng(0).choice(M, R, replace=False))
    got = dC.view(N, M).t()[torch.from_numpy(rows).to(dC.device)].cpu().numpy()
    return rows.astype(np.float64), got


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    # defaults = the regime every number in DESIGN.md / profiles is quoted in (and the driver's): 20 back-to-back launches at
    # boost clocks.  Hundreds of steps heat the chip: the comparator measured after the headline then reads 15-20 % lower than
    # the one before, and averaged "overhead" figures are meaningless (VERDICT r1).
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--size", type=int, default=4096, help="M=N=K of the block each GPU computes (weak scaling)")
    ap.add_argument("--global-size", type=int, default=0,
                    help="G > 0: the headline itself is ONE G^3 product sharded over the P x Q rank grid (strong scaling)")
    ap.add_argument("--strong-size", type=int, default=32768,
                    help="G of the `strong` sub-record (BASELINE.json configs[4]; 0 = skip)")
    ap.add_argument("--id", type=int, default=31, help="fused ABFT kernel id (31 = 256x256 CTA-pair tile, 16 = literal huge 128x128)")
    ap.add_argument("--no-sweep", action="store_true", help="skip the 1024..16384 sweep (N=1)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write C of the last timed step to DIR (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs dumps the GPU path's C; --impl reference has none")
    if args.impl == "reference":
        return run_reference_arm(args)

    import numpy as np
    import torch
    import __graft_entry__ as ge
    pkg = ge.load_package()

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from importlib import import_module
    sharding = import_module("ftsgemm_b200.sharding")
    P, Q = sharding.shard_grid(world)
    alpha, beta = 1.0, -1.5
    W = max(args.warmup, 3)
    steps = args.steps
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    ft = pkg.FtSgemm()
    stream = torch.cuda.current_stream().cuda_stream
    opts = pkg.make_opts(stream=stream)
    opts_reuse = pkg.make_opts(stream=stream, reuse_b_checksums=True)
    o_cmp = pkg.make_opts(stream=stream, baseline_host_sync=True)
    names = {k["id"]: k for k in pkg.kernel_table()}
    last_per_rank = []  # device time of every rank in the most recent timed() call

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, nsteps, after=None):
        """nsteps calls between two CUDA events on the launching stream, barrier + synchronize on both sides, MAX over ranks."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        e0.record()
        for _ in range(nsteps):
            fn()
        if after is not None:
            after()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            every = torch.zeros(world, device="cuda", dtype=torch.float64)
            dist.all_gather_into_tensor(every, t)
            last_per_rank[:] = [float(x) for x in every.tolist()]
            ms = max(last_per_rank)  # MAX over ranks
            dist.barrier()
        return ms

    def gflops(M, N, K, ms):
        return 2.0 * M * N * K / (ms * 1e-3) / 1e9

    class Problem:
        """Operands of one block resident in HBM + the engines timed on them."""
        def __init__(self, M, N, K):
            self.M, self.N, self.K = M, N, K
            self.dA = fill_ref_dist(torch.empty(M * K, device="cuda"), g)
            self.dB = fill_ref_dist(torch.empty(N * K, device="cuda"), g)
            self.dC = torch.zeros(M * N, device="cuda")

        def run(self, kid, o):
            ft.run(kid, self.M, self.N, self.K, self.dA, self.dB, self.dC, alpha, beta, o)

        def time_engine(self, kid, nsteps, o=None, warm=2):
            o = o or o_cmp
            self.dC.zero_()
            for _ in range(warm):
                self.run(kid, o)
            ms = timed(lambda: self.run(kid, o), nsteps) / nsteps
            return gflops(self.M, self.N, self.K, ms)

    # ------------------------------------------------------------------ headline problem
    n = args.size
    M = N = K = n
    if args.global_size > 0:
        G = args.global_size
        if G % (P * 256) or G % (Q * 256):
            raise SystemExit("--global-size must be a multiple of 256 * the rank grid")
        M, N, K = G // P, G // Q, G
    prob = Problem(M, N, K)
    flops_per_step = 2.0 * M * N * K
    plain_id = {31: 21, 32: 22}.get(args.id, args.id - 10)

    # the one exchange step of the sharded path: every rank's verdict vector to every rank.  Default: FUSED into the GEMM
    # kernel (its last CTA stores the vector into every rank's mailbox over NVLink peer memory; sharding.PeerVerdict);
    # fallback when CUDA IPC is unavailable: snapshot kernel + asynchronous NCCL all-gather (sharding.VerdictExchange)
    exch, peer = None, None
    if dist is not None:
        mode = os.environ.get("FTSGEMM_BENCH_EXCHANGE", "fused")  # fused | nccl | none (none: experiments only)
        if mode == "fused":
            try:
                peer = sharding.PeerVerdict(ft, dist)  # (succeeds or raises on ALL ranks together)
            except Exception as e:  # noqa: BLE001
                sys.stderr.write(f"[bench] rank {rank}: {e}; using the NCCL all-gather\n")
                peer = None
        if peer is None and mode != "none":
            exch = sharding.VerdictExchange(lambda buf: ft.stats_device(buf, stream), dist, dev)

    def step_ft():
        prob.run(args.id, opts)
        if exch is not None:
            exch.step()

    comp = {}
    cublas_before = prob.time_engine(7, steps)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    prob.dC.zero_()
    for _ in range(W):  # warm-up directly in front of the timed region (the clocks ramp down during any idle gap)
        step_ft()
    if exch is not None:
        exch.join()
    ft.stats()  # counters from here on belong to the timed region
    launches0 = ft.launch_count()
    t_wall0 = time.time()
    ms_total = timed(step_ft, steps, after=(exch.join if exch is not None else None))
    gpu_launches = ft.launch_count() - launches0
    ms_per_rank = [round(x / steps, 4) for x in last_per_rank]
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    verdict = exch.verdict() if exch is not None else (peer.verdict() if peer is not None else None)
    st = ft.stats()
    dump = sample_rows(prob.dC, M, N, DUMP_BYTES // world) if args.dump_outputs else None  # (the comparators below overwrite C)
    ms_step = ms_total / steps
    value = world * flops_per_step / (ms_step * 1e-3) / 1e9
    comp["plain"] = prob.time_engine(plain_id, steps)
    cublas_after = prob.time_engine(7, steps)
    comp["cublas_tf32"] = 0.5 * (cublas_before + cublas_after)
    # dominant kernel alone (checksum vectors reused -> no encode launch), same event method
    k_gf = prob.time_engine(args.id, steps, o=opts_reuse)
    k_ms = flops_per_step / (k_gf * 1e9) * 1e3
    for name, kid, reps in (("cublas_fp32", 0, 5), ("abft_baseline_tf32", 30, 2), ("abft_baseline", 10, 2)):
        comp[name] = prob.time_engine(kid, reps, warm=1)
    ft.stats()
    expected_rows = steps * M * (-(-N // names[args.id]["tile"][1]))
    if st["rows_checked"] != expected_rows:
        raise SystemExit(f"rank {rank}: rows_checked {st['rows_checked']} != {expected_rows}: the ABFT check did not run on every tile")
    if verdict is not None and verdict["rows_checked"] != world * expected_rows:
        raise SystemExit(f"verdict exchange: world-summed rows_checked {verdict['rows_checked']} != {world * expected_rows}")

    # ------------------------------------------------------------------ BASELINE.json configs[1] literally: id 16 (128x128x8)
    id16 = None
    if args.id != 16 and args.global_size == 0:
        s16 = min(steps, 50)
        id16 = {"abft_kernel_huge_gflops": round(prob.time_engine(16, s16, o=opts), 1),
                "kernel_sgemm_huge_gflops": round(prob.time_engine(6, s16), 1), "steps": s16,
                "note": "BASELINE.json configs[1] literally (tile 128x128, one CTA per tile); the headline uses the CTA-pair tile 256x256"}
        id16["overhead_pct_vs_cublas_tf32"] = round(100.0 * (comp["cublas_tf32"] / id16["abft_kernel_huge_gflops"] - 1.0), 2)
        ft.stats()

    # ------------------------------------------------------------------ the two optional modes of the same path, same buffers
    modes = None
    if args.global_size == 0:
        s_m = min(steps, 10)
        modes = {"steps": s_m,
                 "x3_fp32_grade_gflops": round(prob.time_engine(args.id, s_m, o=pkg.make_opts(stream=stream, precision=1)), 1),
                 "check_segments_4_gflops": round(prob.time_engine(args.id, s_m, o=pkg.make_opts(stream=stream, check_segments=4)), 1),
                 "protect_epilogue_gflops": round(prob.time_engine(args.id, s_m, o=pkg.make_opts(stream=stream, protect_epilogue=True)), 1),
                 "note": "opts.precision = 1: 3xTF32, three fault-tolerant passes (element-wise FP32 parity); opts.check_segments = 4: "
                         "intra-K checking, four verified K-segments (reference cadence: K/20, ft_sgemm_huge.cuh:324); "
                         "opts.protect_epilogue = 1: checked store pass (the reference's epilogue, ft_sgemm_huge.cuh:573-690, is unprotected)"}
        ft.stats()

    # ------------------------------------------------------------------ parity of the bench's own result (outside timing)
    parity = None
    if rank == 0:
        from oracle import oracle as O
        hA, hB = prob.dA.cpu().numpy(), prob.dB.cpu().numpy()
        prob.dC.zero_()
        ft.run(args.id, M, N, K, prob.dA, prob.dB, prob.dC, 1.0, 0.0, opts)
        got = prob.dC.cpu().numpy().reshape(N, M).T  # column-major M x N -> [m, n]
        rows = np.linspace(0, M - 1, 24 if K <= 8192 else 6).astype(np.int32)
        want = O.sgemm_nt_rows(M, N, K, 1.0, hA, hB, 0.0, None, rows)
        num = float(np.sum((want.astype(np.float64) - got[rows].astype(np.float64)) ** 2))
        den = float(np.sum(want.astype(np.float64) ** 2))
        parity = {"rel_fro": float(np.sqrt(num / den)), "rows": int(len(rows)), "cols": int(N), "K": int(K), "tolerance": 1e-3,
                  "oracle": "oracle_sgemm_nt_rows (port of cpu_gemm, utils/utils.cu:79-89: sequential-k fp32)",
                  "ok": bool(np.sqrt(num / den) < 1e-3)}
        if not parity["ok"]:
            raise SystemExit(f"parity check failed: {parity}")
        del hA, hB
    ft.stats()

    # ------------------------------------------------------------------ e2e: host buffers through the C ABI
    hA = torch.empty(M * K, dtype=torch.float32).pin_memory(); hA.copy_(prob.dA)
    hB = torch.empty(N * K, dtype=torch.float32).pin_memory(); hB.copy_(prob.dB)
    hC = torch.zeros(M * N, dtype=torch.float32).pin_memory()
    e2e_steps = max(3, min(steps, 8))

    def step_e2e():
        ft.run_host(args.id, M, N, K, hA.data_ptr(), hB.data_ptr(), hC.data_ptr(), alpha, beta, opts)
        if exch is not None:
            exch.step()

    step_e2e()
    hC.zero_()
    e2e_ms = timed(step_e2e, e2e_steps, after=(exch.join if exch is not None else None)) / e2e_steps
    e2e_val = world * flops_per_step / (e2e_ms * 1e-3) / 1e9
    result_ok = bool(torch.isfinite(hC).all())
    del hA, hB, hC
    ft.stats()

    # ------------------------------------------------------------------ sweep 1024..16384 (N = 1)
    sweep = None
    if world == 1 and not args.no_sweep and args.global_size == 0:
        del prob
        torch.cuda.empty_cache()
        sweep = []
        cell = min(steps, 20)
        big = Problem(16384, 16384, 16384)
        for s in range(1024, 16385, 1024):
            sub = Problem.__new__(Problem)
            sub.M = sub.N = sub.K = s
            sub.dA, sub.dB, sub.dC = big.dA, big.dB, big.dC
            res = {"abft": [], "plain": [], "cublas_tf32": []}
            for _ in range(3):  # engines interleaved, idle gaps in between: every cell in the same clock state
                # ids 40 / 20: the library's per-shape choice (ftsgemm_select_kernel): 256x256 pair tile from 1536 / 2048 on
                for key, kid, o in (("cublas_tf32", 7, o_cmp), ("abft", pkg.ID_ABFT_AUTO, opts), ("plain", pkg.ID_SGEMM_AUTO, o_cmp)):
                    time.sleep(0.02)
                    res[key].append(sub.time_engine(kid, cell, o=o, warm=3))
            med = {k: statistics.median(v) for k, v in res.items()}
            sweep.append({"n": s, "abft_id": pkg.select_kernel(s, s, s, True), "plain_id": pkg.select_kernel(s, s, s, False),
                          "steps": cell, "abft_gflops": round(med["abft"], 1),
                          "plain_gflops": round(med["plain"], 1), "cublas_tf32_gflops": round(med["cublas_tf32"], 1),
                          "overhead_pct_vs_cublas_tf32": round(100.0 * (med["cublas_tf32"] / med["abft"] - 1.0), 2),
                          "overhead_pct_vs_own_plain_kernel": round(100.0 * (med["plain"] / med["abft"] - 1.0), 2)})
        ft.stats()
        del big, sub
        torch.cuda.empty_cache()
    else:
        del prob
        torch.cuda.empty_cache()

    # ------------------------------------------------------------------ strong: ONE G^3 product on the P x Q rank grid
    strong = None
    G = args.strong_size
    if G > 0 and G % (P * 256) == 0 and G % (Q * 256) == 0 and args.global_size == 0:
        Ms, Ns, Ks = G // P, G // Q, G
        need = 4.0 * (Ms * Ks + Ns * Ks + Ms * Ns)
        if need < 0.8 * torch.cuda.get_device_properties(local_rank).total_memory:
            sp = Problem(Ms, Ns, Ks)
            s_steps = 3

            def step_strong():
                sp.run(args.id, opts)
                if exch is not None:
                    exch.step()

            ft.stats()
            cb = sp.time_engine(7, s_steps, warm=1)
            sp.dC.zero_()
            step_strong()
            s_ms = timed(step_strong, s_steps, after=(exch.join if exch is not None else None)) / s_steps
            sv = exch.verdict() if exch is not None else (peer.verdict() if peer is not None else None)
            s_st = ft.stats()
            s_plain = sp.time_engine(plain_id, s_steps, warm=1)
            ca = sp.time_engine(7, s_steps, warm=1)
            s_val = 2.0 * G ** 3 / (s_ms * 1e-3) / 1e9
            cub = 0.5 * (cb + ca)
            strong = {"global_size": G, "grid": [P, Q], "block": [Ms, Ns, Ks], "steps": s_steps, "ms_per_step": round(s_ms, 3),
                      "value": round(s_val, 1), "unit": "GFLOPS", "per_gpu_gflops": round(s_val / world, 1),
                      "cublas_tf32_gflops_same_block": round(cub, 1), "plain_kernel_gflops_same_block": round(s_plain, 1),
                      "overhead_pct_vs_cublas_tf32": round(100.0 * (cub / (s_val / world) - 1.0), 2),
                      "roofline_frac": round(s_val / world / 1e3 / (_peaks()["bf16_tflops"] / 2.0), 4),
                      "rows_checked": (sv or s_st)["rows_checked"], "detected": (sv or s_st)["detected"],
                      "includes": "encode + checksum GEMM + check + GEMM, one launch" + (
                          (" + verdict exchange fused into the kernel (peer stores over NVLink)" if peer is not None else
                           " + verdict exchange (NCCL all-gather of the device-side vectors)") if world > 1 else "")}
            del sp
            torch.cuda.empty_cache()

    if dump is not None:
        out_dir = Path(args.dump_outputs)
        out_dir.mkdir(parents=True, exist_ok=True)
        sfx = f"_rank{rank}" if world > 1 else ""
        np.save(out_dir / f"C_row_index{sfx}.npy", dump[0])
        np.save(out_dir / f"C_rows{sfx}.npy", dump[1])

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    peaks = _peaks()
    tf32_peak = peaks["bf16_tflops"] / 2.0  # kind::tf32 issues at half the kind::f16 rate on tcgen05
    achieved = flops_per_step / (k_ms * 1e-3) / 1e12
    info = names[args.id]
    region_ms = ms_total
    capped = bool(clocks and "sw_power_cap" in (clocks.get("reasons") or []))
    at_boost = bool(clocks and clocks.get("sm_mhz") and clocks.get("sm_max_mhz") and clocks["sm_mhz"] >= 0.97 * clocks["sm_max_mhz"])
    regime = "power-capped (sw_power_cap sampled)" if capped else ("boost clocks, no throttle reason sampled" if at_boost else "below boost clocks")
    out = {
        "metric": METRIC if (n == 4096 and args.global_size == 0) else
                  METRIC.replace("M=N=K=4096", f"one {args.global_size}^3 product" if args.global_size > 0 else f"M=N=K={n}"),
        "value": round(value, 1), "unit": "GFLOPS", "n_gpus": world, "steps": steps, "warmup": W,
        "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "strong" if args.global_size > 0 else "weak",
        "vs_baseline": round(value / world / README_ABFT_HUGE_4096, 2) if (n == 4096 and args.global_size == 0) else None,
        "dtype": "tf32 multiply, f32 accumulate", "data": "synthetic",
        "config": {"workload": f"fused ABFT SGEMM id {args.id} ({info['name']}, tile {info['tile'][0]}x{info['tile'][1]}), "
                               + (f"one {args.global_size}^3 product, block M={M} N={N} K={K} per GPU" if args.global_size > 0 else f"M=N=K={n} per GPU")
                               + ", alpha=1, beta=-1.5 (sgemm.cu:22,234), reference input distribution",
                   "sharding": (f"{P}x{Q} C-block grid, A/B row-panels resident per GPU; per step every rank's verdict vector reaches "
                                f"every rank: " + ("fused into the GEMM kernel (last CTA stores to every rank's mailbox over NVLink peer "
                                                   "memory, no collective launch)" if peer is not None else
                                                   "snapshot kernel + asynchronous NCCL all-gather, joined inside the timed region"))
                               if world > 1 else "single GPU",
                   "l2": (f"inputs {4 * (M * K + N * K + M * N) / 2**20:.0f} MiB per step vs 126 MB L2: larger than L2, no flush needed"
                          if 4 * (M * K + N * K + M * N) > 160e6 else "L2-resident working set (small size)"),
                   "baseline_note": "vs_baseline = per-GPU value / 4005 GFLOPS (README.md:53 abft_kernel_huge @4096, GPU unspecified)"},
        "abft": {"overhead_pct_vs_cublas_tf32": round(100.0 * (comp["cublas_tf32"] / (value / world) - 1.0), 2),
                 "overhead_pct_vs_own_plain_kernel": round(100.0 * (comp["plain"] / (value / world) - 1.0), 2),
                 "cublas_tf32_gflops": round(comp["cublas_tf32"], 1),
                 "cublas_tf32_gflops_before_after": [round(cublas_before, 1), round(cublas_after, 1)],
                 "comparator_steps": steps, "cublas_fp32_gflops": round(comp["cublas_fp32"], 1),
                 "plain_kernel_gflops": round(comp["plain"], 1), "abft_baseline_gflops": round(comp["abft_baseline"], 1),
                 "abft_baseline_tf32_gflops": round(comp["abft_baseline_tf32"], 1),
                 "encode_us_per_step": round((ms_step - k_ms) * 1e3, 2),
                 "tiles_checked": st["tiles"], "rows_checked": st["rows_checked"], "detected": st["detected"],
                 "max_abs_residual": st["max_abs_residual"], "max_rel_residual": st["max_rel_residual"]},
        "roofline": {"bound": "tensor", "achieved": round(achieved, 1), "peak": round(tf32_peak, 1), "unit": "TFLOP/s",
                     "frac": round(achieved / tf32_peak, 4), "traffic": None,
                     "regime": regime, "timed_region_ms": round(region_ms, 3),
                     "note": f"kernel ftsgemm_tc_kernel alone (checksum vectors reused: no encode launch), 2*M*N*K per launch / "
                             f"CUDA-event mean over {steps} back-to-back launches; peak = bf16 burst {peaks['bf16_tflops']} / 2 "
                             f"(kind::tf32 issues at half the kind::f16 rate; no TF32 peak is measured), {peaks['src']}; "
                             f"clocks during the headline region: {regime}"},
        "e2e": {"value": round(e2e_val, 1), "unit": "GFLOPS", "h2d_bytes_per_step": 4 * (M * K + N * K + M * N), "d2h_bytes_per_step": 4 * M * N,
                "steps": e2e_steps, "finite": result_ok},
        # counted by the library (ftsgemm_launch_count) over the timed region: ftsgemm_tc_kernel with the encode as its front
        # phase (+ stats_vector_kernel per step when the verdict is exchanged)
        "gpu_launches": gpu_launches,
        "clocks": clocks,
        "parity": parity,
    }
    if world > 1:
        out["ms_per_step_per_rank"] = ms_per_rank  # the headline is their maximum
    if verdict is not None:
        out["verdict"] = {k: verdict[k] for k in ("tiles", "rows_checked", "detected", "corrected", "uncorrectable", "clean")}
    if id16 is not None:
        out["id16"] = id16
    if modes is not None:
        out["modes"] = modes
    if sweep is not None:
        out["sweep"] = sweep
    if strong is not None:
        out["strong"] = strong
    tp = ROOT / "profiles" / "traffic.json"
    if tp.exists():
        try:
            t = json.loads(tp.read_text()).get(str(args.id))
            out["roofline"]["traffic"] = t.get(str(n)) if isinstance(t, dict) else (t if n == 4096 else None)
        except Exception:
            pass
    if not args.no_cpu and world == 1:  # (rank 0 at N = 1 only: torchrun pins OMP_NUM_THREADS=1)
        out["cpu_baseline"] = _cpu_port_baseline(n if n <= 4096 else 4096)
    _emit(out)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
