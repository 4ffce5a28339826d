#!/usr/bin/env python
"""bench.py — the measured headline of this repository.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--mnk M_N_K] [--acc fp32|fp16] [--impl ours|reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Metric (BASELINE.json): HGEMM TFLOP/s, offline mode (back-to-back calls), per (M,N,K). One "step" is ONE
GEMM of the workload shape through the C ABI (libb200_hgemm.so). Default workload = BASELINE config[1]:
4096_4096_4096, fp32 accumulate.  Synthetic N(0,1) fp16 operands, as the reference harness draws them
(benchmarking_utils.py:36-37).

What is timed
  value   K steps with operands resident in HBM, CUDA events on the launching (legacy default) stream, bracketed
          by barrier + device synchronize, MAX over ranks; FLOPs = 2*M*N*K per step per rank (unpadded).
          Successive steps rotate over operand sets whose total size exceeds the 126 MB L2 several times.
  e2e     the same GEMM through b200_hgemm_host(): pinned HOST buffers, H2D of A and B + kernel + D2H of C inside
          the timed region every step.
  roofline  achieved = 2MNK / (average kernel duration from the same CUDA events); peak = measured cuBLAS bf16
          burst TFLOP/s from MEASURED_PEAKS.json (fallback 1590, said so in `peak_source`).
  cpu_baseline  the reference's CPU path, verbatim: torch.matmul(a.float(), b.float()).half() on the host cores
          (zero_one_correctness_check.py:87-90), a bounded ~10 s sample of the same shape, rank 0, N=1 only.
  --impl reference   times that same CPU path as the whole job (the reference has no other CPU implementation
          and its GPU kernels target sm_80/sm_90 — see DESIGN.md), K bounded steps, rank 0 only.

  sustained  the same step loop run for ~1 s (the power-capped state a long job lives in), reported beside the burst value.
  sweep   BASELINE config 5: the 1000-shape grid (+ 2048_11008_4096) through the same C ABI, shapes dealt to the ranks
          (one problem per GPU at a time, no collective on the GEMM path). Per shape: the harness metric (host clock
          around one call bracketed by device synchronisation, mean of per-sample TFLOP/s, benchmarking_utils.py:23-31)
          and a CUDA-event-timed back-to-back batch. Aggregate = sum of 2MNK over ALL shapes / max over ranks of the
          rank's summed device time, so it grows with N only if the sharding works.

--dump-outputs DIR  writes C of the last timed step (rank 0) as DIR/c.npy, float32, so that two builds can be compared
          output for output: the operands come from seeded generators, so the same arguments give the same inputs. An
          output of more than DUMP_MAX_ELEMS entries is sampled at positions drawn with a fixed seed (sorted flat
          row-major indices, the same for every run of the shape), which keeps the file under 64 MB.

Multi-GPU: the path shards by problem (one GEMM per GPU, no collective on the data path; SURVEY §8e), so
at N > 1 every rank runs the same per-GPU work ("scaling": "weak") and value is the sum over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

import numpy as np  # noqa: E402
import torch  # noqa: E402

L2_BYTES = 126 * 1024 * 1024
FALLBACK_TFLOPS, FALLBACK_HBM = 1590.0, 6650.0
DUMP_MAX_ELEMS = 1 << 23        # 32 MiB of float32


def positive_int(text: str) -> int:
    v = int(text)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {v}")
    return v


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=positive_int, default=2000, help="timed steps (GEMMs) of the headline value")
    p.add_argument("--warmup", type=int, default=20)
    p.add_argument("--mnk", type=str, default="4096_4096_4096")
    p.add_argument("--acc", type=str, default="fp32", choices=["fp32", "fp16"])
    p.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    p.add_argument("--e2e_steps", type=int, default=0, help="steps of the host-buffer leg (default min(steps, 50))")
    p.add_argument("--cpu_seconds", type=float, default=10.0, help="bound on the cpu_baseline sample")
    p.add_argument("--sustained_seconds", type=float, default=1.0, help="length of the power-capped loop (0 = skip)")
    p.add_argument("--sweep", type=str, default="grid", help="'grid' (1001 shapes), 'none', or a comma list of M_N_K")
    p.add_argument("--sweep_ms", type=float, default=25.0, help="sampling budget per shape of the sweep leg")
    p.add_argument("--cpu_threads", type=int, default=0, help="threads of the CPU arms (0 = half the host's logical CPUs)")
    p.add_argument("--dump-outputs", metavar="DIR", default="",
                   help=f"write C of the last timed step as DIR/c.npy (float32; at most {DUMP_MAX_ELEMS} entries, a fixed "
                        "sample when C is larger)")
    return p.parse_args()


def peaks():
    f = REPO / "MEASURED_PEAKS.json"
    if f.exists():
        try:
            d = json.loads(f.read_text())
            return (float(d["bf16_tflops"]), float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json, cuBLAS bf16 burst)",
                    float(d.get("bf16_tflops_sustained", 0.0)) or None)
        except Exception:
            pass
    return FALLBACK_TFLOPS, FALLBACK_HBM, "fallback (B200_PROFILING.md)", 1400.0


class ClockSampler:
    """SM clock, power and throttle reasons sampled DURING the timed regions, every few milliseconds through NVML
    (nvidia-ml-py) from a background thread; falls back to `nvidia-smi -lms` when NVML cannot be loaded."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index: int):
        self.gpu, self.samples, self.thread, self.stop_flag, self.proc, self.path = gpu_index, [], None, False, None, None
        self.max_mhz = None

    def _physical_index(self) -> int:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.gpu])
            except (ValueError, IndexError):
                pass
        return self.gpu

    def start(self):
        try:
            import threading

            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))

            def loop():
                while not self.stop_flag:
                    try:
                        self.samples.append((float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)),
                                             nv.nvmlDeviceGetPowerUsage(h) / 1000.0,
                                             int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))))
                    except Exception:
                        pass
                    time.sleep(0.004)
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        exe = shutil.which("nvidia-smi")
        if not exe:
            return
        fd, self.path = tempfile.mkstemp(suffix=".csv")
        os.close(fd)
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        self.proc = subprocess.Popen([exe, f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20", "-i",
                                      str(self._physical_index())], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)

    def stop(self) -> dict:
        sm, power, reasons = [], [], set()
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            for mhz, watts, mask in self.samples:
                sm.append(mhz); power.append(watts)
                reasons.update(nm for bit, nm in self.REASONS.items() if mask & bit)
            source = "nvml"
        elif self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for line in Path(self.path).read_text().splitlines():
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[0])); self.max_mhz = float(f[1]); power.append(float(f[2]))
                except (ValueError, IndexError):
                    continue
                reasons.update(nm for nm, v in zip(names, f[3:7]) if v.lower().startswith("active"))
            os.unlink(self.path)
            source = "nvidia-smi"
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "neither NVML nor nvidia-smi available"}
        # "under load" = samples taken while the board drew more than half of the highest power seen
        load = [c for c, w in zip(sm, power) if w >= 0.5 * max(power)] if power else []
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(reasons), "samples": len(sm), "samples_under_load": len(load),
                "power_w_max": max(power) if power else None, "source": source}


def set_cpu_threads(requested: int) -> int:
    """Thread count of the CPU arms, set explicitly: torchrun exports OMP_NUM_THREADS=1, which would turn the reference
    arm at N > 1 into a one-thread run (and inflate every ratio computed from it). Default: half the logical CPUs
    (= the physical cores of an SMT-2 host), the count torch itself picks when nothing overrides it."""
    n = requested if requested > 0 else max(1, (os.cpu_count() or 2) // 2)
    torch.set_num_threads(n)
    return torch.get_num_threads()


def reference_cpu_step(a32, b32):
    return torch.matmul(a32, b32).half()          # the reference's truth path (zero_one_correctness_check.py:87-90)


def cpu_baseline(m, n, k, seconds: float, threads: int) -> dict:
    import oracle  # the one place bench.py may use oracle/: the reported CPU baseline (never the measured path)

    cores = set_cpu_threads(threads)
    g = torch.Generator().manual_seed(0)
    a = torch.randn((m, k), generator=g).half()
    b = torch.randn((k, n), generator=g).half()
    reference_cpu_step(a.float(), b.float())      # warm-up
    reps, t0 = 0, time.perf_counter()
    while True:
        oracle.reference_truth(a, b)
        reps += 1
        el = time.perf_counter() - t0
        if (reps >= 3 and el >= seconds) or el >= 3 * seconds:
            break
    tf = 2.0 * m * n * k * reps / el * 1e-12
    return {"value": tf, "unit": "TFLOP/s", "cores": cores, "host_cpus": os.cpu_count(),
            "kind": "reference",
            "sample": f"{reps} x torch.matmul(a.cpu().float(), b.cpu().float()).half() at {m}x{n}x{k} in {el:.1f} s on {cores} threads"}


def run_reference(args, m, n, k, rank, world):
    """--impl reference: the reference's own CPU implementation of the path as the whole job (rank 0 only)."""
    if rank != 0:
        return
    import oracle

    cores = set_cpu_threads(args.cpu_threads)
    g = torch.Generator().manual_seed(0)
    a = torch.randn((m, k), generator=g).half()
    b = torch.randn((k, n), generator=g).half()
    per_step = 2.0 * m * n * k
    # bounded sample: a step is one full GEMM of the workload; cap the step count so the run stays in minutes
    for _ in range(max(1, min(args.warmup, 2))):
        oracle.reference_truth(a, b)
    steps = max(1, args.steps)
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        oracle.reference_truth(a, b)
        done += 1
        if time.perf_counter() - t0 > 120.0:
            break
    el = time.perf_counter() - t0
    tf = per_step * done / el * 1e-12
    sample = f"{done} of {steps} requested steps, each one {m}x{n}x{k} fp32 torch.matmul + .half() on {cores} threads"
    print(json.dumps({
        "impl": "reference", "metric": "HGEMM TFLOP/s, offline mode, per (M,N,K)", "value": tf, "unit": "TFLOP/s",
        "n_gpus": world, "steps": done, "warmup": args.warmup, "ms_per_step": el / done * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (fp16 operands widened)",
        "data": "synthetic N(0,1) fp16",
        "config": {"workload": f"{m}_{n}_{k} --acc_precise {args.acc} --mode offline", "parallelism": "cpu threads",
                   "note": "reference CPU path = its ground-truth expression; its GPU kernels target sm_80/sm_90"},
        "cpu_baseline": {"value": tf, "unit": "TFLOP/s", "cores": cores, "host_cpus": os.cpu_count(),
                         "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS"), "kind": "reference", "sample": sample},
        "e2e": {"value": tf, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def sweep_shapes(spec: str):
    from cuda_l2_b200 import farm

    if spec == "grid":
        return farm.grid_shapes()
    return [tuple(int(x) for x in s.split("_")) for s in spec.split(",") if s]


def sweep_cost(shape) -> float:
    """Seconds one shape costs a rank in the sweep leg (sampling budget floor + a handful of calls)."""
    m, n, k = shape
    t = max(2.0 * m * n * k / 1.3e15, 2.0 * (m * k + n * k + m * n) / 5.5e12, 6e-6)
    return 0.027 + 9 * t


def sweep_partition(shapes, world: int):
    """Longest-first onto the least loaded rank (the farm's rule with this leg's cost model)."""
    loads = [0.0] * world
    parts = [[] for _ in range(world)]
    for s in sorted(shapes, key=lambda s: (-sweep_cost(s), s)):
        r = min(range(world), key=lambda i: (loads[i], i))
        parts[r].append(s)
        loads[r] += sweep_cost(s)
    return parts


def run_sweep(args, capi, rank: int, world: int, dist) -> dict | None:
    """BASELINE config 5 on this job's GPUs. Returns the report on rank 0."""
    shapes = sweep_shapes(args.sweep)
    mine = sweep_partition(shapes, world)[rank]
    lib = capi.hgemm_lib()
    fn = lib.b200_hgemm_f32acc if args.acc == "fp32" else lib.b200_hgemm_f16acc
    max_e = max(max(m * k, n * k, m * n) for m, n, k in shapes)
    g = torch.Generator(device="cuda").manual_seed(99 + rank)
    buf_a = torch.randn(max_e, device="cuda", generator=g).half()
    buf_b = torch.randn(max_e, device="cuda", generator=g).half()
    buf_c = torch.empty(max_e, dtype=torch.half, device="cuda")
    pa, pb, pc = buf_a.data_ptr(), buf_b.data_ptr(), buf_c.data_ptr()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync, clock = torch.cuda.synchronize, time.perf_counter
    budget = args.sweep_ms * 1e-3
    launches0 = capi.launch_count()
    recs = []
    sync()
    t_leg0 = clock()
    for (m, n, k) in mine:
        def call():
            st = fn(pa, None, pb, pc, m, n, k, None)
            if st:
                raise RuntimeError(f"b200_hgemm failed on {m}x{n}x{k}: {capi.strerror(st)}")
        flops = 2.0 * m * n * k
        call(); call(); sync()
        # the harness metric: host clock around ONE call bracketed by device synchronisation
        tf_sum, ms_sum, cnt, t_shape = 0.0, 0.0, 0, clock()
        while cnt < 3 or (clock() - t_shape < budget and cnt < 200):
            sync(); t0 = clock(); call(); sync(); dt = clock() - t0
            tf_sum += flops / dt * 1e-12; ms_sum += dt * 1e3; cnt += 1
        # device time of back-to-back calls (offline throughput), CUDA events on the launching stream
        reps = max(3, min(64, int(2e-3 / max(ms_sum / cnt * 1e-3, 1e-6))))
        e0.record()
        for _ in range(reps):
            call()
        e1.record(); sync()
        recs.append((m, n, k, tf_sum / cnt, ms_sum / cnt, e0.elapsed_time(e1) / reps))
    sync()
    leg_s = clock() - t_leg0
    launches = capi.launch_count() - launches0
    dev_s = sum(r[5] for r in recs) * 1e-3
    mine_report = {"rank": rank, "shapes": len(recs), "device_s": dev_s, "leg_s": leg_s, "launches": launches,
                   "flops": sum(2.0 * r[0] * r[1] * r[2] for r in recs), "recs": recs}
    if dist is not None:
        bucket = [None] * world
        dist.all_gather_object(bucket, mine_report)      # a few KB of Python numbers; the GEMM path itself has no collective
    else:
        bucket = [mine_report]
    if rank != 0:
        return None
    peak_tf, peak_hbm, _, _ = peaks()
    allrecs = [r for b in bucket for r in b["recs"]]
    total_flops = sum(b["flops"] for b in bucket)
    makespan_dev = max(b["device_s"] for b in bucket)
    roof_s = sum(max(2.0 * m * n * k / (peak_tf * 1e12), 2.0 * (m * k + n * k + m * n) / (peak_hbm * 1e9))
                 for m, n, k, *_ in allrecs)
    named = {f"{m}_{n}_{k}": {"harness_tflops": tf, "device_us": us * 1e3}
             for m, n, k, tf, _, us in allrecs if (m, n, k) in ((64, 4096, 64), (4096, 4096, 4096), (8192, 8192, 8192), (2048, 11008, 4096))}
    return {
        "what": "BASELINE config 5: every (M,N,K) of the grid once per job, shapes dealt longest-first to the ranks, no collective on the GEMM path",
        "shapes": len(allrecs), "acc": args.acc,
        "aggregate_tflops": total_flops / makespan_dev * 1e-12,       # whole sweep / slowest rank's summed device time
        "aggregate_definition": "sum(2MNK over all shapes) / max over ranks of sum(per-shape CUDA-event time of back-to-back calls)",
        "sum_device_s": sum(b["device_s"] for b in bucket), "makespan_device_s": makespan_dev,
        "makespan_wall_s": max(b["leg_s"] for b in bucket),
        "harness_mean_tflops": sum(r[3] for r in allrecs) / len(allrecs),   # the reference's per-shape metric, averaged
        "roofline_frac": roof_s / sum(b["device_s"] for b in bucket),       # sum of per-shape roofline minima / measured
        "roofline_min_s": roof_s,
        "per_rank": [{k: b[k] for k in ("rank", "shapes", "device_s", "leg_s", "launches")} for b in bucket],
        "baseline_config_shapes": named,
        "l2_policy": "operands of a shape stay where the previous call left them (L2-resident when they fit), as in the reference harness which times a call right after writing its operands",
    }


def output_sample(c: torch.Tensor) -> np.ndarray:
    """``c`` as float32 on the host: whole up to DUMP_MAX_ELEMS entries, otherwise the entries at sorted flat indices
    drawn with seed 0 (they depend on the shape only, so runs of the same shape are comparable entry for entry)."""
    if c.numel() <= DUMP_MAX_ELEMS:
        return c.float().cpu().numpy()
    g = torch.Generator().manual_seed(0)
    idx = torch.randint(c.numel(), (DUMP_MAX_ELEMS,), generator=g).unique()
    return c.reshape(-1)[idx.to(c.device)].float().cpu().numpy()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    m, n, k = (int(x) for x in args.mnk.split("_"))
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the GPU path's output; --impl reference has none")
        run_reference(args, m, n, k, rank, world)
        return 0

    from cuda_l2_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the HGEMM path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    capi.hgemm_lib()   # fail loudly now if the library is missing

    # operand sets: enough of them that a step never finds its inputs in L2
    set_bytes = 2 * (m * k + n * k + m * n)
    nsets = max(2, min(16, -(-4 * L2_BYTES // set_bytes)))
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    sets = []
    for _ in range(nsets):
        a = torch.randn((m, k), device="cuda", generator=g).half()
        bt = torch.randn((n, k), device="cuda", generator=g).half()      # K-major B (the harness's b_col_major)
        c = torch.empty((m, n), dtype=torch.half, device="cuda")
        sets.append((a, bt.view(k, n), c))

    def step(i):
        a, b_col_major, c = sets[i % nsets]
        capi.hgemm(a, b_col_major, c, args.acc)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    warm = max(args.warmup, 3)
    for i in range(warm):
        step(i)
    barrier()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.1)
    launches0 = capi.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        step(i)
    e1.record()
    barrier()
    launches = capi.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None      # the clock record of the region `value` is computed from
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    if dist is not None:
        lt = torch.tensor([launches], device="cuda", dtype=torch.int64)
        dist.all_reduce(lt)
        launches = int(lt.item())
    flops_step = 2.0 * m * n * k
    value = flops_step * args.steps * world / (ms_total * 1e-3) * 1e-12
    # taken now: the legs below run the same operand sets again
    dump = output_sample(sets[(args.steps - 1) % nsets][2]) if args.dump_outputs and rank == 0 else None

    # ---- sustained: the same loop for about a second (power-capped clocks), same timing rules
    sustained = None
    if args.sustained_seconds > 0:
        sus_steps = max(args.steps, int(args.sustained_seconds / max(ms_total / args.steps * 1e-3, 1e-6)))
        sus_sampler = ClockSampler(local_rank)
        if rank == 0:
            sus_sampler.start()
        barrier()
        e0.record()
        for i in range(sus_steps):
            step(i)
        e1.record()
        barrier()
        sus_ms = max_over_ranks(e0.elapsed_time(e1))
        sustained = {"value": flops_step * sus_steps * world / (sus_ms * 1e-3) * 1e-12, "unit": "TFLOP/s", "steps": sus_steps,
                     "ms_per_step": sus_ms / sus_steps, "seconds": sus_ms * 1e-3,
                     "clocks": sus_sampler.stop() if rank == 0 else None}

    # ---- end-to-end leg: host buffers through the C ABI, copies inside the timed region
    # host buffers are allocated (and the calls made) from the CPUs local to this rank's GPU — what numactl would do
    with capi.host_near_gpu(local_rank) as near:
        ha = torch.randn((m, k)).half().pin_memory()
        hbt = torch.randn((n, k)).half().pin_memory()
        hc = torch.empty((m, n), dtype=torch.half).pin_memory()
        e2e_steps = args.e2e_steps or max(1, min(args.steps, 50))
        for _ in range(3):
            capi.hgemm_host(ha, hbt.view(k, n), hc, args.acc)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            capi.hgemm_host(ha, hbt.view(k, n), hc, args.acc)
        torch.cuda.synchronize()
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        near_cpus = len(near.cpus) if near.cpus else None
    e2e_value = flops_step * e2e_steps * world / e2e_s * 1e-12

    # ---- BASELINE config 5: the shape sweep sharded over this job's GPUs
    sweep = None
    if args.sweep != "none":
        del sets
        torch.cuda.empty_cache()
        barrier()
        sweep = run_sweep(args, capi, rank, world, dist)
        if dist is not None:
            lt = torch.tensor([capi.launch_count() - launches0], device="cuda", dtype=torch.int64)
            dist.all_reduce(lt)
            total_launches = int(lt.item())
        else:
            total_launches = capi.launch_count() - launches0
    else:
        total_launches = None

    if rank == 0:
        peak_tf, peak_hbm, peak_src, peak_sustained = peaks()
        sec_per_launch = ms_total / args.steps * 1e-3                      # per launch, from the CUDA events above
        ai = (m * n * k) / (m * k + n * k + m * n)                         # FLOP per byte
        ridge = peak_tf * 1e12 / (peak_hbm * 1e9)
        if ai >= ridge:
            bound, achieved, peak, unit = "tensor", flops_step / sec_per_launch * 1e-12, peak_tf, "TFLOP/s"
        else:
            bound, achieved, peak, unit = "hbm", set_bytes / sec_per_launch * 1e-9, peak_hbm, "GB/s"
        cfg_id, group_m, splits = capi.select(args.acc, m, n, k)
        cfg = capi.configs()[cfg_id]
        traffic, traffic_src = None, None
        tf = REPO / "profiles" / "dram_traffic.json"
        if tf.exists():
            traffic = json.loads(tf.read_text()).get(f"{args.mnk}_{args.acc}")
            traffic_src = ("profiles/dram_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` "
                           "capture of this kernel on this workload (a profiler run, NOT measured inside this timed run)")
        out = {
            "metric": "HGEMM TFLOP/s, offline mode, per (M,N,K)",
            "value": value, "unit": "TFLOP/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 x f16 -> " + ("f32" if args.acc == "fp32" else "f16") + " accumulate -> f16",
            "data": "synthetic N(0,1) fp16",
            "config": {"workload": f"{args.mnk} --acc_precise {args.acc} --mode offline", "parallelism": f"1 GEMM per GPU x {world}",
                       "l2_policy": f"rotating {nsets} operand sets ({nsets * set_bytes >> 20} MiB > 126 MiB L2)",
                       "kernel_config": {"tile": f"{128 * cfg['cta_group'] * cfg.get('m_rep', 1)}x{cfg['bn']}x64", "stages": cfg["stages"],
                                         "cta_group": cfg["cta_group"], "cluster": f"{cfg['cluster_m']}x{cfg['cluster_n']}", "group_m": group_m,
                                         "split_k": splits}},
            "sustained": sustained,
            "e2e": {"value": e2e_value, "unit": "TFLOP/s", "h2d_bytes_per_step": 2 * (m * k + n * k),
                    "d2h_bytes_per_step": 2 * m * n, "steps": e2e_steps, "api": "b200_hgemm_host (pinned host buffers, row-block pipelined H2D / GEMM / D2H)",
                    "host_cpus_local_to_gpu": near_cpus},
            "gpu_launches": launches,
            "gpu_launches_all_legs": total_launches,
            "clocks": clocks,
            "roofline": {"bound": bound, "achieved": achieved, "peak": peak, "unit": unit,
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "arithmetic_intensity": ai, "ridge": ridge,
                         "peak_sustained": peak_sustained if bound == "tensor" else None,
                         "frac_sustained_of_sustained_peak": (sustained["value"] / world / peak_sustained)
                         if (sustained and peak_sustained and bound == "tensor") else None,
                         "algorithmic_flops_per_launch": flops_step, "algorithmic_bytes_per_launch": set_bytes},
            "sweep": sweep,
        }
        if world == 1:
            out["cpu_baseline"] = cpu_baseline(m, n, k, args.cpu_seconds, args.cpu_threads)
        if dump is not None:
            Path(args.dump_outputs).mkdir(parents=True, exist_ok=True)
            np.save(Path(args.dump_outputs) / "c.npy", dump)
        print(json.dumps(out))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
