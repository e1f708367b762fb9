#!/usr/bin/env python
"""Benchmark of the hot path: converged ascent-NLP solves per second.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W

A "step" = one pass of the hot path over one batch: BASELINE.json configs[3], ONE 65,536-instance
dispersion batch (thrust, Isp, initial mass, angular-acceleration limit, target perilune/apolune; nt=200,
NODES=2) solved to a scaled KKT error of 1e-10.  With N GPUs the batch is index-sharded over the ranks by the
product's own `sharded_solve` (problem i -> rank floor(i*N/B)) and ONE NCCL allgather returns the per-problem
results to every rank: STRONG scaling, the total work is fixed (`--scaling weak` keeps 65,536 problems per
GPU instead; a weak-scaling measurement also rides along in the default line as `weak_scaling`).
`--config 5` selects BASELINE's dense-mesh stress (4,096 problems, nt=2001).

Prints ONE JSON line (rank 0).  `value` is device-resident throughput (parameters already in
HBM, results left in HBM); `e2e` is the same metric through the public host API
(`AscentSolver.solve_rows` on pinned host tensors = lmato_solve_batch_host: H2D of the
parameters, solve, D2H of tf / final mass / status / iterations / KKT error and the full
[10, nt, B] trajectory block).
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# algorithmic work per mesh stage per IPM iteration (SURVEY.md section 8(d), Appendix F)
FLOP_PER_STAGE = 2147.0
BYTE_PER_STAGE = 336.0
METRIC = "converged ascent-NLP solves/sec at batch 64K"
# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel, from the `ncu --set full`
# captures summarised under profiles/ (a profiler figure cannot be measured inside an un-profiled run): keyed
# by (dcost on, problems in the launch, nt) and reported only when the run matches that workload, otherwise null.
NCU_TRAFFIC = {(True, 65536, 200): (217.761e9 + 123.660e9, "profiles/r02_ncu_ascent_ipm_kernel_metrics.csv"),
               (True, 4096, 2001): (596.359e9 + 265.691e9, "profiles/r02_ncu_ascent_coop_kernel_cfg5_metrics.csv")}
DUMP_BYTES = 48 * 2**20        # --dump-outputs: all files together stay below this (a full config-4 step is ~1 GB)


def dump_outputs(dirname, raw, traj_offset=0):
    """Write the arrays one step returned (``solve_rows``' dict) as ``dirname/<name>.npy``, all float64 (status and
    iterations convert exactly).  The per-problem results cover the whole batch when they fit a quarter of
    DUMP_BYTES, the [10, nt, n] trajectory block as many problems as the rest allows; where not every problem
    fits, the problems are a fixed seeded sample.  ``index.npy`` / ``traj_index.npy`` name the problems (index
    in the batch) row for row, so the files of two builds run with the same arguments compare element-wise."""
    import numpy as np
    import torch

    def pick(B, bytes_per_problem, budget):
        n = min(B, budget // bytes_per_problem)
        if n == B:
            return torch.arange(B)
        return torch.randperm(B, generator=torch.Generator().manual_seed(0))[:n].sort().values

    keys = [k for k in ("tf", "final_mass", "status", "iterations", "kkt") if raw.get(k) is not None]
    idx = pick(int(raw["tf"].shape[0]), 8 * (len(keys) + 1), DUMP_BYTES // 4)
    out = {k: raw[k][idx.to(raw[k].device)] for k in keys}
    out["index"] = idx
    traj = raw.get("traj")
    if traj is not None:
        used = sum(8 * v.numel() for v in out.values())
        j = pick(int(traj.shape[2]), 8 * (traj.shape[0] * traj.shape[1] + 1), DUMP_BYTES - used)
        out["traj"] = traj[:, :, j.to(traj.device)]
        out["traj_index"] = j + traj_offset
    os.makedirs(dirname, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(dirname, f"{k}.npy"), v.cpu().numpy().astype(np.float64))


def bind_to_gpu_numa_node(index):
    """Pin this rank to the CPUs NVML reports as local to its GPU, so that the pinned host buffers of the
    end-to-end leg (first touch) live on the NUMA node the GPU's PCIe root hangs on.  Multi-rank runs only:
    eight ranks each stream 1 GB of results per step into host memory."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clocks / throttle reasons sampled DURING the timed region, every 200 ms, through NVML
    (nvidia_ml_py) from a thread.  (An `nvidia-smi -lms 200` subprocess was measured to cost ~17 %
    of a 140 ms step here, so the same counters are read in-process instead; nvidia-smi is the
    fallback.)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples = []          # (sm_mhz, max_mhz, reasons-bitmask)
        self.stop_flag = threading.Event()
        self.thread = None
        self.mode = None
        self.proc = None
        self.lines = []

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES if it is a plain list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if vis and all(t.strip().isdigit() for t in vis.split(",")):
                idx = int(vis.split(",")[self.index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.mode = "nvml"
            # prime every query once (the first NVML call of each kind is slow)
            pynvml.nvmlDeviceGetClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            try:
                pynvml.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.mode = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.mode = "smi"
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((float(sm), float(mx), int(rs)))
            except Exception:
                pass
            self.stop_flag.wait(float(os.environ.get("LMATO_CLOCK_PERIOD_S", "0.2")))

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.mode == "nvml":
            self.stop_flag.set()
            self.thread.join(timeout=2)
            nv = self.nv
            names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                     "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                     "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
            sm = [s[0] for s in self.samples]
            mx = [s[1] for s in self.samples]
            reasons = sorted({n for n, bit in names.items() for s in self.samples if s[2] & bit})
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                    "reasons": reasons, "samples": len(sm), "source": "nvml"}
        if self.mode != "smi" or self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def probe_gekko():
    """BASELINE.md section 2: before timing the CPU arm, see whether the reference's own stack is importable on
    this box.  Returns (usable, note)."""
    try:
        import gekko  # noqa: F401
    except Exception as e:                      # not in this image: no network, not in /opt/wheelhouse
        return False, f"import gekko failed: {type(e).__name__}: {e}"
    try:
        from tools.probe_gekko import solve_reference_model
        tf, wall = solve_reference_model(nt=200)
        return True, f"GEKKO(remote=False) solved the reference model: tf*470 = {tf * 470.0:.6f} s in {wall:.2f} s"
    except Exception as e:
        return False, f"gekko imports but the local solve failed: {type(e).__name__}: {e}"


def run_reference(args, rank, world):
    """The reference's CPU implementation of the path on all host cores.  GEKKO/apm/IPOPT are probed first; if
    they are not usable (they are absent from this image: no network, not in /opt/wheelhouse) the arm times
    the oracle port and says so."""
    if rank != 0:
        return
    import numpy as np
    import torch
    import lunar_module_ascent_trajectory_optimiser_b200 as lm
    from oracle.cpu_baseline import OraclePool
    gekko_ok, gekko_note = probe_gekko()
    pool = OraclePool(gekko=gekko_ok)
    per_step = pool.cores                      # bounded sample: one problem per core per step
    nt = args.nt
    rows = lm.dispersed_params(max(per_step * (args.steps + args.warmup), 1), seed=11).rows().numpy()
    opts = lm.SolverOptions()
    off = 0
    for _ in range(args.warmup):
        pool.solve(rows[:, off:off + per_step], nt, opts.tol, opts.obj_scale); off += per_step
    t0 = time.perf_counter()
    nconv = 0
    iters = []
    for _ in range(args.steps):
        tf, st, it, _w = pool.solve(rows[:, off:off + per_step], nt, opts.tol, opts.obj_scale)
        off += per_step
        nconv += int((st == 0).sum()); iters += it.tolist()
    wall = time.perf_counter() - t0
    pool.close()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"tf": torch.from_numpy(tf), "status": torch.from_numpy(st),
                                         "iterations": torch.from_numpy(it)})
    val = nconv / wall
    kind = "reference" if gekko_ok else "port"
    sample = f"{per_step} problems per step (one per host core) of the seed-11 cfg{args.config} dispersions, nt={nt}, tol={opts.tol:g}"
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "solves/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall / max(args.steps, 1) * 1e3,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args), "sample_per_step": per_step, "tol": opts.tol},
            "cpu_baseline": {"value": val, "unit": "solves/s", "cores": pool.cores, "kind": kind, "sample": sample,
                             "gekko_probe": gekko_note,
                             "note": ("GEKKO(remote=False), one problem per process" if gekko_ok else
                                      "oracle restatement (numpy/scipy sparse IPM), not GEKKO/IPOPT: those are absent from this image"),
                             "mean_iterations": float(np.mean(iters)) if iters else None},
            "e2e": {"value": val, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def workload_name(args):
    if args.config == 5:
        return (f"cfg5: elliptical ascent, dense mesh nt={args.nt} (2,000 collocation steps), NODES=2, 6-parameter "
                f"dispersions, {args.batch} problems")
    return (f"cfg4: elliptical ascent (Launch_Optimiser.py defaults), nt={args.nt}, NODES=2, 6-parameter dispersions, "
            f"{args.batch} problems")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=4, choices=[4, 5], help="BASELINE.json config: 4 = 65,536 x nt 200 (the metric's), 5 = 4,096 x nt 2001")
    ap.add_argument("--batch", type=int, default=None, help="GLOBAL batch (strong scaling) / per-GPU batch (weak)")
    ap.add_argument("--nt", type=int, default=None)
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--kernel", default="auto", choices=["auto", "thread", "coop"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-traj", action="store_true", help="do not materialise the [10,nt,B] trajectory block")
    ap.add_argument("--no-weak", action="store_true", help="skip the additional weak-scaling measurement at N>1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.batch is None:
        args.batch = 65536 if args.config == 4 else 4096
    if args.nt is None:
        args.nt = 200 if args.config == 4 else 2001
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3                      # timing rules: W >= 3
    import torch
    import torch.distributed as dist
    import lunar_module_ascent_trajectory_optimiser_b200 as lm
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    nt, N = args.nt, args.nt - 1
    strong = args.scaling == "strong"
    Bglob = args.batch if strong else args.batch * world          # problems per step over all ranks
    traj = not args.no_traj
    # the shards of one batch keep the batch warm start even when a shard alone is small (as optimise_batch does)
    opts = lm.SolverOptions(kernel=args.kernel, warm_start=2 if Bglob >= 1024 else 1)
    solver = lm.AscentSolver(lm.Mesh(nt=nt), opts, device=dev)
    lo, hi = lm.shard_bounds(Bglob, world, rank)
    Bloc = hi - lo
    # Successive steps get DIFFERENT batches (three draws of the same dispersion, cycled), so nothing
    # a step computes -- including the warm start's reference solve, which starts from the previous
    # call's reference -- can be a replay of the step before.  Every rank generates the same global batch.
    NBATCH = 3
    rows_hosts = [lm.dispersed_params(Bglob, seed=11 + 1000 * j).rows(Bglob).pin_memory() for j in range(NBATCH)]
    rows_devs = [r.to(dev) for r in rows_hosts]
    step_no = [0]
    out_dev = solver.alloc_outputs(Bloc, traj, on_device=True)      # result buffers of this rank's shard, reused every step
    out_host = solver.alloc_outputs(Bloc, traj, on_device=False)    # pinned host memory for the e2e leg

    def solve_shard(r):
        return solver.solve_rows(r, trajectories=traj, out=out_dev)

    def step_device():
        step_no[0] += 1
        rows = rows_devs[step_no[0] % NBATCH]
        if world > 1:
            # the product path: index partition + one allgather of the per-problem results (tf, final mass,
            # status, iterations, KKT error); every rank ends up with all of them, trajectories stay sharded
            return lm.sharded_solve(rows, solve_shard, gather_traj=False)
        return solve_shard(rows)

    fp64_peak = solver.measure_fp64_peak()
    for _ in range(args.warmup):
        # identical to a timed step, including the host-side bookkeeping: the first use of each torch
        # reduction kernel costs ~0.3 s of lazy module loading that must not land in the timed region
        raw = step_device()
        solver.last_kernel_ms()
        int((raw["status"] == 0).sum()); int(raw["iterations"].sum())
    torch.cuda.synchronize()
    launches0 = solver.kernel_launches()
    sampler = ClockSampler(local_rank)
    if rank == 0 and os.environ.get("LMATO_NO_CLOCKS") != "1":
        sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms, conv, iters_total = 0.0, 0, 0
    ev0.record()
    for _ in range(args.steps):
        raw = step_device()
        kernel_ms += solver.last_kernel_ms()          # CUDA events around this rank's IPM kernel on its stream
        conv += int((raw["status"] == 0).sum())       # over the WHOLE batch (gathered) -- identical on every rank
        iters_total += int(raw["iterations"].sum())
    ev1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    launches = solver.kernel_launches() - launches0
    stats = torch.tensor([ms, kernel_ms, float(launches)], dtype=torch.float64, device=dev)
    if world > 1:
        mx = stats.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms, kernel_ms = float(mx[0]), float(mx[1])
        launches_all = int(sm[2])
    else:
        launches_all = int(launches)
    conv_all, iters_all = float(conv), float(iters_total)
    value = conv_all / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        # `raw` is the last timed step's result: every problem's scalars, this rank's trajectory shard [lo, hi)
        dump_outputs(args.dump_outputs, raw, lo)

    # ---- end-to-end through the host API (pinned host tensors in, pinned host tensors out), this rank's shard ----
    shard_hosts = [r[:, lo:hi].contiguous().pin_memory() for r in rows_hosts]
    for j in range(2):
        solver.solve_rows(shard_hosts[j % NBATCH], trajectories=traj, out=out_host)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    conv_e = 0
    for j in range(args.steps):
        r = solver.solve_rows(shard_hosts[(j + 2) % NBATCH], trajectories=traj, out=out_host)   # synchronous: H2D + solve + D2H
        conv_e += int((r["status"] == 0).sum())
    if world > 1:
        dist.barrier()
    e2e_s = time.perf_counter() - t0
    e = torch.tensor([e2e_s, float(conv_e)], dtype=torch.float64, device=dev)
    if world > 1:
        emx = e.clone(); dist.all_reduce(emx, op=dist.ReduceOp.MAX)
        esm = e.clone(); dist.all_reduce(esm, op=dist.ReduceOp.SUM)
        e2e_s, conv_e_all = float(emx[0]), float(esm[1])
    else:
        conv_e_all = float(conv_e)
    h2d = shard_hosts[0].numel() * 8
    d2h = (10 * nt * Bloc * 8 if traj else 0) + Bloc * (8 * 3 + 4 * 2)

    # ---- N > 1: the weak-scaling figure rides along (65,536 problems per GPU, same product path) ----
    weak = None
    if world > 1 and strong and not args.no_weak:
        Bw = args.batch * world
        wrows = lm.dispersed_params(Bw, seed=4011).rows(Bw).to(dev)
        wl, wh = lm.shard_bounds(Bw, world, rank)
        wout = solver.alloc_outputs(wh - wl, False, on_device=True)
        wfn = lambda r: solver.solve_rows(r, trajectories=False, out=wout)
        for _ in range(2):
            lm.sharded_solve(wrows, wfn, gather_traj=False)
        dist.barrier(); torch.cuda.synchronize()
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record()
        wconv = 0
        for _ in range(args.steps):
            wr = lm.sharded_solve(wrows, wfn, gather_traj=False)
            wconv += int((wr["status"] == 0).sum())
        w1.record(); torch.cuda.synchronize(); dist.barrier()
        wt = torch.tensor([w0.elapsed_time(w1)], dtype=torch.float64, device=dev)
        dist.all_reduce(wt, op=dist.ReduceOp.MAX)
        weak = {"value": wconv / (float(wt[0]) * 1e-3), "unit": "solves/s", "global_batch": Bw, "batch_per_gpu": args.batch,
                "ms_per_step": float(wt[0]) / args.steps, "trajectories": False}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- latency of a single nominal solve through the host API ----
    lat = []
    s1 = lm.AscentSolver(lm.Mesh(nt=nt), lm.SolverOptions(kernel=args.kernel), device=dev)
    r1 = lm.AscentParams().rows(1).pin_memory()
    for i in range(103):        # 2 warm-up calls + 101 timed (SURVEY 8d: median over >= 101 repeats)
        t0 = time.perf_counter(); s1.solve_rows(r1, trajectories=True); dt = time.perf_counter() - t0
        if i >= 2:
            lat.append(dt * 1e3)

    hbm_peak, peak_src = load_peaks()
    # Algorithmic work of the slowest rank's kernel launches: sum over ITS problems of iterations x stages x
    # {336 B | 2147 FLOP}, per second of kernel time (CUDA events on the launching stream).  Only Newton
    # iterations up to convergence are credited: the n_polish extra iterations of every converged problem,
    # inertia retries, rejected line-search trials and the least-squares start are overhead.
    n_polish = 2 if (opts.dcost is None or opts.dcost > 0) else 4
    # (per GPU: the batch's credited iterations divided evenly over the ranks; kernel_ms is the slowest rank's)
    credited = max(iters_all - n_polish * conv_all, 0.0) / world
    stages_gpu = credited * N
    ach_gbs_gpu = stages_gpu * BYTE_PER_STAGE / (kernel_ms * 1e-3) * 1e-9
    ach_gf_gpu = stages_gpu * FLOP_PER_STAGE / (kernel_ms * 1e-3) * 1e-9
    f_hbm, f_fp = ach_gbs_gpu / hbm_peak, ach_gf_gpu / fp64_peak
    coop = (args.kernel == "coop") or (args.kernel == "auto" and Bloc <= 6144)
    tr = NCU_TRAFFIC.get((True, Bloc, nt)) if traj else None
    hbm = {"achieved": ach_gbs_gpu, "peak": hbm_peak, "unit": "GB/s", "frac": f_hbm, "peak_source": peak_src,
           "algorithmic_bytes_per_stage_iter": BYTE_PER_STAGE}
    fp = {"achieved": ach_gf_gpu, "peak": fp64_peak, "unit": "GFLOP/s", "frac": f_fp,
          "peak_source": "measured in this run (DFMA micro-benchmark, lmato_measure_fp64_peak)",
          "algorithmic_flop_per_stage_iter": FLOP_PER_STAGE}
    top = hbm if f_hbm >= f_fp else fp          # SURVEY 8d: report both fractions and name the larger
    line = {
        "metric": METRIC, "value": value, "unit": "solves/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args) + f"; {NBATCH} different draws (seed 11+1000j) cycled over the steps",
                   "global_batch": Bglob, "batch_per_gpu": Bloc, "tol": opts.tol, "obj_scale": opts.obj_scale,
                   "dcost": 1e-5 if opts.dcost is None else opts.dcost, "warm_start": True,
                   "kernel": "ascent_coop_kernel (8 lanes per problem)" if coop else "ascent_ipm_kernel (1 thread per problem)",
                   "trajectories": traj,
                   "parallelism": (f"one batch index-sharded x{world} by sharded_solve, one NCCL allgather of the per-problem results"
                                   + (f"; ranks bound to their GPU's NUMA node ({numa} CPUs)" if numa else "")) if world > 1 else "single GPU",
                   "l2": f"no flush needed: the kernel streams a {solver.workspace_bytes(Bloc) / 2**30:.1f} GiB workspace (>> 126 MB L2) every sweep"},
        "converged_fraction": conv_all / (Bglob * args.steps),
        "mean_iterations": iters_all / (Bglob * args.steps),
        "credited_iterations": (iters_all - n_polish * conv_all) / (Bglob * args.steps),
        "kernel_ms_per_step": kernel_ms / args.steps,
        "p50_latency_ms": {"single_solve_host_api": statistics.median(lat), "batch_per_problem": ms / args.steps / Bglob},
        "e2e": {"value": conv_e_all / e2e_s, "unit": "solves/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_s / args.steps * 1e3,
                "pcie_gbs_per_gpu": (h2d + d2h) / (e2e_s / args.steps) * 1e-9},
        "gpu_launches": launches_all,
        "clocks": clocks,
        "roofline": {"bound": "hbm" if top is hbm else "fp64", "achieved": top["achieved"], "peak": top["peak"],
                     "unit": top["unit"], "frac": top["frac"],
                     "traffic": tr[0] if tr else None, "traffic_source": (tr[1] + " (one launch, bytes; ncu capture, not this run)") if tr else None,
                     "kernel": "ascent_coop_kernel" if coop else "ascent_ipm_kernel",
                     "hbm": hbm, "fp64": fp,
                     "note": "neither roofline binds: the kernels are latency/issue bound (profiles/README.md); the larger algorithmic fraction is named"},
    }
    if weak:
        line["weak_scaling"] = weak
    if world == 1 and not args.no_cpu_baseline:
        import numpy as np
        from oracle.cpu_baseline import OraclePool
        gekko_ok, gekko_note = probe_gekko()
        pool = OraclePool(gekko=gekko_ok)
        n = min(2 * pool.cores, 256) if nt <= 400 else min(pool.cores, 16)
        _tf, st, it, wall = pool.solve(rows_hosts[0][:, :n].numpy(), nt, opts.tol, opts.obj_scale)
        pool.close()
        # parity spot-check of this very run: same inputs, GPU vs oracle
        gpu_tf = solver.solve_rows(rows_devs[0][:, :n].contiguous(), trajectories=False)["tf"].cpu().numpy()
        line["cpu_baseline"] = {"value": float((st == 0).sum() / wall), "unit": "solves/s", "cores": pool.cores,
                                "kind": "reference" if gekko_ok else "port",
                                "sample": f"first {n} problems of the batch, one problem per process on {pool.cores} cores",
                                "gekko_probe": gekko_note,
                                "note": ("GEKKO(remote=False)" if gekko_ok else
                                         "oracle restatement (numpy/scipy sparse IPM), not GEKKO/IPOPT (absent from this image)"),
                                "mean_iterations": float(np.mean(it)),
                                "max_rel_tf_diff_vs_gpu": float(np.max(np.abs(gpu_tf - _tf) / _tf))}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
