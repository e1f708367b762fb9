"""Wall time of the device list on host tensors (lmato_multi_solve_host through AscentMultiSolver.solve_rows): pinned
CPU parameter rows in, the pinned result arrays solve_rows allocates out, trajectories included.  Config 5 (4 096
seed-11 dispersions, nt = 2001) and config 4 (65 536, nt = 200) over every visible GPU, or [0, 0] when only one is
visible (--devices names another list); the options optimise_batch(devices=...) uses (the batch warm start in every shard).  Each figure is the median
of --reps calls after one warm-up call, host clock around the call (it returns after a stream synchronise on every
device), printed with the card's name and power limit.

    python tools/gpu_host_staging_time.py [--reps 7] [--devices 0]
"""
import argparse
import os
import shutil
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import lunar_module_ascent_trajectory_optimiser_b200 as lm  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--devices", default=None, help="comma-separated device list, e.g. 0 (a one-device list writes "
                                                    "pinned trajectories in place); default: every visible GPU")
    a = ap.parse_args()
    smi = shutil.which("nvidia-smi")
    q = subprocess.run([smi, "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines() if smi else []
    n = torch.cuda.device_count()
    devices = [int(d) for d in a.devices.split(",")] if a.devices else list(range(n)) if n > 1 else [0, 0]
    for config, B, nt in ((5, 4096, 2001), (4, 65536, 200)):
        ms = lm.AscentMultiSolver(devices, lm.Mesh(nt=nt), lm.SolverOptions(warm_start=2 if B >= 512 else 1))
        rows = lm.dispersed_params(B, seed=11).rows(B).pin_memory()
        wall = []
        for _ in range(a.reps + 1):
            t0 = time.perf_counter()
            out = ms.solve_rows(rows)
            wall.append((time.perf_counter() - t0) * 1e3)
        conv = int((out["status"] == 0).sum())
        ms.close()
        print(f"config {config}: {B} problems, nt {nt}, devices {devices}: {statistics.median(wall[1:]):.1f} ms per call "
              f"(min {min(wall[1:]):.1f}, max {max(wall[1:]):.1f}), {conv} converged; "
              f"{q[0] if q else torch.cuda.get_device_name(0)}", flush=True)


if __name__ == "__main__":
    main()
