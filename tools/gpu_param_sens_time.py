"""Cost of the sensitivity outputs on config 4 (65 536 seed-11 dispersions, nt = 200, default options, trajectories on
the device): the solve without a sensitivity output, with the four-row output (sensitivities=True) and with the
all-row output (sensitivities="all"), alternated over --reps rounds after one warm-up round, each on one handle per
mode.  Times are CUDA events around the solve (lmato_last_kernel_ms: the launches of one solve, warm-start reference
included); the figure is the median per mode, printed with the card's name and power limit.

    python tools/gpu_param_sens_time.py [--reps 7] [--out param_sens_time.json]
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import lunar_module_ascent_trajectory_optimiser_b200 as lm  # noqa: E402

MODES = {"none": False, "four_rows": True, "all_rows": "all"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None, help="also write the result as JSON here")
    a = ap.parse_args()
    smi = shutil.which("nvidia-smi")
    card = subprocess.run([smi, "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()[0] if smi else torch.cuda.get_device_name(0)
    B = 65536
    rows = lm.dispersed_params(B, seed=11).rows(B).cuda()
    solvers = {m: lm.AscentSolver(lm.Mesh(nt=200), lm.SolverOptions(dcost=1e-5), device=0) for m in MODES}
    outs = {m: s.alloc_outputs(B) for m, s in solvers.items()}
    ms = {m: [] for m in MODES}
    conv = {}
    for r in range(a.reps + 1):
        for m, sens in MODES.items():
            res = solvers[m].solve_rows(rows, out=outs[m], sensitivities=sens)
            t = solvers[m].last_kernel_ms()
            conv[m] = int((res["status"] == 0).sum())
            if r > 0:
                ms[m].append(t)
    med = {m: statistics.median(v) for m, v in ms.items()}
    res = {"config": 4, "B": B, "nt": 200, "card": card, "reps": a.reps,
           "median_ms": med, "min_ms": {m: min(v) for m, v in ms.items()}, "max_ms": {m: max(v) for m, v in ms.items()},
           "overhead_vs_none": {m: med[m] / med["none"] - 1.0 for m in MODES}, "converged": conv}
    print(json.dumps(res), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
