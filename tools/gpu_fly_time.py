"""Post-solve flight time next to solve time, config 4 (65 536 seed-11 dispersions, nt = 200, the default options):
the device solve (lmato_solve_batch, CUDA events around the call) and lmato_fly_control of its result at the default
sub-step count, each the median of five runs after a warm-up, with the card's name and power limit.

    python tools/gpu_fly_time.py [--batch 65536] [--nt 200]
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import lunar_module_ascent_trajectory_optimiser_b200 as lm  # noqa: E402


def timed(fn, reps=5):
    ms = []
    for _ in range(reps + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return sorted(ms[1:])[reps // 2], out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--nt", type=int, default=200)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    solver = lm.AscentSolver(lm.Mesh(nt=a.nt), device=0)
    solver.set_options(lm.SolverOptions(dcost=1e-5))
    rows = lm.dispersed_params(a.batch, seed=11).rows(a.batch).cuda()
    out = solver.alloc_outputs(a.batch)
    solve_ms, raw = timed(lambda: solver.solve_rows(rows, out=out))
    n = lm.default_fly_substeps(solver.time)
    fly_ms, flown = timed(lambda: solver.fly_control(rows, raw["traj"], raw["tf"], n, trajectories=False))
    fly_traj_ms, _ = timed(lambda: solver.fly_control(rows, raw["traj"], raw["tf"], n))
    miss = flown["final"][7]
    print(f"{a.batch} problems, nt {a.nt}, {n} RK4 sub-steps per step: solve {solve_ms:.2f} ms, flight {fly_ms:.2f} ms "
          f"(with flown trajectories {fly_traj_ms:.2f} ms); radius miss {float(miss.min()):+.0f} .. "
          f"{float(miss.max()):+.0f} m; {q[0] if q else torch.cuda.get_device_name(0)}")


if __name__ == "__main__":
    main()
