"""CPU oracle, part 4: a solved control flown through the continuous ascent dynamics.  TEST INFRASTRUCTURE ONLY.

The solver returns the optimum of the transcribed problem (backward Euler on the mesh for NODES = 2, Lobatto
collocation for NODES = 3..6).  This integrates the ODEs themselves (LO:114-136; circular model PDF p.27 src 76-96)
with scipy's DOP853 from mesh node to mesh node, holding the MV of node k on (t_{k-1}, t_k] as both transcriptions
hold it (MV_TYPE = 0, LO:29), from the pinned zeros of node 0 (LO:145-151).  The MV is `angledoubledot` for the
elliptical model and the pitch angle `angle` for the circular one.

    python -m oracle.fly_reference        # the transcription-error table of DESIGN.md section 7
"""
from __future__ import annotations

import math
import os
from typing import Dict

import numpy as np
from scipy.integrate import solve_ivp

from .ascent_nlp import AscentParams, _accel_numeric

STATES = ["y", "ydot", "x", "xdot", "angle", "angledot", "mass"]


def fly(p: AscentParams, time: np.ndarray, mv: np.ndarray, tf: float, rtol: float = 1e-13,
        atol: float = 1e-16) -> Dict[str, np.ndarray]:
    """Fly the per-node MV ``mv`` [nt] (node 0 unused) of a solution with scaled final time ``tf`` on the normalised
    mesh ``time`` [nt].  Returns the flown states [nt] (scaled units, the solution's names) and the terminal misses in
    SI: ``radius_miss_m``, ``speed_miss_mps`` (|v| S - v_target) and ``flight_path_angle_rad``."""
    time = np.asarray(time, dtype=np.float64)
    mv = np.asarray(mv, dtype=np.float64)
    ell = p.model == "elliptical"
    c = p.final_time * tf

    def rhs(t, s, u):
        y, yd, x, xd, a, ad, m = s
        ydd, xdd = _accel_numeric(p, y, x, a if ell else u, m)
        return [c * yd, c * ydd, c * xd, c * xdd, c * ad if ell else 0.0, c * p.asc * u if ell else 0.0,
                p.mflow * c]

    nt = time.shape[0]
    out = np.zeros((len(STATES), nt))
    s = np.zeros(len(STATES))
    for k in range(1, nt):
        r = solve_ivp(rhs, (time[k - 1], time[k]), s, method="DOP853", rtol=rtol, atol=atol, args=(mv[k],))
        if not r.success:
            raise RuntimeError(f"DOP853 failed on step {k}: {r.message}")
        s = r.y[:, -1].copy()
        out[:, k] = s
        if not ell:
            out[STATES.index("angle"), k] = mv[k]
    res = {n: out[i] for i, n in enumerate(STATES)}
    y, vy, x, vx = s[0], s[1], s[2], s[3]
    S, R0 = p.S, p.R0
    Yb = y + R0 / S
    r = math.hypot(Yb, x)
    v = math.hypot(vx, vy)
    res["radius_miss_m"] = (r - (R0 + S) / S) * S                        # LO:161
    res["speed_miss_mps"] = v * S - p.v_target                           # LO:169
    res["flight_path_angle_rad"] = math.asin((Yb * vy + x * vx) / (r * v))   # LO:173
    return res


def fly_fixture(traj: np.ndarray, names, time: np.ndarray, tf: float, p: AscentParams, **kw) -> Dict[str, np.ndarray]:
    """``fly`` for a golden trajectory [nvar, nt] with row names ``names`` (tests/golden)."""
    names = list(names)
    mv = traj[names.index("angledoubledot" if p.model == "elliptical" else "angle")]
    return fly(p, time, mv, tf, **kw)


def _table() -> None:
    golden = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
    rows = []
    for name in ("elliptical_nominal_nt40", "elliptical_nominal_nt200", "elliptical_nominal_nonuniform60"):
        g = np.load(os.path.join(golden, name + ".npz"))
        rows.append((name, fly_fixture(g["traj"], g["names"], g["time"], float(g["tf"]), AscentParams())))
    g = np.load(os.path.join(golden, "elliptical_higher_order_nodes3to6.npz"))
    for n in (3, 4, 5, 6):
        nt = int(g[f"nt_n{n}"])
        rows.append((f"nodes{n}_nt{nt}", fly_fixture(g[f"traj_n{n}"], g["names"], np.linspace(0, 1, nt),
                                                     float(g[f"tf_n{n}"]), AscentParams())))
    g = np.load(os.path.join(golden, "circular_nominal_nt200.npz"))
    rows.append(("circular_nominal_nt200", fly_fixture(g["traj"], g["names"], g["time"], float(g["tf"]),
                                                       AscentParams.circular())))
    for name, r in rows:
        print(f"{name:34s} radius miss {r['radius_miss_m']:+10.3f} m  speed miss {r['speed_miss_mps']:+9.4f} m/s  "
              f"flight-path angle {math.degrees(r['flight_path_angle_rad']):+8.4f} deg")


if __name__ == "__main__":
    _table()
