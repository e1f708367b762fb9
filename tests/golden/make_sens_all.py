"""Generate tests/golden/sens_all_disp6_seed11_nt200.npz: the oracle's central differences of tf with respect to every
row of the parameter block, the reference for the all-row sensitivity output (lmato_set_param_sensitivity_output).
The oracle solves and the process pool are those of make_golden.py.

    python tests/golden/make_sens_all.py
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from make_golden import HERE, AscentParams, _pool_map  # noqa: E402


# Every row of the parameter block (include/lmato_b200.h), in its order, with the relative step of its central difference.
SENS_ALL_NAMES = ["G", "M", "R0", "Ft", "M0", "M_dot", "fuel_mass", "angle_doubledot_max", "r_periapsis", "r_apoapsis",
                  "final_time", "mass_scalar", "angle_ub", "u_bound"]
SENS_ALL_STEPS = {"angle_doubledot_max": 1e-3, "u_bound": 1e-3}     # 1e-4 for every other row


def sens_all(B=6):
    """d tf / d params[p] for all 14 rows p of the parameter block: the problems of make_golden.py --sens-batch (the
    first 6 seed-11 config-4 draws, DCOST 1e-5 and 0) and the circular model's nominal case (DCOST 1e-5 and 0), by
    central differences of oracle solves at nt = 200.  Every row is moved on its own: mass_scalar is set to fuel_mass explicitly, so that a
    step of fuel_mass leaves it where it is (the device's rows are partial derivatives).  The circular model does not
    read angle_doubledot_max and u_bound; their differences are zero there.  tf at both ends and the step are kept, so
    that a test can bound the truncation error by the spread of the one-sided quotients.

        python tests/golden/make_sens_all.py      (398 oracle solves; 3-4.5 min on 8 CPU cores)
    """
    import dataclasses
    import torch  # noqa: F401
    from lunar_module_ascent_trajectory_optimiser_b200.dispersions import dispersed_params
    rows = dispersed_params(B, seed=11).rows(B).numpy()
    dcosts = [1e-5, 0.0]
    fuel = AscentParams().fuel_mass
    base = [[AscentParams(Ft=rows[3, b], M0=rows[4, b], M_dot=rows[5, b], angle_doubledot_max=rows[7, b],
                          r_periapsis=rows[8, b], r_apoapsis=rows[9, b], mass_scalar=fuel, dcost=dc) for b in range(B)]
            for dc in dcosts]
    circ = [dataclasses.replace(AscentParams.circular(), dcost=dc) for dc in dcosts]
    rel = np.array([SENS_ALL_STEPS.get(n, 1e-4) for n in SENS_ALL_NAMES])
    step = np.array([[rel[j] * getattr(base[0][b], n) for j, n in enumerate(SENS_ALL_NAMES)] for b in range(B)])   # [B, 14]
    cstep = np.array([rel[j] * getattr(circ[0], n) for j, n in enumerate(SENS_ALL_NAMES)])
    jobs = []
    for d in range(len(dcosts)):
        for key, p, st in [(("e", d, b), base[d][b], step[b]) for b in range(B)] + [(("c", d, 0), circ[d], cstep)]:
            jobs.append((key + (-1, 0), p, 200))
            for j, n in enumerate(SENS_ALL_NAMES):
                for s in (1, -1):
                    jobs.append((key + (j, s), dataclasses.replace(p, **{n: getattr(p, n) + s * st[j]}), 200))
    res = _pool_map(jobs)
    bad = {k: (r[5], r[4]) for k, r in res.items() if r[5] != 0 and r[4] >= 1e-9}
    assert not bad, bad
    nr = len(SENS_ALL_NAMES)

    def get(kind, d, b, j, s):
        return res[(kind, d, b, j, s)][0]

    tf = np.array([[get("e", d, b, -1, 0) for b in range(B)] for d in range(2)])
    up = np.array([[[get("e", d, b, j, 1) for j in range(nr)] for b in range(B)] for d in range(2)])
    dn = np.array([[[get("e", d, b, j, -1) for j in range(nr)] for b in range(B)] for d in range(2)])
    ctf = np.array([get("c", d, 0, -1, 0) for d in range(2)])
    cup = np.array([[get("c", d, 0, j, 1) for j in range(nr)] for d in range(2)])
    cdn = np.array([[get("c", d, 0, j, -1) for j in range(nr)] for d in range(2)])
    kkt = max(r[4] for r in res.values())
    np.savez(os.path.join(HERE, "sens_all_disp6_seed11_nt200.npz"), names=np.array(SENS_ALL_NAMES), rows=rows,
             dcost=np.array(dcosts), step=step, tf=tf, tf_up=up, tf_dn=dn, dtf=(up - dn) / (2 * step),
             circ_step=cstep, circ_tf=ctf, circ_tf_up=cup, circ_tf_dn=cdn, circ_dtf=(cup - cdn) / (2 * cstep),
             max_kkt=kkt)
    print("sens all: dtf", (up - dn) / (2 * step), "circular", (cup - cdn) / (2 * cstep), "max kkt", kkt)


if __name__ == "__main__":
    sens_all()
