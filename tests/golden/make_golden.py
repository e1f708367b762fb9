"""Generate the golden fixtures in this directory with the CPU oracle.

    python tests/golden/make_golden.py

The reference itself (GEKKO + apm + IPOPT) cannot run in the authoring container, so the
vectors come from the oracle restatement (oracle/ascent_nlp.py + oracle/ipm_reference.py)
converged to a scaled KKT error of 1e-12; the oracle in turn is pinned to the reference's two
published outputs by tests/test_oracle_golden.py.  Inputs are the seeded dispersions of
SURVEY.md section 8(d) (lunar_module_ascent_trajectory_optimiser_b200/dispersions.py).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle.ascent_nlp import AscentNLP, AscentParams  # noqa: E402
from oracle.ipm_reference import IPMOptions, solve_ipm  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
VAR_ROWS = ["y", "ydot", "ydoubledot", "x", "xdot", "xdoubledot", "angle", "angledot", "mass",
            "angledoubledot"]


def solve(p: AscentParams, nt=200, time=None, nodes=2, obj_scale=10.0, tol=1e-12):
    nlp = AscentNLP(p, nt=nt, time=time, nodes=nodes, obj_scale=obj_scale)
    r = solve_ipm(nlp, nlp.initial_guess(0.9), IPMOptions(tol=tol))
    assert r.status == 0, (r.status, r.kkt_error)
    nv = nlp.node_values(r.x)
    names = [n for n in VAR_ROWS if n in nv]
    traj = np.stack([nv[n] for n in names])
    tf = nv["tf"]
    fm = p.M0 - p.fuel_mass * nv["mass"][-1]
    return dict(tf=tf, final_mass=fm, traj=traj, names=np.array(names), iters=r.iterations, kkt=r.kkt_error,
                time=nlp.time)


def main():
    out = {}
    # config 1: the reference script's defaults
    s = solve(AscentParams())
    np.savez(os.path.join(HERE, "elliptical_nominal_nt200.npz"), **s)
    print("elliptical nominal tf_s", s["tf"] * 470, "iters", s["iters"])
    # config 2: circular IB-document model
    s = solve(AscentParams.circular())
    np.savez(os.path.join(HERE, "circular_nominal_nt200.npz"), **s)
    print("circular nominal tf_s", s["tf"] * 470, "iters", s["iters"])
    # small mesh + non-uniform mesh
    s = solve(AscentParams(), nt=40)
    np.savez(os.path.join(HERE, "elliptical_nominal_nt40.npz"), **s)
    t = np.linspace(0.0, 1.0, 60) ** 1.3
    s = solve(AscentParams(), time=t)
    np.savez(os.path.join(HERE, "elliptical_nominal_nonuniform60.npz"), **s)
    # dispersions (config 4 draws: all six columns), first 8 of seed 11
    import torch  # noqa: F401
    from lunar_module_ascent_trajectory_optimiser_b200.dispersions import dispersed_params
    dp = dispersed_params(8, seed=11)
    rows = dp.rows().numpy()
    tfs, fms, trajs = [], [], []
    for b in range(rows.shape[1]):
        p = AscentParams(Ft=rows[3, b], M0=rows[4, b], M_dot=rows[5, b], angle_doubledot_max=rows[7, b],
                         r_periapsis=rows[8, b], r_apoapsis=rows[9, b])
        s = solve(p)
        tfs.append(s["tf"]); fms.append(s["final_mass"]); trajs.append(s["traj"])
        print("dispersion", b, "tf_s", s["tf"] * 470, "iters", s["iters"])
    np.savez(os.path.join(HERE, "elliptical_dispersions8_seed11_nt200.npz"), rows=rows, tf=np.array(tfs),
             final_mass=np.array(fms), traj=np.stack(trajs), names=np.array(VAR_ROWS))


if __name__ == "__main__" and not any(a in sys.argv for a in ("--dense", "--dcost", "--sens", "--nodes", "--config3", "--circular-dcost", "--config4", "--coarse", "--sens-batch")):
    main()


def dense_mesh():
    """Dense-mesh case (the direction of config 5): nt = 801, nominal parameters; every 10th node is
    kept.  (The general sparse LU of the oracle fills in badly because of the dense tf column; nt =
    2001 does not finish in reasonable time here, the structured device solver has no such issue.)"""
    s = solve(AscentParams(), nt=801, tol=2e-7)   # the general sparse LU stalls near 5e-8 on this mesh
    keep = np.arange(0, 801, 10)
    np.savez(os.path.join(HERE, "elliptical_nominal_nt801_every10.npz"), tf=s["tf"], final_mass=s["final_mass"],
             traj=s["traj"][:, keep], names=s["names"], nodes=keep, iters=s["iters"], kkt=s["kkt"])
    print("dense mesh tf_s", s["tf"] * 470, "iters", s["iters"], "kkt", s["kkt"])


if __name__ == "__main__" and "--dense" in sys.argv:
    dense_mesh()


def dcost():
    """The reference's move suppression (angledoubledot.DCOST = 1e-5, LO:99) with the objective summed
    over the nt-1 steps (APMonitor IMODE 6): nominal case + the first 4 seed-11 dispersions."""
    import torch  # noqa: F401
    from lunar_module_ascent_trajectory_optimiser_b200.dispersions import dispersed_params
    rows = dispersed_params(4, seed=11).rows().numpy()
    tfs, fms, trajs = [], [], []
    for b in range(rows.shape[1]):
        p = AscentParams(Ft=rows[3, b], M0=rows[4, b], M_dot=rows[5, b], angle_doubledot_max=rows[7, b],
                         r_periapsis=rows[8, b], r_apoapsis=rows[9, b], dcost=1e-5)
        nlp = AscentNLP(p, nt=200, obj_scale=10.0)
        r = solve_ipm(nlp, nlp.initial_guess(0.9), IPMOptions(tol=1e-12, max_iter=500))
        assert r.status == 0, (r.status, r.kkt_error)
        nv = nlp.node_values(r.x)
        tfs.append(nv["tf"]); fms.append(p.M0 - p.fuel_mass * nv["mass"][-1])
        trajs.append(np.stack([nv[n] for n in VAR_ROWS]))
        print("dcost", b, "tf_s", nv["tf"] * 470, "iters", r.iterations, "kkt", r.kkt_error)
    np.savez(os.path.join(HERE, "elliptical_dcost1e-5_disp4_seed11_nt200.npz"), rows=rows, tf=np.array(tfs),
             final_mass=np.array(fms), traj=np.stack(trajs), names=np.array(VAR_ROWS), dcost=1e-5,
             objective_nodes=199)


if __name__ == "__main__" and "--dcost" in sys.argv:
    dcost()


def sensitivities():
    """d tf / d parameter of the nominal problem (nt = 40, no DCOST) by central finite differences of
    oracle solves: the independent check of the device's multiplier-based sensitivities (SURVEY 8f.4)."""
    import dataclasses
    base = AscentParams()
    names = ["Ft", "M0", "M_dot", "angle_doubledot_max"]
    steps = {"Ft": 1e-4, "M0": 1e-4, "M_dot": 1e-4, "angle_doubledot_max": 1e-3}
    out = {}
    for n in names:
        v = getattr(base, n)
        h = steps[n] * v
        up = solve(dataclasses.replace(base, **{n: v + h}), nt=40)["tf"]
        dn = solve(dataclasses.replace(base, **{n: v - h}), nt=40)["tf"]
        out[n] = (up - dn) / (2 * h)
        print("d tf / d", n, "=", out[n])
    np.savez(os.path.join(HERE, "sens_nominal_nt40.npz"), names=np.array(names),
             dtf=np.array([out[n] for n in names]), tf=solve(base, nt=40)["tf"])


if __name__ == "__main__" and "--sens" in sys.argv:
    sensitivities()


def higher_order():
    """NODES = 3..6 (LO:25; SURVEY Appendix B.2): Lobatto collocation with NODES-1 points per step, MV held over the
    step, no DCOST term.  Nominal case on coarse meshes for every NODES, three seed-11 dispersions for NODES = 3."""
    import torch  # noqa: F401
    from lunar_module_ascent_trajectory_optimiser_b200.dispersions import dispersed_params
    out = {}
    for nodes, nt in ((3, 40), (4, 30), (5, 24), (6, 20)):
        s = solve(AscentParams(dcost=0.0), nt=nt, nodes=nodes, tol=1e-11)
        out[f"tf_n{nodes}"] = s["tf"]; out[f"fm_n{nodes}"] = s["final_mass"]; out[f"traj_n{nodes}"] = s["traj"]
        out[f"nt_n{nodes}"] = nt
        print("nodes", nodes, "nt", nt, "tf_s", s["tf"] * 470, "iters", s["iters"], "kkt", s["kkt"])
    rows = dispersed_params(4, seed=11).rows().numpy()[:, 1:4]
    tfs, fms, trajs = [], [], []
    for b in range(rows.shape[1]):
        p = AscentParams(Ft=rows[3, b], M0=rows[4, b], M_dot=rows[5, b], angle_doubledot_max=rows[7, b],
                         r_periapsis=rows[8, b], r_apoapsis=rows[9, b], dcost=0.0)
        s = solve(p, nt=60, nodes=3, tol=1e-11)
        tfs.append(s["tf"]); fms.append(s["final_mass"]); trajs.append(s["traj"])
        print("nodes 3 dispersion", b, "tf_s", s["tf"] * 470, "iters", s["iters"])
    np.savez(os.path.join(HERE, "elliptical_higher_order_nodes3to6.npz"), names=np.array(VAR_ROWS), rows=rows,
             disp_tf=np.array(tfs), disp_fm=np.array(fms), disp_traj=np.stack(trajs), disp_nt=60, **out)


if __name__ == "__main__" and "--nodes" in sys.argv:
    higher_order()


def _cfg3_one(args):
    b, row = args
    p = AscentParams(Ft=row[3], M0=row[4], M_dot=row[5], angle_doubledot_max=row[7], r_periapsis=row[8],
                     r_apoapsis=row[9], dcost=0.0)
    nlp = AscentNLP(p, nt=200, obj_scale=10.0)
    # the oracle's line search can run out of FP64 resolution between 1e-10 and 1e-12: such a point is kept
    # with its KKT error on record (the test reads it)
    r = None
    for tf0 in (0.9, 0.95, 0.85, 0.92):     # (no restoration phase in the oracle either: other starts instead)
        r = solve_ipm(nlp, nlp.initial_guess(tf0), IPMOptions(tol=1e-12))
        if r.status == 0 or r.kkt_error < 1e-9:
            break
    nv = nlp.node_values(r.x)
    traj = np.stack([nv[n] for n in VAR_ROWS])
    return b, nv["tf"], p.M0 - p.fuel_mass * nv["mass"][-1], traj, r.iterations, r.kkt_error


def config3(B=1024, stride=20):
    """Config 3 as BASELINE.json states it: 1 024 dispersions over thrust, Isp, initial mass and the
    angular-acceleration limit (columns 0-3 of the seed-11 draws, SURVEY 8(d)), every one solved by the oracle
    (no DCOST term, KKT error 1e-12).  Kept per problem: tf, final mass, and all ten variables at every
    `stride`-th node plus the final node -- small enough to commit, dense enough to pin the whole batch."""
    import multiprocessing as mp
    import torch  # noqa: F401
    from lunar_module_ascent_trajectory_optimiser_b200.dispersions import dispersed_params
    rows = dispersed_params(B, seed=11, columns=(0, 1, 2, 3)).rows(B).numpy()
    keep = np.unique(np.concatenate([np.arange(0, 200, stride), [199]]))
    tf = np.zeros(B); fm = np.zeros(B); traj = np.zeros((B, 10, keep.size)); iters = np.zeros(B, np.int32)
    kkt = np.zeros(B)
    with mp.Pool(int(os.environ.get("GOLDEN_PROCS", os.cpu_count()))) as pool:
        for n, (b, t, f, tr, it, kk) in enumerate(pool.imap_unordered(_cfg3_one, [(b, rows[:, b]) for b in range(B)], chunksize=4)):
            tf[b] = t; fm[b] = f; traj[b] = tr[:, keep]; iters[b] = it; kkt[b] = kk
            if n % 64 == 0:
                print("config 3:", n, "of", B, "solved", flush=True)
    np.savez_compressed(os.path.join(HERE, f"elliptical_config3_disp{B}_seed11_nt200.npz"), rows=rows, tf=tf, final_mass=fm,
                        traj=traj, nodes=keep, names=np.array(VAR_ROWS), iters=iters, kkt=kkt)
    print("config 3 fixture: tf_s range", tf.min() * 470, tf.max() * 470, "max iters", iters.max(), "max kkt", kkt.max())


if __name__ == "__main__" and "--config3" in sys.argv:
    config3()


def circular_dcost():
    """The circular IB-document model WITH its move suppression (PDF p.27 src 69-73: DCOST = 1e-5 on the MV `angle`),
    objective summed over the nt-1 steps as for the elliptical model."""
    import dataclasses
    p = dataclasses.replace(AscentParams.circular(), dcost=1e-5)
    nlp = AscentNLP(p, nt=200, obj_scale=10.0)
    r = solve_ipm(nlp, nlp.initial_guess(0.9), IPMOptions(tol=1e-12, max_iter=500))
    assert r.status == 0 or r.kkt_error < 1e-9, (r.status, r.kkt_error)
    nv = nlp.node_values(r.x)
    names = [n for n in VAR_ROWS if n in nv]
    np.savez(os.path.join(HERE, "circular_dcost1e-5_nt200.npz"), tf=nv["tf"], final_mass=p.M0 - p.fuel_mass * nv["mass"][-1],
             traj=np.stack([nv[n] for n in names]), names=np.array(names), iters=r.iterations, kkt=r.kkt_error,
             dcost=1e-5, objective_nodes=199)
    print("circular with DCOST: tf_s", nv["tf"] * 470, "iters", r.iterations, "kkt", r.kkt_error)


if __name__ == "__main__" and "--circular-dcost" in sys.argv:
    circular_dcost()


def _cfg4_one(args):
    b, row = args
    p = AscentParams(Ft=row[3], M0=row[4], M_dot=row[5], angle_doubledot_max=row[7], r_periapsis=row[8],
                     r_apoapsis=row[9], dcost=1e-5)
    nlp = AscentNLP(p, nt=200, obj_scale=10.0)
    r = None
    for tf0 in (0.9, 0.95, 0.85, 0.92):
        r = solve_ipm(nlp, nlp.initial_guess(tf0), IPMOptions(tol=1e-12, max_iter=500))
        if r.status == 0 or r.kkt_error < 1e-9:
            break
    nv = nlp.node_values(r.x)
    traj = np.stack([nv[n] for n in VAR_ROWS])
    return b, nv["tf"], p.M0 - p.fuel_mass * nv["mass"][-1], traj, r.iterations, r.kkt_error


def config4_slice(B=512, stride=20):
    """A slice of config 4 on the DEFAULT path: the first 512 of the seed-11 dispersions over all six parameters
    (thrust, Isp, initial mass, angular-acceleration limit, target perilune and apolune), with the reference's move
    suppression (DCOST = 1e-5, slack pairs in the oracle), every one solved by the oracle.  Kept per problem: tf, final
    mass, the ten variables at every `stride`-th node and the final node."""
    import multiprocessing as mp
    import torch  # noqa: F401
    from lunar_module_ascent_trajectory_optimiser_b200.dispersions import dispersed_params
    rows = dispersed_params(B, seed=11).rows(B).numpy()
    keep = np.unique(np.concatenate([np.arange(0, 200, stride), [199]]))
    tf = np.zeros(B); fm = np.zeros(B); traj = np.zeros((B, 10, keep.size)); iters = np.zeros(B, np.int32)
    kkt = np.zeros(B)
    with mp.Pool(int(os.environ.get("GOLDEN_PROCS", os.cpu_count()))) as pool:
        for n, (b, t, f, tr, it, kk) in enumerate(pool.imap_unordered(_cfg4_one, [(b, rows[:, b]) for b in range(B)], chunksize=2)):
            tf[b] = t; fm[b] = f; traj[b] = tr[:, keep]; iters[b] = it; kkt[b] = kk
            if n % 32 == 0:
                print("config 4 slice:", n, "of", B, "solved", flush=True)
    np.savez_compressed(os.path.join(HERE, f"elliptical_config4_dcost_disp{B}_seed11_nt200.npz"), rows=rows, tf=tf,
                        final_mass=fm, traj=traj, nodes=keep, names=np.array(VAR_ROWS), iters=iters, kkt=kkt, dcost=1e-5,
                        objective_nodes=199)
    print("config 4 slice fixture: tf_s range", tf.min() * 470, tf.max() * 470, "max iters", iters.max(), "max kkt", kkt.max())


if __name__ == "__main__" and "--config4" in sys.argv:
    config4_slice()


def _oracle_one(args):
    """One oracle solve for the pooled modes below: (key, AscentParams, nt) -> key, tf, final mass, trajectory,
    iterations, KKT error.  Other start times are tried when the first stops short (no restoration phase)."""
    key, p, nt = args
    nlp = AscentNLP(p, nt=nt, obj_scale=10.0)
    r = None
    for tf0 in (0.9, 0.95, 0.85, 0.92):
        r = solve_ipm(nlp, nlp.initial_guess(tf0), IPMOptions(tol=1e-12, max_iter=500))
        if r.status == 0:
            break
    nv = nlp.node_values(r.x)
    traj = np.stack([nv[n] for n in VAR_ROWS if n in nv])
    return key, nv["tf"], p.M0 - p.fuel_mass * nv["mass"][-1], traj, r.iterations, r.kkt_error, r.status


def _pool_map(jobs):
    import multiprocessing as mp
    with mp.Pool(int(os.environ.get("GOLDEN_PROCS", os.cpu_count()))) as pool:
        return {r[0]: r[1:] for r in pool.imap_unordered(_oracle_one, jobs, chunksize=1)}


COARSE_CASES = [(nt, dc) for nt in (4, 5, 9, 17, 33) for dc in (0.0, 1e-5)] + [(3, 1e-5)]


def coarse():
    """Coarse meshes: the nominal problem at nt = 4, 5, 9, 17, 33, each without and with DCOST = 1e-5, and nt = 3
    with DCOST only (without it the oracle's line search fails there, status 2).  Meshes this small leave lanes of
    the cooperative kernel without a stage and let its record ring prefetch past the last stage.  Kept per case: tf,
    final mass, all ten variables at every node, iterations and KKT error (converged to 1e-12).

        python tests/golden/make_golden.py --coarse        (11 oracle solves; 7 s on 8 CPU cores)
    """
    import dataclasses
    jobs = [(i, dataclasses.replace(AscentParams(), dcost=dc), nt) for i, (nt, dc) in enumerate(COARSE_CASES)]
    res = _pool_map(jobs)
    out = dict(nt=np.array([c[0] for c in COARSE_CASES]), dcost=np.array([c[1] for c in COARSE_CASES]),
               names=np.array(VAR_ROWS))
    for k in ("tf", "final_mass", "iters", "kkt"):
        out[k] = np.array([res[i][("tf", "final_mass", "traj", "iters", "kkt").index(k)] for i in range(len(jobs))])
    for i in range(len(jobs)):
        tf, fm, traj, it, kkt, st = res[i]
        assert st == 0, (COARSE_CASES[i], st, kkt)
        out[f"traj_{i}"] = traj
        print("coarse nt", COARSE_CASES[i][0], "dcost", COARSE_CASES[i][1], "tf", tf, "iters", it, "kkt", kkt)
    np.savez(os.path.join(HERE, "elliptical_coarse_nt3to33.npz"), **out)


if __name__ == "__main__" and "--coarse" in sys.argv:
    coarse()


SENS_NAMES = ["Ft", "M0", "M_dot", "angle_doubledot_max"]
SENS_STEPS = {"Ft": 1e-4, "M0": 1e-4, "M_dot": 1e-4, "angle_doubledot_max": 1e-3}   # relative, as --sens


def sens_batch(B=6):
    """d tf / d (Ft, M0, M_dot, angle_doubledot_max) for the first 6 problems of the config-4 draws
    (dispersed_params(., seed=11), problem 0 = the nominal case) at nt = 200, with DCOST = 1e-5 and without it, by
    central differences of oracle solves (relative steps of --sens); and d tf / d (Ft, M0, M_dot) of the circular
    model's nominal case, with and without its DCOST.  tf at both ends of every difference is kept, so that a test can
    bound the truncation error by |forward - backward| difference quotient.

        python tests/golden/make_golden.py --sens-batch    (122 oracle solves; 2 min on 8 CPU cores)
    """
    import dataclasses
    import torch  # noqa: F401
    from lunar_module_ascent_trajectory_optimiser_b200.dispersions import dispersed_params
    rows = dispersed_params(B, seed=11).rows(B).numpy()
    dcosts = [1e-5, 0.0]
    base = [[AscentParams(Ft=rows[3, b], M0=rows[4, b], M_dot=rows[5, b], angle_doubledot_max=rows[7, b],
                          r_periapsis=rows[8, b], r_apoapsis=rows[9, b], dcost=dc) for b in range(B)] for dc in dcosts]
    circ = [dataclasses.replace(AscentParams.circular(), dcost=dc) for dc in dcosts]
    step = np.array([[SENS_STEPS[n] * getattr(base[0][b], n) for n in SENS_NAMES] for b in range(B)])   # [B, 4]
    cstep = np.array([SENS_STEPS[n] * getattr(circ[0], n) for n in SENS_NAMES[:3]])
    jobs = []
    for d in range(len(dcosts)):
        for b in range(B):
            p = base[d][b]
            jobs.append((("e", d, b, -1, 0), p, 200))
            for j, n in enumerate(SENS_NAMES):
                for s in (1, -1):
                    jobs.append((("e", d, b, j, s), dataclasses.replace(p, **{n: getattr(p, n) + s * step[b, j]}), 200))
        p = circ[d]
        jobs.append((("c", d, 0, -1, 0), p, 200))
        for j, n in enumerate(SENS_NAMES[:3]):
            for s in (1, -1):
                jobs.append((("c", d, 0, j, s), dataclasses.replace(p, **{n: getattr(p, n) + s * cstep[j]}), 200))
    res = _pool_map(jobs)
    assert max(r[4] for r in res.values()) < 1e-9, max(r[4] for r in res.values())
    tf = np.array([[res[("e", d, b, -1, 0)][0] for b in range(B)] for d in range(2)])
    up = np.array([[[res[("e", d, b, j, 1)][0] for j in range(4)] for b in range(B)] for d in range(2)])
    dn = np.array([[[res[("e", d, b, j, -1)][0] for j in range(4)] for b in range(B)] for d in range(2)])
    ctf = np.array([res[("c", d, 0, -1, 0)][0] for d in range(2)])
    cup = np.array([[res[("c", d, 0, j, 1)][0] for j in range(3)] for d in range(2)])
    cdn = np.array([[res[("c", d, 0, j, -1)][0] for j in range(3)] for d in range(2)])
    kkt = max(r[4] for r in res.values())
    np.savez(os.path.join(HERE, "sens_disp6_seed11_nt200.npz"), names=np.array(SENS_NAMES), rows=rows,
             dcost=np.array(dcosts), step=step, tf=tf, tf_up=up, tf_dn=dn, dtf=(up - dn) / (2 * step),
             circ_step=cstep, circ_tf=ctf, circ_tf_up=cup, circ_tf_dn=cdn, circ_dtf=(cup - cdn) / (2 * cstep),
             max_kkt=kkt)
    print("sens batch: dtf", (up - dn) / (2 * step), "circular", (cup - cdn) / (2 * cstep), "max kkt", kkt)


if __name__ == "__main__" and "--sens-batch" in sys.argv:
    sens_batch()
