"""Every kernel instantiation that `lmato_solve_batch` can launch, against the oracle.

The launch plan (csrc/ascent_plan.h: plan_solve) picks, by batch size, DCOST, model and options, one of
    ascent_ipm_kernel<Sweeps7 | Sweeps8>          one problem per thread (above 6 144 problems, or kernel="thread")
    ascent_coop_kernel<G, GP, MOVE, BPS>          GP = 32 lanes per problem up to 8 problems per SM, else 8;
                                                  BPS = 2 CTAs per SM once one CTA per SM cannot hold the batch;
                                                  MOVE = 0 no DCOST, 1 DCOST, 2 the circular model with DCOST
and every instantiation writes the shared start points (start_rollout / start_from_guess / start_from_ref) through its
own workspace layout (SW::store_node) and reads the converged iterate through it (SW::node) for the shared result writer
(csrc/ascent_result.cuh), which the cooperative kernels run with the problem's lanes summing over the group.  The
table below reaches each of them; a
test id names the instantiation.  Batch sizes are derived from the device's SM
count with the dispatch rules of tests/dispatch_rules.py, which test_device_source_on_host.py checks against
plan_solve itself, so the same table picks the same kernels on any GPU (a variant whose batch-size window is empty
there is skipped).

Each batch carries known problems: the seed-11 dispersions are prefix-stable, so `dispersed_params(B, seed=11)` starts
with the rows of the oracle fixtures, and copies of the nominal problem (problem 0 of every such batch) sit at warp,
chunk and CTA boundaries, in the last partial chunk and at B - 1.  All copies of one launch start from the same point
(the same warm-start reference, or the same cold start), so they must come back bitwise identical.

The whole file takes about 6 s on a B200 (148 SMs, 1000 W power limit).
"""
import os

import numpy as np
import pytest
import torch

from dispatch_rules import VARIANTS

pytestmark = pytest.mark.gpu

VAR_ROWS = ["y", "ydot", "ydoubledot", "x", "xdot", "xdoubledot", "angle", "angledot", "mass",
            "angledoubledot"]
CIRCULAR_ROWS = ["y", "ydot", "ydoubledot", "x", "xdot", "xdoubledot", "mass", "angle"]   # the model's Vars and MV
SENS_NAMES = ["Ft", "M0", "M_dot", "angle_doubledot_max"]
STATE_RTOL = 1e-4
# d tf / d (Ft, M0, M_dot) against the oracle's central differences, relative, per regime: ten times the worst error
# measured over all variants on a B200 (1000 W): 2.9e-6 with DCOST, 5.3e-7 without, 1.2e-8 for the circular model.
SENS_RTOL = {"dcost": 3e-5, "nodcost": 5e-6, "circular": 1.2e-7}
# d tf / d angle_doubledot_max: tf has kinks in this parameter close to some draws (problem 4: the central quotient moves
# by 1.5e-3 between relative steps of 1e-3 and 2.5e-4), so the oracle's quotient carries an error up to its
# one-sided spread |forward - backward| / |central|, which is added to this floor
SENS_ADDM_RTOL = 1e-5


@pytest.fixture(scope="module")
def lm(built_lib):
    import lunar_module_ascent_trajectory_optimiser_b200 as lm
    assert torch.cuda.is_available()
    return lm


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _copies(B, gp):
    """Positions of the nominal copies: 0, warp boundary, chunk boundaries of the cooperative kernel (a warp holds
    32/GP problems), CTA boundary of the thread kernel, the middle, the last partial chunk and B - 1."""
    pos = {0, 31, 32, 255, 256, B // 2, B - 2, B - 1}
    if gp == 8:
        pos |= {35, 36, 4 * (B // 4) - 1}
    return sorted(p for p in pos if 0 <= p < B)


def _solver(lm, v, nt=200):
    return lm.AscentSolver(lm.Mesh(nt=nt), lm.SolverOptions(dcost=v.dcost, kernel=v.kernel, coop_lanes=v.coop_lanes),
                           device=0, model=v.model)


def _rows(lm, v, B, pos):
    """Parameter block of the variant's batch and the nominal row its copies carry."""
    if v.model == "circular":
        return lm.AscentParams.circular().rows(B)
    rows = lm.dispersed_params(B, seed=11).rows(B)
    rows[:, pos] = rows[:, :1]             # problem 0 is the nominal case
    return rows


def _rel_err(full, gold, nodes):
    """Per problem and variable: max |device - oracle| over the fixture's nodes, relative to the device's range."""
    scale = np.abs(full).max(axis=2, keepdims=True) + 1e-300
    return (np.abs(full[:, :, nodes] - gold) / scale).max(axis=2)


def _assert_copies_identical(raw, pos):
    for k in ("tf", "final_mass", "status", "iterations", "kkt"):
        x = raw[k][pos]
        assert torch.equal(x, x[:1].expand_as(x)), (k, pos, x.tolist())
    t = raw["traj"][:, :, pos]
    bad = (t != t[:, :, :1]).any(dim=1).any(dim=0)
    assert not bool(bad.any()), [pos[i] for i in torch.nonzero(bad).flatten().tolist()]
    d = raw["dtf"][:, pos]
    assert bool(((d == d[:, :1]) | (torch.isnan(d) & torch.isnan(d[:, :1]))).all()), d


_SENS = {}     # variant id -> d tf / d parameter of its first 6 problems (CPU), for the cross-variant check


def _solve_variant(lm, v, S):
    B = v.batch(S)
    if B is None:
        pytest.skip(f"{v.id}: empty batch-size window on a GPU with {S} SMs")
    exp = v.expect(S, B)
    if exp[0] == "coop":
        assert "-".join(["coop", f"gp{exp[1]}", f"bps{exp[2]}", f"move{exp[3]}"]) in v.id, (v.id, B, exp)
    else:
        assert f"sweeps{exp[1]}" in v.id, (v.id, B, exp)
    # (a circular batch is B copies of the model's nominal problem: every position is checked)
    pos = list(range(B)) if v.model == "circular" else _copies(B, exp[1] if exp[0] == "coop" else 32)
    rows = _rows(lm, v, B, pos)
    solver = _solver(lm, v)
    raw = solver.solve_rows(rows.cuda(), trajectories=True, sensitivities=True)
    torch.cuda.synchronize()
    _SENS[v.id] = raw["dtf"][:, :6].cpu().numpy()
    return B, pos, rows, solver, raw


@pytest.mark.parametrize("v", VARIANTS, ids=[v.id for v in VARIANTS])
def test_variant_matches_oracle(lm, golden_dir, sms, v):
    """Oracle parity of the embedded problems, bitwise position invariance of the copies, and d tf / d parameter
    of the first six problems against central differences of oracle solves (make_golden.py --sens-batch)."""
    B, pos, rows, solver, raw = _solve_variant(lm, v, sms)
    assert int((raw["status"] != 0).sum()) == 0, torch.bincount(raw["status"].cpu().long())
    _assert_copies_identical(raw, pos)
    sg = np.load(os.path.join(golden_dir, "sens_disp6_seed11_nt200.npz"))
    d = 0 if v.dcost > 0 else 1
    assert float(sg["dcost"][d]) == v.dcost and list(sg["names"]) == SENS_NAMES     # the rows of lmato_sens_t
    dtf = raw["dtf"].cpu().numpy()
    if v.model == "circular":
        gold = np.load(os.path.join(golden_dir, "circular_dcost1e-5_nt200.npz" if v.dcost > 0 else "circular_nominal_nt200.npz"))
        names = list(gold["names"])
        tf = float(raw["tf"][0])
        tf_err = abs(tf - float(gold["tf"])) / float(gold["tf"])
        assert tf_err < 1e-10, tf_err
        t = raw["traj"][:, :, 0].cpu().numpy()
        st_err = max(np.abs(t[VAR_ROWS.index(n)] - gold["traj"][names.index(n)]).max() /
                     np.abs(gold["traj"][names.index(n)]).max() for n in CIRCULAR_ROWS)
        assert st_err < 1e-6, st_err                 # (the bounds of test_circular_model_matches_golden_and_pdf)
        # d tf / d (Ft, M0, M_dot); the pitch-acceleration limit is not a parameter of this model: NaN
        sens_err = np.abs(dtf[:3, 0] - sg["circ_dtf"][d]) / np.abs(sg["circ_dtf"][d])
        sens_tol = np.full(3, SENS_RTOL["circular"])
        assert np.isnan(dtf[3]).all()
        mv99 = 0.0
    else:
        if v.dcost > 0:
            g = np.load(os.path.join(golden_dir, "elliptical_config4_dcost_disp512_seed11_nt200.npz"))
            nodes = g["nodes"]
        else:
            g = np.load(os.path.join(golden_dir, "elliptical_dispersions8_seed11_nt200.npz"))
            nodes = np.arange(200)
        n = g["tf"].size
        keep = np.array([b for b in range(n) if b == 0 or b not in pos])
        assert np.array_equal(rows[:, keep].numpy(), g["rows"][:, keep])
        ok = keep[g["kkt"][keep] < 1e-9] if "kkt" in g.files else keep
        assert ok.size > 0.99 * keep.size
        tf = raw["tf"][:n].cpu().numpy(); fm = raw["final_mass"][:n].cpu().numpy()
        tf_err = float(np.max(np.abs(tf - g["tf"])[ok] / g["tf"][ok]))
        fm_err = float(np.max(np.abs(fm - g["final_mass"])[ok] / g["final_mass"][ok]))
        assert tf_err < 1e-7 and fm_err < 1e-7, (tf_err, fm_err)
        full = raw["traj"][:, :, :n].permute(2, 0, 1).cpu().numpy()          # [n, 10, nt]
        err = _rel_err(full, g["traj"], nodes)[ok]
        st_err = float(err[:, :9].max())
        mv99 = float(np.quantile(err[:, 9], 0.99))
        assert st_err < STATE_RTOL, err[:, :9].max(axis=0)
        assert mv99 < 5e-3, mv99                                         # the MV on the singular arc
        assert np.all(full[:, :, 0] == 0.0)                              # node 0 pinned
        fd = sg["dtf"][d]                                                          # [6, 4]
        sens_err = np.abs(dtf[:, :6].T - fd) / np.abs(fd)
        spread = np.abs(sg["tf_up"][d] - 2 * sg["tf"][d][:, None] + sg["tf_dn"][d]) / sg["step"] / np.abs(fd)
        sens_tol = np.full((6, 4), SENS_RTOL["dcost" if v.dcost > 0 else "nodcost"])
        sens_tol[:, 3] = SENS_ADDM_RTOL + spread[:, 3]
        # physically: more thrust shortens the burn, more mass lengthens it
        assert np.all(dtf[0, :6] < 0) and np.all(dtf[1, :6] > 0)
    print(f"\n[kernel-matrix] {v.id} B={B}: tf {tf_err:.1e} states {st_err:.1e} mv99 {mv99:.1e} "
          f"sens {sens_err.reshape(-1, sens_err.shape[-1]).max(axis=0)} of {sens_tol.reshape(-1, sens_tol.shape[-1]).min(axis=0)} "
          f"(err/tol {np.max(sens_err / sens_tol):.2f}; addm {sens_err.reshape(-1, sens_err.shape[-1])[:, -1]})")
    assert np.all(sens_err < sens_tol), (sens_err, sens_tol)
    if v.id == "thread-sweeps7":
        # host entry point (staged copies) and device entry point give the same bits, sensitivities included (on a
        # fresh handle: a used one starts its warm-start reference solve from the previous reference)
        host = _solver(lm, v).solve_rows(rows, trajectories=True, sensitivities=True)
        for k in ("tf", "status", "iterations", "dtf", "traj"):
            assert torch.equal(host[k], raw[k].cpu()), k


def test_sensitivities_agree_across_variants(lm, sms):
    """The same problem's d tf / d parameter from every kernel instantiation: the multipliers of the same
    converged point, read through each workspace layout and writer."""
    for v in VARIANTS:
        if v.id not in _SENS and v.model == "elliptical" and v.batch(sms) is not None:
            _solve_variant(lm, v, sms)
    for dcost in (1e-5, 0.0):
        got = np.stack([_SENS[v.id] for v in VARIANTS if v.model == "elliptical" and v.dcost == dcost and v.id in _SENS])
        assert got.shape[0] >= 2
        spread = float((np.abs(got - got[:1]) / np.abs(got[:1])).max())
        print(f"\n[kernel-matrix] dcost {dcost}: d tf / d parameter spread across {got.shape[0]} variants {spread:.1e}")
        assert spread < 1e-8, spread


START_POINTS = [("thread-sweeps8", "thread", 0, 1e-5), ("thread-sweeps7", "thread", 0, 0.0),
                ("coop-gp8", "coop", 8, 1e-5), ("coop-gp8-move0", "coop", 8, 0.0), ("coop-gp32", "coop", 32, 1e-5)]


@pytest.mark.parametrize("vid,kernel,lanes,dcost", START_POINTS, ids=[s[0] for s in START_POINTS])
def test_start_points(lm, golden_dir, vid, kernel, lanes, dcost):
    """`guess=` on each kernel (start_from_guess through its own layout): the fixture problems started from the solutions of the same problems
    at +0.5 % thrust reach the oracle's optimum in fewer iterations than from the cold start; on the thread kernel an
    all-zero start point is abandoned and the problem restarted from the roll-out, which reaches the cold optimum."""
    if dcost > 0:
        g = np.load(os.path.join(golden_dir, "elliptical_config4_dcost_disp512_seed11_nt200.npz"))
        B, nodes = 64, g["nodes"]
    else:
        g = np.load(os.path.join(golden_dir, "elliptical_dispersions8_seed11_nt200.npz"))
        B, nodes = 8, np.arange(200)
    rows = lm.dispersed_params(B, seed=11).rows(B)
    assert np.array_equal(rows.numpy(), g["rows"][:, :B])
    solver = lm.AscentSolver(lm.Mesh(), lm.SolverOptions(dcost=dcost, kernel=kernel, coop_lanes=lanes), device=0)
    rows = rows.cuda()
    up = rows.clone()
    up[3] *= 1.005                                      # row LMATO_P_FT (thrust)
    near = solver.solve_rows(up)
    cold = solver.solve_rows(rows)
    warm = solver.solve_rows(rows, guess={"traj": near["traj"], "tf": near["tf"]})
    torch.cuda.synchronize()
    for r in (near, cold, warm):
        assert int((r["status"] != 0).sum()) == 0
    ok = np.arange(B)[g["kkt"][:B] < 1e-9] if "kkt" in g.files else np.arange(B)
    tf = warm["tf"].cpu().numpy()
    assert np.max(np.abs(tf - g["tf"][:B])[ok] / g["tf"][:B][ok]) < 1e-7
    full = warm["traj"].permute(2, 0, 1).cpu().numpy()
    err = _rel_err(full, g["traj"][:B], nodes)[ok]
    assert err[:, :9].max() < STATE_RTOL and np.quantile(err[:, 9], 0.99) < 5e-3
    it_warm, it_cold = float(warm["iterations"].double().mean()), float(cold["iterations"].double().mean())
    print(f"\n[kernel-matrix] start points {vid}: iterations {it_warm:.1f} from the neighbours' solutions, {it_cold:.1f} cold")
    # The start point is consumed (the iterates differ from the cold start's).  It carries primal values only: the
    # barrier parameter starts again at mu_init, so a neighbour's solution costs about as many iterations as the
    # roll-out (measured on a B200: 30.2 against 29.9 with DCOST, 26.5 against 26.0 without).
    assert not torch.equal(warm["iterations"], cold["iterations"])
    assert it_warm <= it_cold + 1.0
    if kernel == "thread":
        zero = solver.solve_rows(rows, trajectories=False,
                                 guess={"traj": torch.zeros_like(near["traj"]), "tf": torch.zeros_like(near["tf"])})
        torch.cuda.synchronize()
        assert int((zero["status"] != 0).sum()) == 0, zero["status"].tolist()
        assert float(((zero["tf"] - cold["tf"]).abs() / cold["tf"]).max()) < 1e-8


COARSE_KERNELS = [("thread", 0), ("coop", 8), ("coop", 32)]


def _coarse_cases():
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "elliptical_coarse_nt3to33.npz"))
    return [(i, int(nt), float(dc)) for i, (nt, dc) in enumerate(zip(g["nt"], g["dcost"]))]


@pytest.mark.parametrize("kernel,lanes", COARSE_KERNELS, ids=["thread", "coop-gp8", "coop-gp32"])
@pytest.mark.parametrize("case,nt,dcost", _coarse_cases(),
                         ids=[f"nt{nt}-{'dcost' if dc > 0 else 'nodcost'}" for _, nt, dc in _coarse_cases()])
def test_coarse_mesh(lm, golden_dir, case, nt, dcost, kernel, lanes):
    """Meshes of 3 to 33 nodes: a cooperative group then has lanes that own no stage, and its record ring prefetches
    past the last stage.  One problem alone and 40 copies of it against the oracle (make_golden.py --coarse)."""
    g = np.load(os.path.join(golden_dir, "elliptical_coarse_nt3to33.npz"))
    gold = g[f"traj_{case}"]
    solver = lm.AscentSolver(lm.Mesh(nt=nt), lm.SolverOptions(dcost=dcost, kernel=kernel, coop_lanes=lanes), device=0)
    rows = lm.AscentParams().rows(40).cuda()
    worst = 0.0
    for B in (1, 40):
        raw = solver.solve_rows(rows[:, :B].contiguous())
        torch.cuda.synchronize()
        assert raw["status"].tolist() == [0] * B
        tf = raw["tf"].cpu().numpy()
        assert np.abs(tf - float(g["tf"][case])).max() < 1e-9, (tf[0], float(g["tf"][case]))
        t = raw["traj"].cpu().numpy()                       # [10, nt, B]
        assert np.all(t[:, 0, :] == 0.0)                    # node 0 pinned
        err = (np.abs(t[:9] - gold[:9, :, None]) / (np.abs(gold[:9]).max(axis=1)[:, None, None] + 1e-300)).max()
        worst = max(worst, float(err))
        assert err < 1e-6, err
        assert np.all(t == t[:, :, :1]) and np.all(tf == tf[0])
        assert np.all(raw["iterations"].cpu().numpy() == int(raw["iterations"][0]))
    print(f"\n[kernel-matrix] coarse nt={nt} dcost={dcost} {kernel}/{lanes}: tf {abs(tf[0] - float(g['tf'][case])):.1e} "
          f"states {worst:.1e}")
