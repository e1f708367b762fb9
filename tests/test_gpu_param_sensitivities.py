"""d tf / d params[p] for every row p of the parameter block (lmato_set_param_sensitivity_output) on the GPU: every
NODES = 2 kernel instantiation of tests/dispatch_rules.py against the oracle's central differences (make_sens_all.py)
and against each other, the exact identities of the rows on a 4 096-problem batch, the host and device
entry points, the device list, the other outputs' bits, and the final-mass derivatives that the Python API forms
from these rows.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from dispatch_rules import VARIANTS

pytestmark = pytest.mark.gpu

NAMES = ["G", "M", "R0", "Ft", "M0", "M_dot", "fuel_mass", "angle_doubledot_max", "r_periapsis", "r_apoapsis",
         "final_time", "mass_scalar", "angle_ub", "u_bound"]
P = {n: i for i, n in enumerate(NAMES)}
OLD = [P["Ft"], P["M0"], P["M_dot"], P["angle_doubledot_max"]]          # the rows of lmato_sens_t, in its order
HOMOGENEOUS = [P[n] for n in ("Ft", "M0", "M_dot", "fuel_mass", "mass_scalar")]
KEYS = ("tf", "final_mass", "status", "iterations", "kkt", "traj")


@pytest.fixture(scope="module")
def lm(built_lib):
    import lunar_module_ascent_trajectory_optimiser_b200 as lm
    assert torch.cuda.is_available()
    return lm


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def fixture(golden_dir):
    g = np.load(os.path.join(golden_dir, "sens_all_disp6_seed11_nt200.npz"))
    assert list(g["names"]) == NAMES
    return g


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p()


def _solver(lm, v, nt=200):
    return lm.AscentSolver(lm.Mesh(nt=nt), lm.SolverOptions(dcost=v.dcost, kernel=v.kernel, coop_lanes=v.coop_lanes),
                           device=0, model=v.model)


def _copies(B, gp):
    """Positions of the nominal copies (as tests/test_gpu_kernel_matrix.py places them)."""
    pos = {0, 31, 32, 255, 256, B // 2, B - 2, B - 1}
    if gp == 8:
        pos |= {35, 36, 4 * (B // 4) - 1}
    return sorted(p for p in pos if 0 <= p < B)


def _rows(lm, v, B, pos):
    if v.model == "circular":
        return lm.AscentParams.circular().rows(B)
    rows = lm.dispersed_params(B, seed=11).rows(B)
    rows[:, pos] = rows[:, :1]
    return rows


def _check_against_fd(got, fd, up, dn, tf0, step, raw, tf, dcost):
    """got, fd: [14] (NaN rows skipped).  The bounds of test_param_sensitivities_on_host.py: rows of lmato_sens_t as
    test_gpu_kernel_matrix.py bounds them, every other row err < rtol + spread, rows of zero derivative absolutely."""
    rtol = 3e-5 if dcost > 0 else 5e-6
    worst = 0.0
    for j in range(14):
        if np.isnan(got[j]):
            continue
        if abs(fd[j] * raw[j] / tf) < 1e-9:
            assert abs(got[j] * raw[j] / tf) < 1e-6, (NAMES[j], got[j], fd[j])
            continue
        err = abs(got[j] - fd[j]) / abs(fd[j])
        spread = abs(up[j] - 2 * tf0 + dn[j]) / step[j] / abs(fd[j])
        tol = 1e-5 + spread if j == P["angle_doubledot_max"] else rtol if j in OLD else rtol + spread
        worst = max(worst, err / tol)
        assert err < tol, (NAMES[j], dcost, got[j], fd[j], err, tol)
    return worst


_ALL = {}     # variant id -> d tf / d params of its first 6 problems, for the cross-variant check


@pytest.mark.parametrize("v", VARIANTS, ids=[v.id for v in VARIANTS])
def test_variant_matches_oracle(lm, fixture, sms, v):
    """Every kernel instantiation: the fixture problems against the oracle's central differences of all 14 rows,
    and every copy of the nominal problem in one launch with the same bits."""
    B = v.batch(sms)
    if B is None:
        pytest.skip(f"{v.id}: empty batch-size window on a GPU with {sms} SMs")
    exp = v.expect(sms, B)
    pos = list(range(B)) if v.model == "circular" else _copies(B, exp[1] if exp[0] == "coop" else 32)
    rows = _rows(lm, v, B, pos)
    raw = _solver(lm, v).solve_rows(rows.cuda(), trajectories=False, sensitivities="all")
    torch.cuda.synchronize()
    assert "dtf" not in raw and tuple(raw["dtf_all"].shape) == (14, B)
    assert int((raw["status"] != 0).sum()) == 0
    d = raw["dtf_all"][:, pos]
    assert bool(((d == d[:, :1]) | (torch.isnan(d) & torch.isnan(d[:, :1]))).all()), d
    dtf, tf, g = raw["dtf_all"].cpu().numpy(), raw["tf"].cpu().numpy(), fixture
    k = 0 if v.dcost > 0 else 1
    assert float(g["dcost"][k]) == v.dcost
    if v.model == "circular":
        assert np.isnan(dtf[[P["angle_doubledot_max"], P["u_bound"]]]).all()
        worst = _check_against_fd(dtf[:, 0], g["circ_dtf"][k], g["circ_tf_up"][k], g["circ_tf_dn"][k], g["circ_tf"][k],
                                  g["circ_step"], rows[:, 0].numpy(), tf[0], v.dcost)
    else:
        assert not np.isnan(dtf[:, :6]).any()
        assert np.array_equal(rows[:, :6].numpy(), g["rows"])
        worst = max(_check_against_fd(dtf[:, b], g["dtf"][k, b], g["tf_up"][k, b], g["tf_dn"][k, b], g["tf"][k, b],
                                      g["step"][b], g["rows"][:, b], tf[b], v.dcost) for b in range(6))
        _ALL[v.id] = dtf[:, :6]
    print(f"\n[param-sens] {v.id} B={B}: worst err/tol {worst:.2f}")


def test_variants_agree(lm, sms):
    """The same problems' rows from every elliptical instantiation agree to 1e-8 (rows of zero derivative: against
    1e-3 of an elasticity)."""
    if len(_ALL) < 2:
        pytest.skip("needs the variant tests of this module")
    tf_scale = 1e-3 * 0.92
    rows = lm.dispersed_params(6, seed=11).rows(6).numpy()
    for dcost in (1e-5, 0.0):
        got = np.stack([_ALL[v.id] for v in VARIANTS if v.model == "elliptical" and v.dcost == dcost and v.id in _ALL])
        assert got.shape[0] >= 2
        scale = np.maximum(np.abs(got[:1]), tf_scale / np.abs(rows))
        spread = float((np.abs(got - got[:1]) / scale).max())
        print(f"\n[param-sens] dcost {dcost}: spread across {got.shape[0]} variants {spread:.1e}")
        assert spread < 1e-8, spread


def _identities(d, rows, tf):
    gm = rows[P["G"]] * d[P["G"]]
    out = {"G*M": (gm - rows[P["M"]] * d[P["M"]]).abs() / gm.abs()}
    terms = rows[HOMOGENEOUS] * d[HOMOGENEOUS]
    out["homogeneous"] = terms.sum(0).abs() / terms.abs().sum(0)
    out["T"] = (rows[P["final_time"]] * d[P["final_time"]] + tf).abs() / tf
    return out


@pytest.mark.parametrize("kernel", ["thread", "coop"])
def test_identities_on_a_dispersed_batch(lm, kernel):
    """4 096 dispersions (seed 5): G dtf/dG = M dtf/dM and the degree-0 homogeneity in (Ft, M0, M_dot, fuel_mass,
    mass_scalar) with and without DCOST; T dtf/dT = -tf without DCOST where tf < tf_ub."""
    B = 4096
    rows = lm.dispersed_params(B, seed=5).rows(B).cuda()
    for dcost in (1e-5, 0.0):
        s = lm.AscentSolver(lm.Mesh(), lm.SolverOptions(dcost=dcost, kernel=kernel), device=0)
        raw = s.solve_rows(rows, trajectories=False, sensitivities="all")
        torch.cuda.synchronize()
        ok = raw["status"] == 0
        assert float(ok.double().mean()) > 0.99
        tf = raw["tf"]
        res = _identities(raw["dtf_all"], rows, tf)
        tf_ub = torch.clamp(rows[P["fuel_mass"]] / (rows[P["M_dot"]] * rows[P["final_time"]]), max=1.0)
        worst = {}
        for k, r in res.items():
            m = ok & (tf < tf_ub) if k == "T" else ok
            if k == "T" and dcost > 0:
                continue
            worst[k] = float(r[m].max())
            assert int(m.sum()) > 0.9 * B, k
        print(f"\n[param-sens] identities {kernel} dcost {dcost}: {worst}")
        assert all(w < 1e-8 for w in worst.values()), worst


def _solve_with(lm, rows, old, new, kernel="thread", dcost=0.0, model="elliptical"):
    """One solve on a fresh handle with the four-row output and / or the new one registered on the device."""
    s = lm.AscentSolver(lm.Mesh(), lm.SolverOptions(dcost=dcost, kernel=kernel), device=0, model=model)
    B = int(rows.shape[1])
    extra = torch.full((14, B), float("nan"), dtype=torch.float64, device="cuda") if new else None
    L = lm._cabi.lib()
    if new:
        assert L.lmato_set_param_sensitivity_output(s._h, _ptr(extra)) == 0
    raw = s.solve_rows(rows.cuda(), trajectories=True, sensitivities=old)
    torch.cuda.synchronize()
    L.lmato_set_param_sensitivity_output(s._h, C.c_void_p())
    s.close()
    out = {k: v.cpu() for k, v in raw.items() if v is not None}
    if new:
        out["dtf_all"] = extra.cpu()
    return out


@pytest.mark.parametrize("kernel,dcost,model", [("thread", 0.0, "elliptical"), ("thread", 1e-5, "elliptical"),
                                                ("coop", 0.0, "elliptical"), ("coop", 1e-5, "elliptical"),
                                                ("coop", 1e-5, "circular")])
def test_other_outputs_keep_their_bits(lm, kernel, dcost, model):
    """Registering the new output changes no bit of tf, final mass, trajectories, status, iterations, KKT error or
    the four-row output, on the device, whether the four-row output is registered or not; the new output's four
    overlapping rows are the four-row output's bits.  (The four-row output itself has always written the trajectory's
    acceleration rows from the derivative pass, which may differ from the plain evaluation in the last bit.)"""
    B = 600                                          # >= 512: the batch warm start runs too
    rows = (lm.AscentParams.circular().rows(B) if model == "circular" else lm.dispersed_params(B, seed=11).rows(B))
    none = _solve_with(lm, rows, False, False, kernel, dcost, model)
    old = _solve_with(lm, rows, True, False, kernel, dcost, model)
    new = _solve_with(lm, rows, False, True, kernel, dcost, model)
    both = _solve_with(lm, rows, True, True, kernel, dcost, model)
    for k in KEYS:
        assert torch.equal(new[k], none[k]), k
        assert torch.equal(both[k], old[k]), k
        if k != "traj":
            assert torch.equal(old[k], none[k]), k
    eq = lambda a, b: bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all())
    assert eq(old["dtf"], both["dtf"])
    assert eq(new["dtf_all"], both["dtf_all"])
    assert eq(both["dtf_all"][OLD], both["dtf"])


def test_host_and_device_entries_give_the_same_bits(lm):
    """lmato_solve_batch_host with a pinned and with a pageable output, and lmato_solve_batch: the same bits."""
    B = 1000
    rows = lm.dispersed_params(B, seed=11).rows(B)
    opt = lm.SolverOptions(dcost=0.0, kernel="thread")

    def run(rows_in, dest=None):
        s = lm.AscentSolver(lm.Mesh(), opt, device=0)
        if dest is not None:
            assert lm._cabi.lib().lmato_set_param_sensitivity_output(s._h, C.c_void_p(dest.data_ptr())) == 0
            r = s.solve_rows(rows_in, trajectories=True)
            lm._cabi.lib().lmato_set_param_sensitivity_output(s._h, C.c_void_p())
            r = dict(r, dtf_all=dest)
        else:
            r = s.solve_rows(rows_in, trajectories=True, sensitivities="all")
        torch.cuda.synchronize()
        s.close()
        return {k: v.cpu() for k, v in r.items() if v is not None}

    dev = run(rows.cuda())
    pinned = run(rows.pin_memory())
    pageable = run(rows, dest=torch.full((14, B), float("nan"), dtype=torch.float64))
    assert not pageable["dtf_all"].is_pinned()
    for r in (pinned, pageable):
        for k in KEYS + ("dtf_all",):
            assert torch.equal(r[k], dev[k]), k
    # the device entry refuses a host buffer, the host entry a device buffer
    s = lm.AscentSolver(lm.Mesh(), opt, device=0)
    L = lm._cabi.lib()
    for rows_in, dest in ((rows.cuda(), torch.zeros((14, B), dtype=torch.float64)),
                          (rows, torch.zeros((14, B), dtype=torch.float64, device="cuda"))):
        assert L.lmato_set_param_sensitivity_output(s._h, C.c_void_p(dest.data_ptr())) == 0
        with pytest.raises(lm.LmatoError):
            s.solve_rows(rows_in, trajectories=False)
        L.lmato_set_param_sensitivity_output(s._h, C.c_void_p())
    s.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_devices_give_the_same_bits(lm):
    """devices=[0, 1] against one GPU (thread kernel, cold starts: every problem's solve is independent of its
    shard)."""
    B = 300
    p = lm.dispersed_params(B, seed=11)
    opt = lm.SolverOptions(dcost=0.0, kernel="thread")
    one = lm.optimise_batch(p, options=opt, device=0, sensitivities="all", trajectories=False)
    two = lm.optimise_batch(p, options=opt, devices=[0, 1], sensitivities="all", trajectories=False)
    for n in NAMES:
        assert torch.equal(one.dtf_dparam[n].cpu(), two.dtf_dparam[n].cpu()), n
        assert torch.equal(one.dfinal_mass_dparam[n].cpu(), two.dfinal_mass_dparam[n].cpu()), n
    assert torch.equal(one.tf.cpu(), two.tf.cpu())


def test_nodes3_rejects_the_output(lm):
    s = lm.AscentSolver(lm.Mesh(nt=40, nodes=3), lm.SolverOptions(dcost=0.0), device=0)
    with pytest.raises(lm.LmatoError):
        s.solve_rows(lm.AscentParams(dcost=0.0).rows(2).cuda(), sensitivities="all")
    s.close()
    with pytest.raises(lm.LmatoError):
        lm.optimise_batch(lm.AscentParams(dcost=0.0), mesh=lm.Mesh(nt=40, nodes=3), batch=2, sensitivities="all")


def test_final_mass_derivatives_match_resolves(lm):
    """dfinal_mass_dparam, formed in Python from the rows, against central differences of final_mass over re-solves
    on the GPU: four dispersions, every row moved by a relative step (1e-3 for angle_doubledot_max and u_bound, 1e-4
    for the others), all 4 x 29 problems in one launch."""
    nb = 4
    base = lm.dispersed_params(nb, seed=11).rows(nb)
    rel = torch.tensor([1e-3 if n in ("angle_doubledot_max", "u_bound") else 1e-4 for n in NAMES], dtype=torch.float64)
    step = rel[:, None] * base                                         # [14, nb]
    cols = [base]
    for j in range(14):
        for s in (1.0, -1.0):
            r = base.clone()
            r[j] += s * step[j]
            cols.append(r)
    rows = torch.cat(cols, dim=1)                                      # [14, nb * 29]
    opt = lm.SolverOptions(dcost=0.0, kernel="thread")
    sol = lm.optimise_batch(lm.AscentParams(**{n: rows[i] for i, n in enumerate(NAMES)}, dcost=0.0), options=opt,
                            device=0, trajectories=False, sensitivities="all")
    assert int((sol.status != 0).sum()) == 0
    fm = sol.final_mass.cpu().reshape(29, nb)
    tf = sol.tf.cpu()[:nb]
    worst = 0.0
    for j, n in enumerate(NAMES):
        up, dn = fm[1 + 2 * j], fm[2 + 2 * j]
        fd = (up - dn) / (2 * step[j])
        spread = (up - 2 * fm[0] + dn).abs() / step[j]
        got = sol.dfinal_mass_dparam[n].cpu()[:nb]
        for b in range(nb):
            elastic = abs(float(fd[b] * base[j, b] / fm[0, b]))
            if elastic < 1e-9:
                assert abs(float(got[b] * base[j, b] / fm[0, b])) < 1e-6, (n, b)
                continue
            err = abs(float(got[b] - fd[b])) / abs(float(fd[b]))
            tol = 5e-6 + float(spread[b]) / abs(float(fd[b]))
            worst = max(worst, err / tol)
            assert err < tol, (n, b, float(got[b]), float(fd[b]), err, tol)
    # the formula itself: M0 - M_dot * final_time * tf
    i = P
    want = -(base[i["M_dot"]] * base[i["final_time"]]) * sol.dtf_dparam["Ft"].cpu()[:nb]
    assert torch.equal(sol.dfinal_mass_dparam["Ft"].cpu()[:nb], want)
    assert float(tf.min()) > 0
    print(f"\n[param-sens] final mass: worst err/tol {worst:.2f}")


def test_circular_model_rows_it_does_not_read_are_nan(lm):
    sol = lm.optimise_batch(lm.AscentParams.circular(), batch=3, sensitivities="all", trajectories=False)
    assert int((sol.status != 0).sum()) == 0
    for n in NAMES:
        v = sol.dtf_dparam[n].cpu()
        if n in ("angle_doubledot_max", "u_bound"):
            assert torch.isnan(v).all() and torch.isnan(sol.dfinal_mass_dparam[n].cpu()).all(), n
        else:
            assert not torch.isnan(v).any(), n
    # sensitivities=True keeps its four keys
    four = lm.optimise_batch(lm.AscentParams.circular(), batch=3, sensitivities=True, trajectories=False)
    assert list(four.dtf_dparam) == ["Ft", "M0", "M_dot", "angle_doubledot_max"] and four.dfinal_mass_dparam is None
