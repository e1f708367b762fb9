"""d tf / d params[p] for every row p of the parameter block (lmato_set_param_sensitivity_output), as the kernels' result
writer (csrc/ascent_result.cuh) forms it, run on the CPU through tools/hostsim in the thread workspace layout
(hostsim_solve: Sweeps7 / Sweeps8) and the cooperative one (hostsim_solve_coop).

Three independent checks: the oracle's central differences (make_sens_all.py), identities that follow from
how the parameters enter the model and need no differences at all, and agreement between the two layouts.  Registering
the output must change no other output bit.
"""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
NAMES = ["G", "M", "R0", "Ft", "M0", "M_dot", "fuel_mass", "angle_doubledot_max", "r_periapsis", "r_apoapsis",
         "final_time", "mass_scalar", "angle_ub", "u_bound"]
P = {n: i for i, n in enumerate(NAMES)}
OLD = [P["Ft"], P["M0"], P["M_dot"], P["angle_doubledot_max"]]        # the rows of lmato_sens_t, in its order
HOMOGENEOUS = [P[n] for n in ("Ft", "M0", "M_dot", "fuel_mass", "mass_scalar")]
LAYOUTS = ("hostsim_solve", "hostsim_solve_coop")
CIRCULAR = np.array([6.674e-11, 7.346e22, 1738100.0, 15346.0, 4821.0, 5.053, 2376.0, 5e-4, 53108.4, 53108.4, 470.0,
                     2576.0, np.pi / 3, 1.0])


@pytest.fixture(scope="module")
def hostsim(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    so = str(tmp_path_factory.mktemp("hostsim") / "libhostsim.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-I",
                           os.path.join(ROOT, "lunar_module_ascent_trajectory_optimiser_b200", "csrc"),
                           os.path.join(ROOT, "tools", "hostsim", "hostsim.cpp"), "-o", so])
    return C.CDLL(so)


@pytest.fixture(scope="module")
def fixture():
    return np.load(os.path.join(GOLDEN, "sens_all_disp6_seed11_nt200.npz"))


def _regime(monkeypatch, dcost, circular=False):
    """The environment hostsim reads: the move weight of the library's default objective (obj_scale * dcost / (nt - 1))
    and its polish count, and the model."""
    if dcost > 0:
        monkeypatch.setenv("WDC", repr(10.0 * dcost / 199)); monkeypatch.setenv("NPOL", "2")
    else:
        monkeypatch.delenv("WDC", raising=False); monkeypatch.delenv("NPOL", raising=False)
    if circular:
        monkeypatch.setenv("CIRCULAR", "1")
    else:
        monkeypatch.delenv("CIRCULAR", raising=False)
    monkeypatch.delenv("VREC", raising=False)


def _solve(L, raw, fn, old=False, new=True, nt=200):
    """One solve with the old four-row output and / or the new one registered: every output of it."""
    raw = np.ascontiguousarray(raw, dtype=np.float64)
    traj = np.empty((10, nt))
    tf, it, kkt = C.c_double(), C.c_int(), C.c_double()
    s4, s14 = np.full(4, np.nan), np.full(14, np.nan)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    L.hostsim_set_sensitivity_output(ptr(s4) if old else None)
    L.hostsim_set_param_sensitivity_output(ptr(s14) if new else None)
    try:
        st = getattr(L, fn)(ptr(raw), nt, None, C.c_double(1e-10), C.c_double(10.0), C.c_double(1e-3), ptr(traj),
                            C.byref(tf), C.byref(it), C.byref(kkt))
    finally:
        L.hostsim_set_sensitivity_output(None)
        L.hostsim_set_param_sensitivity_output(None)
    return dict(status=st, tf=tf.value, iters=it.value, kkt=kkt.value, traj=traj, dtf=s4, dtf_all=s14)


def _check_against_fd(got, fd, up, dn, tf0, step, raw, tf, dcost, old_rows_tol):
    """got, fd: [14].  Per row: err < rtol + spread (the one-sided quotients' spread bounds the truncation error at a
    kink); rows whose quotient is zero (an inactive bound) in absolute terms; the rows of lmato_sens_t keep the bounds
    of test_sensitivity_writer_matches_finite_differences.  Returns the worst err / tol."""
    rtol = 3e-5 if dcost > 0 else 5e-6
    worst = 0.0
    for j in range(14):
        if np.isnan(got[j]):
            continue
        if abs(fd[j] * raw[j] / tf) < 1e-9:
            e = abs(got[j] * raw[j] / tf)
            assert e < 1e-6, (NAMES[j], got[j], fd[j])
            continue
        err = abs(got[j] - fd[j]) / abs(fd[j])
        spread = abs(up[j] - 2 * tf0 + dn[j]) / step[j] / abs(fd[j])
        if j in old_rows_tol:
            tol = old_rows_tol[j](spread)
        else:
            tol = rtol + spread
        worst = max(worst, err / tol)
        assert err < tol, (NAMES[j], dcost, got[j], fd[j], err, tol)
    return worst


def _layouts_agree(a, b, raw, tf):
    for j in range(14):
        if np.isnan(a[j]) or np.isnan(b[j]):
            assert np.isnan(a[j]) and np.isnan(b[j]), NAMES[j]
            continue
        scale = max(abs(a[j]), 1e-3 * tf / abs(raw[j]))      # (rows of zero derivative: against 1e-3 of an elasticity)
        assert abs(a[j] - b[j]) / scale < 1e-8, (NAMES[j], a[j], b[j])


def test_every_row_matches_the_oracle_on_both_layouts(hostsim, fixture, monkeypatch):
    """The six seed-11 dispersions at DCOST 1e-5 and 0, and the circular model's nominal problem, against the oracle's
    central differences of every row; both layouts read the multipliers of the same optimum."""
    g = fixture
    assert list(g["names"]) == NAMES
    for d, dcost in enumerate(g["dcost"].tolist()):
        rtol = 3e-5 if dcost > 0 else 5e-6
        old_tol = {P["Ft"]: lambda s: rtol, P["M0"]: lambda s: rtol, P["M_dot"]: lambda s: rtol,
                   P["angle_doubledot_max"]: lambda s: 1e-5 + s}
        _regime(monkeypatch, dcost)
        worst = 0.0
        for b in range(6):
            raw = g["rows"][:, b]
            got = {}
            for fn in LAYOUTS:
                r = _solve(hostsim, raw, fn)
                assert r["status"] == 0
                got[fn] = r["dtf_all"]
                assert not np.isnan(got[fn]).any()
                worst = max(worst, _check_against_fd(got[fn], g["dtf"][d, b], g["tf_up"][d, b], g["tf_dn"][d, b],
                                                     g["tf"][d, b], g["step"][b], raw, r["tf"], dcost, old_tol))
            _layouts_agree(got[LAYOUTS[0]], got[LAYOUTS[1]], raw, r["tf"])
        print(f"\n[param-sens] dcost {dcost}: worst err/tol {worst:.2f}")
        # the circular model (the cooperative layout carries its move term, the thread layout does not)
        _regime(monkeypatch, dcost, circular=True)
        fns = ("hostsim_solve_coop",) if dcost > 0 else LAYOUTS
        got = {}
        for fn in fns:
            r = _solve(hostsim, CIRCULAR, fn)
            assert r["status"] == 0
            got[fn] = r["dtf_all"]
            assert np.isnan(got[fn][[P["angle_doubledot_max"], P["u_bound"]]]).all()
            w = _check_against_fd(got[fn], g["circ_dtf"][d], g["circ_tf_up"][d], g["circ_tf_dn"][d], g["circ_tf"][d],
                                  g["circ_step"], CIRCULAR, r["tf"], dcost, {})
            print(f"[param-sens] circular dcost {dcost} {fn}: worst err/tol {w:.2f}")
        if len(got) == 2:
            _layouts_agree(got[LAYOUTS[0]], got[LAYOUTS[1]], CIRCULAR, r["tf"])


def _identities(d, raw, tf, check_t):
    """The three exact identities of the parameter rows, as relative residuals."""
    gm = raw[P["G"]] * d[P["G"]]
    out = {"G*M": abs(gm - raw[P["M"]] * d[P["M"]]) / abs(gm)}
    terms = raw[HOMOGENEOUS] * d[HOMOGENEOUS]
    out["homogeneous"] = abs(terms.sum()) / np.abs(terms).sum()
    if check_t:
        out["T"] = abs(raw[P["final_time"]] * d[P["final_time"]] + tf) / tf
    return out


def test_identities_on_the_oracle_fixture(fixture):
    """The identities hold for the oracle's own central differences (to their truncation and solve error): only G*M
    enters; tf is homogeneous of degree 0 in (Ft, M0, M_dot, fuel_mass, mass_scalar), which leaves the thrust
    acceleration, mflow and tf_ub unchanged; without the move term T enters only through the burn time T*tf."""
    g = fixture
    for d, dcost in enumerate(g["dcost"].tolist()):
        for b in range(6):
            tf = g["tf"][d, b]
            tf_ub = min(1.0, g["rows"][P["fuel_mass"], b] / (g["rows"][P["M_dot"], b] * g["rows"][P["final_time"], b]))
            res = _identities(g["dtf"][d, b], g["rows"][:, b], tf, dcost == 0 and tf < tf_ub)
            assert all(v < 1e-5 for v in res.values()), (dcost, b, res)
        if dcost == 0:
            res = _identities(g["circ_dtf"][d], CIRCULAR, g["circ_tf"][d], True)
            assert all(v < 1e-5 for v in res.values()), res


def test_identities_hold_exactly_on_both_layouts(hostsim, fixture, monkeypatch):
    """The same identities on the writer's rows, to 1e-8: each follows from the transcribed NLP itself, so the
    multipliers of its optimum satisfy it up to the solve's tolerance."""
    g = fixture
    for dcost in (1e-5, 0.0):
        _regime(monkeypatch, dcost)
        worst = {}
        for b in range(6):
            raw = g["rows"][:, b]
            tf_ub = min(1.0, raw[P["fuel_mass"]] / (raw[P["M_dot"]] * raw[P["final_time"]]))
            for fn in LAYOUTS:
                r = _solve(hostsim, raw, fn)
                assert r["status"] == 0
                res = _identities(r["dtf_all"], raw, r["tf"], dcost == 0 and r["tf"] < tf_ub)
                for k, v in res.items():
                    worst[k] = max(worst.get(k, 0.0), v)
                assert all(v < 1e-8 for v in res.values()), (dcost, b, fn, res)
        print(f"\n[param-sens] identities dcost {dcost}: worst {worst}")
        assert ("T" in worst) == (dcost == 0)


def test_registering_the_output_changes_no_other_bit(hostsim, fixture, monkeypatch):
    """tf, trajectories, status, iterations, KKT error and the four-row output are the same bits with and without the
    new output; the new output's rows Ft, M0, M_dot and angle_doubledot_max are the four-row output's bits."""
    g = fixture
    for dcost, circular in ((1e-5, False), (0.0, False), (0.0, True)):
        _regime(monkeypatch, dcost, circular)
        raws = [CIRCULAR] if circular else [g["rows"][:, b] for b in (0, 3)]
        for raw in raws:
            for fn in LAYOUTS:
                none = _solve(hostsim, raw, fn, old=False, new=False)
                old = _solve(hostsim, raw, fn, old=True, new=False)
                new = _solve(hostsim, raw, fn, old=False, new=True)
                both = _solve(hostsim, raw, fn, old=True, new=True)
                for k in ("status", "tf", "iters", "kkt"):
                    assert none[k] == old[k] == new[k] == both[k], (k, fn)
                assert np.array_equal(new["traj"], none["traj"]) and np.array_equal(both["traj"], old["traj"]), fn
                assert np.array_equal(old["dtf"], both["dtf"], equal_nan=True)
                assert np.array_equal(new["dtf_all"], both["dtf_all"], equal_nan=True)
                assert np.array_equal(both["dtf_all"][OLD], both["dtf"], equal_nan=True)


def test_final_mass_rows_follow_from_the_tf_rows():
    """dfinal_mass_dparam (api.py) is the chain rule through final_mass = M0 - M_dot * final_time * tf: against
    autograd of that formula with tf a function of the rows whose gradient is the given d tf / d row."""
    import torch
    from lunar_module_ascent_trajectory_optimiser_b200.api import dfinal_mass_dparam
    g = np.load(os.path.join(GOLDEN, "sens_all_disp6_seed11_nt200.npz"))
    rows = torch.tensor(g["rows"], dtype=torch.float64)                  # [14, 6]
    dtf = torch.tensor(g["dtf"][1].T.copy(), dtype=torch.float64)       # [14, 6]
    tf = torch.tensor(g["tf"][1], dtype=torch.float64)
    got = dfinal_mass_dparam(dtf, rows, tf)
    r = rows.clone().requires_grad_(True)
    tf_lin = tf + ((r - rows.detach()) * dtf).sum(0)                    # first order in the rows, exact gradient dtf
    fm = r[P["M0"]] - r[P["M_dot"]] * r[P["final_time"]] * tf_lin
    fm.sum().backward()
    assert torch.allclose(got, r.grad, rtol=1e-14, atol=0)
