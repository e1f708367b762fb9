"""The device solver's SOURCE, compiled for the host.

`csrc/ascent_model.cuh`, `ascent_ipm.cuh`, `ascent_ipm_dc.cuh`, `ascent_coop.cuh`, `ascent_colloc.cuh` and
`ascent_result.cuh` are written so that g++ accepts them (tools/hostsim): the parameter derivation, the sweeps, the
IPM driver with its start and restart steps (`ipm_start` / `ipm_restart`, the collocation start ladder included),
the model derivatives and the result writer below are the very lines the CUDA kernels run, executed by one CPU
thread.  Only the kernels' problem queue (`solve_queue`) is not run here.  The launch plan of `ascent_plan.h`
(which kernel, grid and workspace a batch gets) is checked here too.  This gives the CPU-only test tier a check of the solver's logic against the oracle's golden vectors,
and of the hand-derived derivatives and the sensitivity output against finite differences.  It is test
infrastructure only: the product has no CPU path (`_cabi.lib()` raises without
the CUDA library), and nothing here is imported by the package.
"""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
NOMINAL = np.array([6.674e-11, 7.346e22, 1738100.0, 15346.0, 4821.0, 5.053, 2376.0, 5e-4, 17703.0, 88615.0, 470.0,
                    2376.0, np.pi / 3, 1.0])


@pytest.fixture(scope="module")
def hostsim(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    so = str(tmp_path_factory.mktemp("hostsim") / "libhostsim.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-I",
                           os.path.join(ROOT, "lunar_module_ascent_trajectory_optimiser_b200", "csrc"),
                           os.path.join(ROOT, "tools", "hostsim", "hostsim.cpp"), "-o", so])
    L = C.CDLL(so)
    L.hostsim_check_derivatives.restype = C.c_double
    L.hostsim_check_derivatives.argtypes = [C.c_void_p] + [C.c_double] * 4
    return L


def _solve(L, raw, nt=200, time=None, tol=1e-10, fn="hostsim_solve"):
    raw = np.ascontiguousarray(raw, dtype=np.float64)
    traj = np.empty((10, nt))
    tf, it, kkt = C.c_double(), C.c_int(), C.c_double()
    tp = None if time is None else np.ascontiguousarray(time, dtype=np.float64).ctypes.data_as(C.c_void_p)
    st = getattr(L, fn)(raw.ctypes.data_as(C.c_void_p), nt, tp, C.c_double(tol), C.c_double(10.0), C.c_double(1e-3),
                         traj.ctypes.data_as(C.c_void_p), C.byref(tf), C.byref(it), C.byref(kkt))
    return st, tf.value, it.value, traj


def _rel(traj, gold):
    return (np.abs(traj - gold) / (np.abs(gold).max(axis=1, keepdims=True) + 1e-300)).max(axis=1)


def test_model_derivatives_match_finite_differences(hostsim):
    """accel_first / accel_second (LO:127-136 differentiated by hand) at points along a trajectory."""
    raw = NOMINAL.copy()
    for y, x, a, m in [(0.0, 0.0, 0.05, 0.0), (0.4, -3.0, 0.3, 0.3), (-0.36, -16.4, 0.51, 0.92), (1.2, -9.0, 0.9, 0.6)]:
        err = hostsim.hostsim_check_derivatives(raw.ctypes.data_as(C.c_void_p), y, x, a, m)
        assert err < 2e-6, (y, x, a, m, err)


def test_device_ipm_source_matches_goldens(hostsim, monkeypatch):
    monkeypatch.delenv("WDC", raising=False)
    monkeypatch.delenv("CIRCULAR", raising=False)
    # config 1 (7-state sweeps, no DCOST) and a non-uniform mesh
    g = np.load(os.path.join(GOLDEN, "elliptical_nominal_nt200.npz"))
    st, tf, it, traj = _solve(hostsim, NOMINAL)
    assert st == 0 and abs(tf - float(g["tf"])) / float(g["tf"]) < 1e-8
    err = _rel(traj, g["traj"])
    assert err[:9].max() < 1e-4 and err[9] < 2e-4, err
    g = np.load(os.path.join(GOLDEN, "elliptical_nominal_nonuniform60.npz"))
    st, tf, it, traj = _solve(hostsim, NOMINAL, nt=60, time=g["time"])
    assert st == 0 and abs(tf - float(g["tf"])) / float(g["tf"]) < 1e-8
    assert _rel(traj, g["traj"])[:9].max() < 1e-4
    # the reference's objective with DCOST (8-state sweeps)
    g = np.load(os.path.join(GOLDEN, "elliptical_dcost1e-5_disp4_seed11_nt200.npz"))
    monkeypatch.setenv("WDC", repr(10.0 * 1e-5 / 199))
    for b in range(2):
        st, tf, it, traj = _solve(hostsim, g["rows"][:, b])
        assert st == 0 and abs(tf - g["tf"][b]) / g["tf"][b] < 1e-8
        err = _rel(traj, g["traj"][b])
        assert err[:9].max() < 1e-4 and err[9] < 2e-4, err
    monkeypatch.delenv("WDC")
    # config 2: the circular model (structural flag coup5 = 0)
    g = np.load(os.path.join(GOLDEN, "circular_nominal_nt200.npz"))
    monkeypatch.setenv("CIRCULAR", "1")
    raw = NOMINAL.copy(); raw[8] = raw[9] = 53108.4; raw[11] = 2576.0
    st, tf, it, traj = _solve(hostsim, raw)
    assert st == 0 and abs(tf - float(g["tf"])) / float(g["tf"]) < 1e-8


def test_cooperative_sweeps_source_matches_goldens_and_thread_sweeps(hostsim, monkeypatch):
    """csrc/ascent_coop.cuh run by one lane (G = 1: the group primitives are identities): the stored-model
    phases, the row-wise congruence with its symmetrisation, the forward / adjoint recursions.  Same optimum
    and the same number of iterations as the one-thread-per-problem sweeps, on every golden case."""
    monkeypatch.delenv("WDC", raising=False)
    monkeypatch.delenv("CIRCULAR", raising=False)
    monkeypatch.delenv("NPOL", raising=False)

    def both(raw, gold_tf, gold_traj=None, tf_rtol=1e-8, iter_tol=1, **kw):
        a = _solve(hostsim, raw, fn="hostsim_solve", **kw)
        b = _solve(hostsim, raw, fn="hostsim_solve_coop", **kw)
        assert a[0] == 0 and b[0] == 0
        assert abs(a[1] - gold_tf) / gold_tf < tf_rtol and abs(b[1] - gold_tf) / gold_tf < tf_rtol
        assert abs(a[1] - b[1]) / a[1] < 1e-11
        assert abs(a[2] - b[2]) <= iter_tol, (a[2], b[2])             # iterations
        if gold_traj is not None:
            err = _rel(b[3], gold_traj)
            assert err[:9].max() < 1e-4 and err[9] < 2e-4, err
        assert _rel(b[3], a[3] + 0.0)[:9].max() < 1e-5

    g = np.load(os.path.join(GOLDEN, "elliptical_nominal_nt200.npz"))
    both(NOMINAL, float(g["tf"]), g["traj"])
    g = np.load(os.path.join(GOLDEN, "elliptical_nominal_nt40.npz"))
    both(NOMINAL, float(g["tf"]), g["traj"], nt=40)
    g = np.load(os.path.join(GOLDEN, "elliptical_nominal_nonuniform60.npz"))
    both(NOMINAL, float(g["tf"]), g["traj"], nt=60, time=g["time"])
    g = np.load(os.path.join(GOLDEN, "elliptical_dcost1e-5_disp4_seed11_nt200.npz"))
    monkeypatch.setenv("WDC", repr(10.0 * 1e-5 / 199))
    monkeypatch.setenv("NPOL", "2")
    for b in range(4):
        both(g["rows"][:, b], g["tf"][b], g["traj"][b])
    monkeypatch.delenv("WDC"); monkeypatch.delenv("NPOL")
    # coarse meshes (nt = 3..33): a cooperative group then has lanes without a stage and its record ring prefetches
    # past the last stage; the move weight is per step of THIS mesh (objective_nodes = nt - 1, as the device sets it)
    g = np.load(os.path.join(GOLDEN, "elliptical_coarse_nt3to33.npz"))
    for i, (nt, dc) in enumerate(zip(g["nt"].tolist(), g["dcost"].tolist())):
        if dc > 0:
            monkeypatch.setenv("WDC", repr(10.0 * dc / (nt - 1))); monkeypatch.setenv("NPOL", "2")
        # nt = 5 with DCOST spends ~50 iterations at mu = 0.1 under inertia correction, where rounding differences
        # grow ~10x per iteration: thrust moved by up to 3 ulp gives either sweep order anywhere from 55 to 73 iterations
        # (the unperturbed problem: 61 and 56).  Every other case agrees to one iteration.
        both(NOMINAL, float(g["tf"][i]), g[f"traj_{i}"], tf_rtol=5e-13, iter_tol=8 if (nt, dc > 0) == (5, True) else 1,
             nt=nt)
        monkeypatch.delenv("WDC", raising=False); monkeypatch.delenv("NPOL", raising=False)
    g = np.load(os.path.join(GOLDEN, "circular_nominal_nt200.npz"))
    monkeypatch.setenv("CIRCULAR", "1")
    raw = NOMINAL.copy(); raw[8] = raw[9] = 53108.4; raw[11] = 2576.0
    both(raw, float(g["tf"]))
    # the circular model WITH its move suppression (PDF p.27 src 69-73: DCOST = 1e-5 on the MV `angle`): the MV slot
    # of the 8-state cooperative sweeps holds the pitch angle; the oracle carries the term as slack pairs on the MV
    g = np.load(os.path.join(GOLDEN, "circular_dcost1e-5_nt200.npz"))
    monkeypatch.setenv("WDC", repr(10.0 * 1e-5 / 199)); monkeypatch.setenv("NPOL", "2")
    st, tf, it, traj = _solve(hostsim, raw, fn="hostsim_solve_coop")
    assert st == 0 and abs(tf - float(g["tf"])) / float(g["tf"]) < 1e-10
    names = list(g["names"])
    for n in names:
        ref = g["traj"][names.index(n)]
        mine = traj[["y", "ydot", "ydoubledot", "x", "xdot", "xdoubledot", "angle", "angledot", "mass"].index(n)]
        assert np.abs(mine - ref).max() / np.abs(ref).max() < 1e-7, n
    assert np.array_equal(traj[9], traj[6]) and np.abs(traj[7]).max() == 0.0     # MV slot == angle, angledot pinned at 0


def test_sensitivity_writer_matches_finite_differences(hostsim, monkeypatch):
    """d tf / d parameter as the kernels' result writer (csrc/ascent_result.cuh) forms it, through the thread and the
    cooperative workspace layouts, against the oracle's central differences (make_golden.py --sens-batch) with the
    bounds of tests/test_gpu_kernel_matrix.py.  Both layouts read the multipliers of the same optimum."""
    monkeypatch.delenv("CIRCULAR", raising=False)
    monkeypatch.delenv("VREC", raising=False)
    sg = np.load(os.path.join(GOLDEN, "sens_disp6_seed11_nt200.npz"))
    for d, dcost in enumerate(sg["dcost"].tolist()):
        if dcost > 0:
            monkeypatch.setenv("WDC", repr(10.0 * dcost / 199)); monkeypatch.setenv("NPOL", "2")
        else:
            monkeypatch.delenv("WDC", raising=False); monkeypatch.delenv("NPOL", raising=False)
        fd = sg["dtf"][d]                                                          # [6 problems, 4 parameters]
        spread = np.abs(sg["tf_up"][d] - 2 * sg["tf"][d][:, None] + sg["tf_dn"][d]) / sg["step"] / np.abs(fd)
        tol = np.full((6, 4), 3e-5 if dcost > 0 else 5e-6)
        tol[:, 3] = 1e-5 + spread[:, 3]               # angle_doubledot_max: the quotient's one-sided spread (kinks in tf)
        got = {}
        for fn in ("hostsim_solve", "hostsim_solve_coop"):
            got[fn] = np.full((6, 4), np.nan)
            for b in range(6):
                hostsim.hostsim_set_sensitivity_output(got[fn][b].ctypes.data_as(C.c_void_p))
                try:
                    assert _solve(hostsim, sg["rows"][:, b], fn=fn)[0] == 0
                finally:
                    hostsim.hostsim_set_sensitivity_output(None)
            err = np.abs(got[fn] - fd) / np.abs(fd)
            print(f"\n[sens] {fn} dcost {dcost}: worst per parameter {err.max(axis=0)} (err/tol {np.max(err / tol):.2f})")
            assert np.all(err < tol), (fn, dcost, err, tol)
        a, b = got["hostsim_solve"], got["hostsim_solve_coop"]
        assert (np.abs(b - a) / np.abs(a)).max() < 1e-8, (dcost, a, b)


def test_higher_order_collocation_source_matches_goldens(hostsim):
    """csrc/ascent_colloc.cuh (NODES = 3..6, LO:25) run by one lane against the oracle's fixtures: per-step LU
    condensation, dense Riccati on the coupling unknowns, multipliers from the stored factors.  The collocation
    rule comes from the C ABI (lmato_collocation_rule) and must equal the oracle's (APMonitor's tables)."""
    from lunar_module_ascent_trajectory_optimiser_b200 import _cabi
    from oracle.ascent_nlp import collocation_matrix
    g = np.load(os.path.join(GOLDEN, "elliptical_higher_order_nodes3to6.npz"))
    fn = hostsim.hostsim_solve_colloc

    def solve(raw, nt, nodes):
        m = nodes - 1
        tau = np.zeros(m); Nc = np.zeros((m, m))
        assert _cabi.lib().lmato_collocation_rule(nodes, tau.ctypes.data_as(C.c_void_p), Nc.ctypes.data_as(C.c_void_p)) == 0
        t_or, N_or = collocation_matrix(nodes)
        assert np.abs(tau - t_or[1:]).max() < 1e-14 and np.abs(Nc - N_or).max() < 1e-12
        raw = np.ascontiguousarray(raw, dtype=np.float64)
        traj = np.empty((10, nt)); tf, it, kkt = C.c_double(), C.c_int(), C.c_double()
        st = fn(raw.ctypes.data_as(C.c_void_p), nt, None, nodes, Nc.ctypes.data_as(C.c_void_p), tau.ctypes.data_as(C.c_void_p),
                C.c_double(1e-10), C.c_double(10.0), C.c_double(1e-3), traj.ctypes.data_as(C.c_void_p), C.byref(tf),
                C.byref(it), C.byref(kkt))
        return st, tf.value, it.value, traj

    for nodes in (3, 4, 5, 6):
        nt = int(g[f"nt_n{nodes}"])
        st, tf, it, traj = solve(NOMINAL, nt, nodes)
        assert st == 0 and abs(tf - float(g[f"tf_n{nodes}"])) / tf < 1e-9, (nodes, st, tf)
        err = _rel(traj, g[f"traj_n{nodes}"])
        assert err[:9].max() < 1e-6 and err[9] < 1e-4, (nodes, err)
    for b in range(3):
        st, tf, it, traj = solve(g["rows"][:, b], int(g["disp_nt"]), 3)
        assert st == 0 and abs(tf - g["disp_tf"][b]) / tf < 1e-9
        assert _rel(traj, g["disp_traj"][b])[:9].max() < 1e-5


def test_collocation_start_ladder_counts_every_start(hostsim, monkeypatch):
    """The collocation start ladder (ascent_colloc.cuh: ipm_start / ipm_restart) as the kernel runs it.  From a burn
    time guess of 0.1 the nominal problem at NODES = 3, nt = 60 fails from every start without reaching MAX_ITER, so
    the ladder runs to its last start; the first start alone takes 31 iterations before its line search fails, and
    the reported count covers all starts, not only the last."""
    from oracle.ascent_nlp import collocation_matrix
    monkeypatch.delenv("NPOL", raising=False)
    monkeypatch.setenv("TF0", "0.1")
    nt, nodes = 60, 3
    t_or, N_or = collocation_matrix(nodes)
    tau, Nc = np.ascontiguousarray(t_or[1:], dtype=np.float64), np.ascontiguousarray(N_or, dtype=np.float64)
    traj = np.empty((10, nt)); tf, it, kkt = C.c_double(), C.c_int(), C.c_double()
    st = hostsim.hostsim_solve_colloc(NOMINAL.ctypes.data_as(C.c_void_p), nt, None, nodes, Nc.ctypes.data_as(C.c_void_p),
                                      tau.ctypes.data_as(C.c_void_p), C.c_double(1e-10), C.c_double(10.0),
                                      C.c_double(1e-3), traj.ctypes.data_as(C.c_void_p), C.byref(tf), C.byref(it),
                                      C.byref(kkt))
    assert st not in (0, 1), (st, it.value)          # neither converged nor stopped at MAX_ITER: the ladder ran out
    assert it.value >= 31, it.value


def test_start_points_on_every_layout(hostsim, monkeypatch):
    """Start points through the kernels' own ipm_start / ipm_restart on both thread layouts (hostsim_solve: Sweeps8
    with DCOST, Sweeps7 without) and the cooperative layout (hostsim_solve_coop: MOVE 1 / 0): the batch reference of
    hostsim_reference (the ref_mode 1 solve), a caller's start point, an all-zero start point that has to be
    restarted from the roll-out, and a reference column that holds no reference (REF_OK = 0)."""
    monkeypatch.delenv("CIRCULAR", raising=False)
    monkeypatch.delenv("VREC", raising=False)
    nt, ref_rows = 200, 23                 # the reference buffer as the handle sizes it (the 8-state REF_ROWS)
    ptr = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    for fixture, dcost in (("elliptical_dcost1e-5_disp4_seed11_nt200.npz", True),
                           ("elliptical_dispersions8_seed11_nt200.npz", False)):
        g = np.load(os.path.join(GOLDEN, fixture))
        rows, gold_tf, gold_traj = g["rows"][:, :4], g["tf"][:4], g["traj"][:4]
        if dcost:
            monkeypatch.setenv("WDC", repr(10.0 * 1e-5 / 199)); monkeypatch.setenv("NPOL", "2")
        else:
            monkeypatch.delenv("WDC", raising=False); monkeypatch.delenv("NPOL", raising=False)
        ref = np.zeros((ref_rows, nt))
        mean = np.ascontiguousarray(rows.mean(axis=1))              # the batch-mean problem (mean_params_kernel)
        assert hostsim.hostsim_reference(ptr(mean), nt, C.c_double(1e-3), ptr(ref)) == 0
        no_ref = np.zeros((ref_rows, nt))
        # the same reference stored at twice the distance scale S_ref: lengths halved, the multipliers of their rows
        # doubled (csrc/ascent_ipm.cuh: rows F_LAM = 7.., scalar row N_ITER = 17, REF_S = 2).  Every factor is a power
        # of two, so the reader's rescaling must give the same start point bit for bit.
        rescaled = ref.copy()
        rescaled[0:4] /= 2; rescaled[7:11] *= 2; rescaled[17, 2] *= 2

        def solve(fn, b, traj=None, tf=None, column=None):
            hostsim.hostsim_set_start(ptr(traj), ptr(tf), ptr(column))
            try:
                return _solve(hostsim, rows[:, b], nt=nt, fn=fn)
            finally:
                hostsim.hostsim_set_start(None, None, None)

        warm = {}
        for fn in ("hostsim_solve", "hostsim_solve_coop"):
            cold = [solve(fn, b) for b in range(4)]
            warm[fn] = [solve(fn, b, column=ref) for b in range(4)]
            for b in range(4):
                assert cold[b][0] == 0 and warm[fn][b][0] == 0, (fn, b)
                assert abs(warm[fn][b][1] - gold_tf[b]) / gold_tf[b] < 1e-8, (fn, b)
                st, tf, it, traj = solve(fn, b, column=rescaled)
                assert (st, tf, it) == warm[fn][b][:3] and np.array_equal(traj, warm[fn][b][3]), (fn, b)
                # a caller's start point: the solution of the neighbouring problem
                n = b ^ 1
                st, tf, it, _ = solve(fn, b, np.ascontiguousarray(gold_traj[n]), np.array([gold_tf[n]]))
                assert st == 0 and abs(tf - gold_tf[b]) / gold_tf[b] < 1e-8, (fn, b)
                # an all-zero start point fails and is restarted from the roll-out: the cold optimum, more iterations
                st, tf, it, _ = solve(fn, b, np.zeros((10, nt)), np.zeros(1))
                assert st == 0 and abs(tf - cold[b][1]) / cold[b][1] < 1e-8 and it > cold[b][2], (fn, b, it, cold[b][2])
                # a reference column without a reference: the cold start, bit for bit
                st, tf, it, traj = solve(fn, b, column=no_ref)
                assert (st, tf, it) == cold[b][:3] and np.array_equal(traj, cold[b][3]), (fn, b)
            its_warm, its_cold = np.mean([w[2] for w in warm[fn]]), np.mean([c[2] for c in cold])
            print(f"\n[start] {fixture} {fn}: iterations warm {its_warm:.2f} cold {its_cold:.2f}")
            assert its_warm < its_cold, (fn, its_warm, its_cold)
        for a, c in zip(warm["hostsim_solve"], warm["hostsim_solve_coop"]):
            assert abs(a[1] - c[1]) / a[1] < 1e-11 and abs(a[2] - c[2]) <= 1, (a[:3], c[:3])


def test_launch_plan_matches_the_dispatch_rules(hostsim):
    """plan_solve (csrc/ascent_plan.h), the library's choice of kernel, grid, workspace and warm start, against the
    rules written out in tests/dispatch_rules.py, which the GPU kernel matrix uses to reach every kernel variant: on
    three SM counts, for every variant of that matrix at its batch size, and for every kernel / lanes / model / DCOST
    setting one below, at and one above each window edge."""
    from dispatch_rules import COOP_MAX_BATCH, VARIANTS, V
    L, nt = hostsim, 200
    keys = ("kind", "lanes", "bps", "move", "grid", "slots", "ws", "alloc", "warm", "use_dc")

    def plan(S, B, v, nodes=2, warm_start=1, guess=False, warm_batch=None):
        out = (C.c_int64 * len(keys))()
        L.hostsim_plan(S, nt, nodes, 1 if v.model == "circular" else 0, {"auto": 0, "thread": 1, "coop": 2}[v.kernel],
                       v.coop_lanes, C.c_double(v.dcost), warm_start, C.c_int64(B), int(guess),
                       C.c_int64(B if warm_batch is None else warm_batch), out)
        return dict(zip(keys, out))

    coop_doubles = 258 * nt       # DESIGN.md section 3b: X[2][24] + D[16] + M[2][52] + K[10] + H[8] + V[72] per stage
    ref_ws = 8 * coop_doubles * (256 // 32)      # the warm start's reference solve: one warp of one CTA
    grid = lambda B, lanes, cap: min(max(-(-B * lanes // 32), 1), cap)
    for S in (148, 132, 100):
        edges = sorted({0, 1} | {e + d for e in (8 * S, 32 * S, COOP_MAX_BATCH) for d in (-1, 0, 1)})
        cases = [(v, v.batch(S)) for v in VARIANTS if v.batch(S) is not None]
        for model, dcost in (("elliptical", 1e-5), ("elliptical", 0.0), ("circular", 1e-5), ("circular", 0.0)):
            for kernel in ("auto", "thread", "coop"):
                for lanes in (0, 8, 32):
                    cases += [(V("", None, model, dcost, kernel, lanes), B) for B in edges]
        for v, B in cases:
            p, exp = plan(S, B, v), v.expect(S, B)
            tag = (S, B, v.id, v.model, v.dcost, v.kernel, v.coop_lanes)
            assert p["use_dc"] == (v.dcost > 0), tag
            assert p["slots"] == 256 * grid(B, 1, S), tag
            if exp[0] == "thread":
                assert (p["kind"], p["lanes"], p["bps"], p["move"]) == (0, 1, 1, int(exp[1] == 8)), (tag, p)
                assert p["grid"] == grid(B, 1, S), tag
                assert p["ws"] == 8 * (67 if v.dcost > 0 else 55) * nt * 256 * p["grid"], (tag, p)
            else:
                assert (p["kind"], p["lanes"], p["bps"], p["move"]) == (1,) + exp[1:], (tag, p, exp)
                assert p["grid"] == grid(B, exp[1], S * exp[2]), (tag, p)
                assert p["ws"] == 8 * coop_doubles * p["grid"] * (256 // exp[1]), (tag, p)
            warm = not (v.model == "circular" and v.dcost > 0) and B >= 512
            assert p["warm"] == warm, (tag, p)
            assert p["alloc"] == (max(p["ws"], ref_ws) if warm else p["ws"]), (tag, p)
        # NODES = 3..6: the collocation kernel, whatever the kernel options say; no move term, no warm start
        for nodes in (3, 4, 5, 6):
            colloc_doubles = plan(S, 1, V("", 1), nodes)["ws"] // (8 * 8)
            for kernel, lanes in (("auto", 0), ("thread", 0), ("coop", 8)):
                for B in edges:
                    p = plan(S, B, V("", None, kernel=kernel, coop_lanes=lanes), nodes, warm_start=2)
                    gp = 32 if B <= 8 * S else 8
                    assert (p["kind"], p["lanes"], p["bps"], p["move"], p["use_dc"], p["warm"]) == (2, gp, 1, 0, 0, 0), (S, B, p)
                    assert p["grid"] == grid(B, gp, S) and p["slots"] == 256 * grid(B, 1, S), (S, B, p)
                    assert p["ws"] == p["alloc"] == 8 * colloc_doubles * p["grid"] * (256 // gp), (S, B, p)
    # the warm start: warm_start 0 / 1 / 2 around 512 problems, a caller's start point, the circular model with its
    # move term, and a 300-problem shard of a 1 024-problem batch
    S, v = 148, V("", None)
    for B in (511, 512):
        assert [plan(S, B, v, warm_start=w)["warm"] for w in (0, 1, 2)] == [0, int(B >= 512), 1], B
        assert plan(S, B, v, warm_start=2, guess=True)["warm"] == 0
        assert plan(S, B, V("", None, "circular"), warm_start=2)["warm"] == 0
        assert plan(S, B, V("", None, "circular", 0.0), warm_start=2)["warm"] == 1
    assert plan(S, 300, v, warm_batch=1024)["warm"] == 1 and plan(S, 300, v, warm_batch=511)["warm"] == 0
    assert plan(S, 300, v, warm_start=0, warm_batch=1024)["warm"] == 0
    p = plan(S, 1, v, warm_start=2)                   # one warp of one CTA, as the reference solve
    assert p["warm"] == 1 and p["alloc"] == p["ws"] == ref_ws, p
