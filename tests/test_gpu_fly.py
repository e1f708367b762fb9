"""The post-solve flight on the device (``lmato_fly_control``, ``lm.fly``): against its host build, batched against
single flights, on fresh GPU solutions against the oracle's findings, chained into the orbit coast, and its argument
checks."""
import ctypes as C

import numpy as np
import pytest
import torch

from fly_cases import VAR_ROWS, build_hostsim, cases, host_fly, oracle_params
from oracle.fly_reference import fly_fixture

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lm():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import lunar_module_ascent_trajectory_optimiser_b200 as lm
    lm.build_library()
    return lm


def _solver(lm, case):
    return lm.AscentSolver(lm.Mesh(time=list(case.time)), device=0, model="circular" if case.model else "elliptical")


def test_device_flight_matches_host_build(lm, tmp_path):
    """Device (fdlibm kernels, MUFU + Newton) against host (libm) on every golden solution, states and misses."""
    L = build_hostsim(tmp_path)
    if L is None:
        pytest.skip("g++ not available")
    worst = 0.0
    for c in cases():
        s = _solver(lm, c)
        n = lm.default_fly_substeps(torch.as_tensor(c.time))
        dev = torch.device("cuda", 0)
        out = s.fly_control(torch.as_tensor(c.raw, device=dev).reshape(-1, 1), torch.as_tensor(c.traj, device=dev)[:, :, None],
                            torch.tensor([c.tf], dtype=torch.float64, device=dev), n)
        fin_d, traj_d = out["final"][:, 0].cpu().numpy(), out["traj"][:, :, 0].cpu().numpy()
        fin_h, traj_h = host_fly(L, c, n)
        rel = (np.abs(traj_d - traj_h).max(axis=1) / (np.abs(traj_h).max(axis=1) + 1e-300)).max()
        rel_fin = (np.abs(fin_d[:7] - fin_h[:7]) / np.maximum(np.abs(fin_h[:7]), 1e-300)).max()
        miss = np.abs(fin_d[7:9] - fin_h[7:9]).max()
        print(f"\n[device vs host] {c.name}: states {rel:.2e}, end state {rel_fin:.2e}, misses {miss:.2e} m | m/s")
        worst = max(worst, rel)
        # measured on a B200: states 9.0e-16, end state 2.5e-15 of each row's range, misses 5e-10 m
        assert rel < 1e-14 and rel_fin < 2e-14 and miss < 1e-8, (c.name, rel, rel_fin, miss)
        s.close()
    print(f"\n[device vs host] worst {worst:.2e}")


def test_batched_flight_equals_single_flights_and_placements(lm):
    """4 096 dispersions solved and flown as one batch: every column is bitwise the flight of that problem alone, and a
    CPU solution flies to the same numbers as its CUDA original."""
    p = lm.dispersed_params(4096, seed=11)
    pd = lm.AscentParams(**{f: (v.cuda() if isinstance(v, torch.Tensor) else v) for f, v in vars(p).items()})
    sol = lm.optimise_batch(pd, lm.Mesh(nt=200), device=0)
    print(f"\n[dispersions] {int((sol.status == 0).sum())} of 4096 converged (the others are flown as given)")
    flown = lm.fly(sol, pd)
    solver = lm.api._get_solver(lm.Mesh(time=sol.time.tolist()), lm.SolverOptions(), 0, "elliptical")
    rows = pd.rows(4096, device="cuda:0")
    traj = torch.stack([sol.control.transpose(0, 1) if n == "angledoubledot" else sol.states[n].transpose(0, 1)
                        for n in lm._cabi.VAR_ROWS])
    batch = solver.fly_control(rows, traj, sol.tf, flown.substeps)
    fin = torch.stack([flown.final_state[n] for n in lm._cabi.FLY_ROWS[:7]] +
                      [flown.radius_miss_m, flown.speed_miss_mps, flown.flight_path_angle_rad])
    assert torch.equal(batch["final"], fin)
    for b in range(4096):
        one = solver.fly_control(rows[:, b:b + 1].contiguous(), traj[:, :, b:b + 1].contiguous(), sol.tf[b:b + 1], flown.substeps)
        assert torch.equal(one["final"][:, 0], batch["final"][:, b]), b
        assert torch.equal(one["traj"][:, :, 0], batch["traj"][:, :, b]), b
    host = lm.AscentBatchSolution(**{k: (v.cpu() if isinstance(v, torch.Tensor) else
                                         ({n: t.cpu() for n, t in v.items()} if isinstance(v, dict) else v))
                                     for k, v in vars(sol).items()})
    fh = lm.fly(host, p)
    assert not fh.radius_miss_m.is_cuda and not fh.states["y"].is_cuda
    assert torch.equal(fh.radius_miss_m, flown.radius_miss_m.cpu()) and torch.equal(fh.states["x"], flown.states["x"].cpu())
    assert torch.equal(fh.final_state_si(), flown.final_state_si().cpu())
    m = flown.radius_miss_m
    print(f"\n[dispersions] radius miss {float(m.min()):+.1f} .. {float(m.max()):+.1f} m, speed miss "
          f"{float(flown.speed_miss_mps.min()):+.2f} .. {float(flown.speed_miss_mps.max()):+.2f} m/s")
    assert float((3 * flown.states["angle"]).abs().max()) < 3.5


def test_gpu_solutions_reproduce_the_oracle_findings(lm):
    """Fresh GPU solutions flown: NODES = 2 misses by kilometres as the oracle says, NODES = 4 by metres; the circular
    model flies with its pitch angle held."""
    ref = {c.name: fly_fixture(c.traj, VAR_ROWS, c.time, c.tf, oracle_params(c)) for c in cases()}
    p = lm.AscentParams(dcost=0.0)
    for nt, name in ((40, "elliptical_nominal_nt40"), (200, "elliptical_nominal_nt200")):
        f = lm.fly(lm.optimise(p, lm.Mesh(nt=nt), device=0), p)
        for key, got in (("radius_miss_m", f.radius_miss_m), ("speed_miss_mps", f.speed_miss_mps)):
            assert abs(float(got[0]) / ref[name][key] - 1) < 5e-3, (nt, key, float(got[0]), ref[name][key])
        print(f"\n[nodes 2, nt {nt}] radius miss {float(f.radius_miss_m[0]):+.2f} m, speed miss {float(f.speed_miss_mps[0]):+.3f} m/s")
    f = lm.fly(lm.optimise(p, lm.Mesh(nt=30, nodes=4), device=0), p)
    print(f"\n[nodes 4, nt 30] radius miss {float(f.radius_miss_m[0]):+.3f} m")
    assert abs(float(f.radius_miss_m[0])) < 10
    pc = lm.AscentParams.circular()
    pc.dcost = 0.0
    sol = lm.optimise(pc, lm.Mesh(nt=200), device=0)
    f = lm.fly(sol, pc)
    assert set(f.states) == set(sol.states) and "angle" not in f.states
    assert float(f.final_state["angle"][0]) == float(sol.control[-1]) and float(f.final_state["angledot"][0]) == 0.0
    r = ref["circular_nominal_nt200"]
    assert abs(float(f.radius_miss_m[0]) / r["radius_miss_m"] - 1) < 1e-2
    assert abs(float(f.speed_miss_mps[0]) / r["speed_miss_mps"] - 1) < 1e-2


def test_flown_insertion_state_coasts(lm):
    """coast_orbit starts from the flown insertion state; its perilune differs from the coast of the discrete end state."""
    p = lm.AscentParams()
    sol = lm.optimise_batch(p, lm.Mesh(nt=200), device=0, batch=1)
    solver = lm.api._get_solver(lm.Mesh(nt=200), lm.SolverOptions(), 0, "elliptical")
    flown = lm.fly(sol, p)
    a = solver.coast_orbit(flown.final_state_si().cuda(), t_coast=6600.0, dt=1e-2)
    b = solver.coast_orbit(lm.final_state_si(sol, p).cuda(), t_coast=6600.0, dt=1e-2)
    ra, rb = float(a["r_min"][0]), float(b["r_min"][0])
    print(f"\n[coast] r_min flown {ra:.1f} m, discrete {rb:.1f} m, difference {ra - rb:+.1f} m")
    assert np.isfinite(ra) and ra != rb


def test_argument_errors(lm):
    s = lm.AscentSolver(lm.Mesh(nt=40), device=0)
    L = lm._cabi.lib()
    dev = torch.device("cuda", 0)
    rows = lm.AscentParams().rows(2, device=dev)
    traj = torch.zeros((10, 40, 2), dtype=torch.float64, device=dev)
    tf = torch.full((2,), 0.9, dtype=torch.float64, device=dev)
    fin = torch.empty((10, 2), dtype=torch.float64, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())
    call = lambda h, B, sub, r=rows, t=traj, f=tf, o=fin: lm._cabi.check(
        L.lmato_fly_control(h, p(r) if r is not None else None, B, p(t) if t is not None else None,
                            p(f) if f is not None else None, sub, p(o) if o is not None else None, None, None), "fly")
    with pytest.raises(lm.LmatoError):
        call(None, 2, 4)                                   # NULL handle
    for kw in (dict(r=None), dict(t=None), dict(f=None), dict(o=None)):
        with pytest.raises(lm.LmatoError):
            call(s._h, 2, 4, **kw)                         # NULL buffer
    with pytest.raises(lm.LmatoError):
        call(s._h, -1, 4)                                  # B < 0
    for sub in (0, -3):
        with pytest.raises(lm.LmatoError):
            call(s._h, 2, sub)                             # substeps < 1
    call(s._h, 0, 4)                                       # B = 0: nothing to do
    call(s._h, 2, 4)
    torch.cuda.synchronize()
    with pytest.raises(lm.LmatoError):
        s.fly_control(rows, traj, tf, 0)
    s.close()
