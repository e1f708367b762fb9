"""The host-buffer entry points stage a solve through device memory and must not change its answer: the host entry
(lmato_solve_batch_host) against the device entry (lmato_solve_batch) bit for bit, a handle's staging buffer as it
grows and shrinks, and the device list (lmato_multi_solve_host) shard by shard against host solves of the shards.
Every comparison uses fresh handles: a handle's warm-start reference carries over from one call to the next."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

NT = 200
KEYS = ("traj", "tf", "final_mass", "status", "iterations", "kkt")


@pytest.fixture(scope="module")
def lm(built_lib):
    import lunar_module_ascent_trajectory_optimiser_b200 as lm
    assert torch.cuda.is_available()
    return lm


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p()


def _rows(lm, B, seed, pinned=True):
    rows = lm.dispersed_params(B, seed=seed).rows(B)
    return rows.pin_memory() if pinned else rows


def _outputs(B, pinned, traj=True, kkt=True):
    """Host result arrays filled with NaN / -1, so that an entry the solve does not write shows."""
    f = lambda shape: torch.full(shape, float("nan"), dtype=torch.float64, pin_memory=pinned)
    i = lambda: torch.full((B,), -1, dtype=torch.int32, pin_memory=pinned)
    return {"traj": f((10, NT, B)) if traj else None, "tf": f((B,)), "final_mass": f((B,)), "status": i(),
            "iterations": i(), "kkt": f((B,)) if kkt else None}


def _device(lm, rows, trajectories=True, sensitivities=False, guess=None):
    s = lm.AscentSolver(lm.Mesh(nt=NT), device=0)
    g = None if guess is None else {k: v.cuda() for k, v in guess.items()}
    r = s.solve_rows(rows.cuda(), trajectories, sensitivities=sensitivities, guess=g)
    torch.cuda.synchronize()
    out = {k: (v.cpu() if v is not None else None) for k, v in r.items()}
    s.close()
    return out


def _host(lm, rows, out=None, trajectories=True, sensitivities=False, guess=None, **opt):
    s = lm.AscentSolver(lm.Mesh(nt=NT), lm.SolverOptions(**opt), device=0)
    r = s.solve_rows(rows, trajectories, out=out, sensitivities=sensitivities, guess=guess)
    s.close()
    return r


def _assert_equal(got, want, keys):
    for k in keys:
        if want[k] is None or got[k] is None:
            assert want[k] is None and got[k] is None, k
        else:
            assert not got[k].is_cuda and torch.equal(got[k], want[k]), k


@pytest.mark.parametrize("B", [300, 700])            # cold start, batch warm start
@pytest.mark.parametrize("pinned", [True, False])    # direct write of the trajectories, staged copies
@pytest.mark.parametrize("trajectories", [True, False])
def test_host_entry_equals_device_entry(lm, B, pinned, trajectories):
    rows = _rows(lm, B, seed=B, pinned=pinned)
    want = _device(lm, rows, trajectories)
    got = _host(lm, rows, out=_outputs(B, pinned, trajectories), trajectories=trajectories)
    _assert_equal(got, want, KEYS)
    assert int((got["status"] != 0).sum()) == 0


def _host_abi(lm, rows, out):
    """lmato_solve_batch_host on a fresh handle, straight through ctypes: every array of `out` as given (None = NULL),
    `out["dtf"]` registered as the sensitivity output when present."""
    from lunar_module_ascent_trajectory_optimiser_b200 import _cabi
    L = _cabi.lib()
    s = lm.AscentSolver(lm.Mesh(nt=NT), device=0)
    if out.get("dtf") is not None:
        _cabi.check(L.lmato_set_sensitivity_output(s._h, _ptr(out["dtf"])), "lmato_set_sensitivity_output")
    _cabi.check(L.lmato_solve_batch_host(s._h, _ptr(rows), rows.shape[1], _ptr(out["traj"]), _ptr(out["tf"]),
                                         _ptr(out["final_mass"]), _ptr(out["status"]), _ptr(out["iterations"]),
                                         _ptr(out["kkt"])), "lmato_solve_batch_host")
    s.close()


@pytest.mark.parametrize("B", [300, 700])
def test_host_entry_without_kkt_output(lm, B):
    rows = _rows(lm, B, seed=B + 1)
    want = _device(lm, rows)
    out = _outputs(B, True, kkt=False)
    _host_abi(lm, rows, out)
    _assert_equal(out, dict(want, kkt=None), KEYS)


@pytest.mark.parametrize("B", [300, 700])
@pytest.mark.parametrize("pinned", [True, False])    # the sensitivity output itself pinned or pageable
def test_host_entry_sensitivities(lm, B, pinned):
    rows = _rows(lm, B, seed=B + 2, pinned=pinned)
    want = _device(lm, rows, sensitivities=True)
    out = dict(_outputs(B, pinned), dtf=torch.full((4, B), float("nan"), dtype=torch.float64, pin_memory=pinned))
    _host_abi(lm, rows, out)
    _assert_equal(out, want, KEYS + ("dtf",))


@pytest.mark.parametrize("B", [300, 700])
def test_host_entry_with_a_start_point(lm, B):
    rows = _rows(lm, B, seed=B + 3)
    start = _device(lm, rows)
    near = rows.clone()
    near[3] *= 1.005                                   # Ft + 0.5 %
    near = near.pin_memory()
    guess = {"traj": start["traj"].pin_memory(), "tf": start["tf"].pin_memory()}
    want = _device(lm, near, guess=guess)
    got = _host(lm, near, guess=guess)
    _assert_equal(got, want, KEYS)
    assert int((got["status"] != 0).sum()) == 0


@pytest.mark.parametrize("pinned", [True, False])
def test_staging_buffer_grows_and_shrinks(lm, pinned):
    """One handle solves 300, then 1 300, then 300 problems: each call equals the same call on a fresh handle."""
    s = lm.AscentSolver(lm.Mesh(nt=NT), device=0)
    for B, seed in ((300, 51), (1300, 52), (300, 53)):
        rows = _rows(lm, B, seed, pinned)
        got = s.solve_rows(rows, out=_outputs(B, pinned), sensitivities=True)
        _assert_equal(got, _host(lm, rows, out=_outputs(B, pinned), sensitivities=True), KEYS + ("dtf",))
    s.close()


def _device_lists():
    return [[0], [0, 0], [0, 0, 0]] + ([[0, 1]] if torch.cuda.device_count() >= 2 else [])


@pytest.mark.parametrize("B", [2, 333, 1300])       # fewer problems than devices; cold shards; warm shards
def test_device_list_equals_host_solves_of_its_shards(lm, B):
    from lunar_module_ascent_trajectory_optimiser_b200 import _cabi
    L = _cabi.lib()
    rows = _rows(lm, B, seed=B + 4)
    want = {}
    for devices in _device_lists():
        G = len(devices)
        if G not in want:
            # the device list keeps the batch warm start of the whole batch in every shard
            parts = [_host(lm, rows[:, lo:hi].contiguous(), warm_start=2 if B >= 512 else 1)
                     for lo, hi in (lm.shard_bounds(B, G, g) for g in range(G)) if hi > lo]
            want[G] = {k: torch.cat([p[k] for p in parts], dim=-1) for k in KEYS}
        for pinned in (True, False):
            for full in (True, False):                 # out_traj and out_kkt given, or both NULL
                out = _outputs(B, pinned, traj=full, kkt=full)
                ms = lm.AscentMultiSolver(devices, lm.Mesh(nt=NT))
                _cabi.check(L.lmato_multi_solve_host(ms._h, _ptr(rows), B, _ptr(out["traj"]), _ptr(out["tf"]),
                                                     _ptr(out["final_mass"]), _ptr(out["status"]),
                                                     _ptr(out["iterations"]), _ptr(out["kkt"])), "lmato_multi_solve_host")
                ms.close()
                _assert_equal(out, want[G] if full else dict(want[G], traj=None, kkt=None), KEYS)
        assert int((want[G]["status"] != 0).sum()) == 0
