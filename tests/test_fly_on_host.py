"""The post-solve flight (csrc/ascent_fly.cuh) compiled for the host (tools/hostsim, ``hostsim_fly``) against the oracle's
DOP853 integration (oracle/fly_reference.py), on the golden solutions of both transcriptions and both models.  No GPU."""
import math

import numpy as np
import pytest

import torch

from fly_cases import VAR_ROWS, build_hostsim, cases, host_fly, oracle_params
from oracle.fly_reference import STATES, fly_fixture
from lunar_module_ascent_trajectory_optimiser_b200.api import default_fly_substeps

ROWS = [0, 1, 3, 4, 6, 7, 8]          # y, ydot, x, xdot, angle, angledot, mass of the [NVAR, nt] layout


@pytest.fixture(scope="module")
def hostsim(tmp_path_factory):
    L = build_hostsim(tmp_path_factory.mktemp("hostsim_fly"))
    if L is None:
        pytest.skip("g++ not available")
    return L


@pytest.fixture(scope="module")
def oracle():
    return {c.name: fly_fixture(c.traj, VAR_ROWS, c.time, c.tf, oracle_params(c)) for c in cases()}


def _rel(out, ref):
    R = np.stack([ref[s] for s in STATES])
    return np.abs(out[ROWS] - R).max(axis=1) / (np.abs(R).max(axis=1) + 1e-300)


def _substeps(case):
    return default_fly_substeps(torch.as_tensor(case.time, dtype=torch.float64))


def test_host_flight_matches_oracle(hostsim, oracle):
    """Flown node states of every fixture, at the default sub-step count, against DOP853 (rtol 1e-13)."""
    for c in cases():
        fin, out = host_fly(hostsim, c, _substeps(c))
        err = _rel(out, oracle[c.name])
        print(f"\n[fly] {c.name}: substeps {_substeps(c)}, worst row error {err.max():.2e}, radius miss "
              f"{fin[7]:+.3f} m (oracle {oracle[c.name]['radius_miss_m']:+.3f}), speed miss {fin[8]:+.4f} m/s")
        assert err.max() < 5e-12, (c.name, err)             # measured: 3.7e-12 (nt = 200), <= 1.4e-12 elsewhere
        np.testing.assert_allclose(fin[:7], out[ROWS, -1], rtol=0, atol=0)
        assert abs(fin[7] - oracle[c.name]["radius_miss_m"]) < 1e-6 * max(1.0, abs(fin[7])), c.name
        assert abs(fin[8] - oracle[c.name]["speed_miss_mps"]) < 1e-7, c.name
        assert abs(fin[9] - oracle[c.name]["flight_path_angle_rad"]) < 1e-10, c.name
        # the acceleration rows are the model's at the flown nodes, the MV row is the input's
        assert np.array_equal(out[9 if c.model == 0 else 6], c.traj[9 if c.model == 0 else 6])
        if c.model == 1:
            assert not out[7].any() and not out[9].any()       # the circular model has no angledot / angledoubledot
        assert not out[:, 0].any()                              # node 0 pinned at zero, as the solve writes it


def test_oracle_pins_the_transcription_error(oracle):
    """The misses of DESIGN.md section 7: NODES = 2 flown misses insertion by kilometres, NODES >= 3 by metres."""
    o = oracle
    nom = o["elliptical_nominal_nt200"]
    assert abs(nom["radius_miss_m"] / 1976.0 - 1) < 5e-3 and abs(nom["speed_miss_mps"] / -10.58 - 1) < 5e-3
    assert abs(o["nodes6_nt20"]["radius_miss_m"]) < 1.0
    circ = o["circular_nominal_nt200"]
    assert abs(circ["radius_miss_m"] / -175.0 - 1) < 1e-2 and abs(circ["speed_miss_mps"] / -2.46 - 1) < 1e-2
    # first order in the step: nt 40 -> 200 shrinks the miss about 199/39 = 5.1 times
    ratio = o["elliptical_nominal_nt40"]["radius_miss_m"] / nom["radius_miss_m"]
    assert 4.5 < ratio < 5.7, ratio
    for n in (3, 4, 5, 6):
        r = [v for k, v in o.items() if k.startswith(f"nodes{n}_")][0]
        assert abs(r["radius_miss_m"]) < 100 and abs(r["speed_miss_mps"]) < 0.1, n


def test_rk4_order_and_exact_rows(hostsim, oracle):
    """Against the oracle the error falls by ~16 per halving of the sub-step (RK4); angle, angledot (polynomial in time
    under a held u) and mass (linear) are exact at any sub-step count."""
    for c in cases():
        errs = []
        for n in (4, 8, 16):
            _, out = host_fly(hostsim, c, n)
            e = _rel(out, oracle[c.name])
            assert e[4:].max() < 1e-13, (c.name, n, e)
            errs.append(e[:4].max())
        print(f"\n[order] {c.name}: errors at 4 / 8 / 16 sub-steps {errs[0]:.2e} {errs[1]:.2e} {errs[2]:.2e}")
        if c.model == 1:
            continue            # the circular flight is already at the rounding level at 8 sub-steps (1.4e-14)
        for a, b in zip(errs, errs[1:]):
            assert 12 < a / b < 20, (c.name, errs)


def test_default_substeps_converge(hostsim):
    """The default sub-step count: multiplied by 4 it moves the flown end state by < 1e-10 relative.  On the reference
    mesh (nt = 200) it is 16, and 8 would not do."""
    for c in cases():
        n = _substeps(c)
        a, _ = host_fly(hostsim, c, n)
        b, _ = host_fly(hostsim, c, 4 * n)
        change = (np.abs(b[:7] - a[:7]) / np.maximum(np.abs(a[:7]), 1e-300)).max()
        print(f"\n[substeps] {c.name}: {n} -> {4 * n} changes the end state by {change:.1e}")
        assert change < 1e-10, (c.name, n, change)
    c = [c for c in cases() if c.name == "elliptical_nominal_nt200"][0]
    assert _substeps(c) == 16
    a, _ = host_fly(hostsim, c, 8)
    b, _ = host_fly(hostsim, c, 32)
    assert (np.abs(b[:7] - a[:7]) / np.abs(a[:7])).max() > 1e-10


def test_pitch_angle_stays_in_the_fast_sincos_range(hostsim):
    """accel_value takes sin and cos of 3*angle from lm_sincos_small, documented for |3*angle| <= ~3.5.  Between nodes
    the flown angle is a quadratic in time under the held u; its largest value over every step of every fixture, with
    the RK4 stage predictors' departure from it (c*asc*|u|*h^2/8 per sub-step) added, stays inside that range."""
    worst = 0.0
    for c in cases():
        _, out = host_fly(hostsim, c, _substeps(c))
        a, ad = out[6], out[7]
        if c.model == 1:
            worst = max(worst, 3 * np.abs(a).max())
            continue
        p = oracle_params(c)
        cc = p.final_time * c.tf
        s = np.linspace(0.0, 1.0, 65)
        for k in range(1, len(c.time)):
            h = c.time[k] - c.time[k - 1]
            u = c.traj[9, k]
            t = s * h
            ang = a[k - 1] + cc * (ad[k - 1] * t + 0.5 * p.asc * u * t * t)
            margin = cc * p.asc * abs(u) * h * h / 8
            worst = max(worst, 3 * (np.abs(ang).max() + margin))
    print(f"\n[sincos] largest |3*angle| of any flight: {worst:.4f} (pi = {math.pi:.4f})")
    assert worst < 3.5
