"""The golden solutions that the flight tests fly (tests/test_fly_on_host.py, tests/test_gpu_fly.py), and the host build of
csrc/ascent_fly.cuh (tools/hostsim, ``hostsim_fly``) that both compare against."""
import ctypes as C
import dataclasses
import os
import shutil
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
VAR_ROWS = ["y", "ydot", "ydoubledot", "x", "xdot", "xdoubledot", "angle", "angledot", "mass", "angledoubledot"]
NOMINAL = np.array([6.674e-11, 7.346e22, 1738100.0, 15346.0, 4821.0, 5.053, 2376.0, 5e-4, 17703.0, 88615.0, 470.0,
                    2376.0, np.pi / 3, 1.0])
CIRCULAR = NOMINAL.copy()
CIRCULAR[8] = CIRCULAR[9] = 53108.4          # circular radii (PDF p.26 src 32-46)
CIRCULAR[11] = 2576.0                         # mass_scalar (PDF p.27 src 67)


@dataclasses.dataclass
class Case:
    name: str
    raw: np.ndarray        # [NPARAM] parameter column
    model: int             # lmato_model_t
    traj: np.ndarray       # [NVAR, nt] in the solve's output layout
    time: np.ndarray       # [nt]
    tf: float
    nodes: int


def _full(traj, names):
    names = list(names)
    out = np.zeros((len(VAR_ROWS), traj.shape[1]))
    for i, n in enumerate(VAR_ROWS):
        if n in names:
            out[i] = traj[names.index(n)]
    return out


def cases():
    """The fixtures of the flight table in DESIGN.md section 7."""
    out = []
    for name in ("elliptical_nominal_nt40", "elliptical_nominal_nt200", "elliptical_nominal_nonuniform60"):
        g = np.load(os.path.join(GOLDEN, name + ".npz"))
        out.append(Case(name, NOMINAL, 0, _full(g["traj"], g["names"]), g["time"], float(g["tf"]), 2))
    g = np.load(os.path.join(GOLDEN, "elliptical_higher_order_nodes3to6.npz"))
    for n in (3, 4, 5, 6):
        nt = int(g[f"nt_n{n}"])
        out.append(Case(f"nodes{n}_nt{nt}", NOMINAL, 0, _full(g[f"traj_n{n}"], g["names"]), np.linspace(0.0, 1.0, nt),
                        float(g[f"tf_n{n}"]), n))
    g = np.load(os.path.join(GOLDEN, "circular_nominal_nt200.npz"))
    out.append(Case("circular_nominal_nt200", CIRCULAR, 1, _full(g["traj"], g["names"]), g["time"], float(g["tf"]), 2))
    return out


def oracle_params(case):
    from oracle.ascent_nlp import AscentParams
    return AscentParams.circular() if case.model == 1 else AscentParams()


def build_hostsim(tmpdir):
    """g++ build of tools/hostsim (None without g++)."""
    if shutil.which("g++") is None:
        return None
    so = os.path.join(str(tmpdir), "libhostsim.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-I",
                           os.path.join(ROOT, "lunar_module_ascent_trajectory_optimiser_b200", "csrc"),
                           os.path.join(ROOT, "tools", "hostsim", "hostsim.cpp"), "-o", so])
    L = C.CDLL(so)
    L.hostsim_fly.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p,
                              C.c_void_p]
    L.hostsim_fly.restype = None
    return L


def host_fly(L, case, substeps):
    """(fin [NFLY], flown trajectory [NVAR, nt]) of ``case`` from the host build."""
    nt = case.traj.shape[1]
    fin, out = np.zeros(10), np.zeros((len(VAR_ROWS), nt))
    raw = np.ascontiguousarray(case.raw, dtype=np.float64)
    time = np.ascontiguousarray(case.time, dtype=np.float64)
    traj = np.ascontiguousarray(case.traj, dtype=np.float64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    L.hostsim_fly(p(raw), case.model, nt, p(time), p(traj), case.tf, substeps, p(fin), p(out))
    return fin, out
