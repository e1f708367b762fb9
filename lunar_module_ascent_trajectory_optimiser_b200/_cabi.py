"""ctypes binding of the C ABI declared in ``include/lmato_b200.h``.

There is deliberately no fallback of any kind here: if the CUDA shared library has not
been built (``python -c "import __graft_entry__ as g; g.build()"``) or no GPU is present,
the product raises.  The CPU oracle under ``oracle/`` is never imported from this package.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import sys
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblmato_b200.so")
CSRC = os.path.join(_HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(_HERE), "include")

NPARAM = 14
NVAR = 10
NSENS = 4
NFLY = 10
FLY_ROWS = ["y", "ydot", "x", "xdot", "angle", "angledot", "mass", "radius_miss_m", "speed_miss_mps",
            "flight_path_angle_rad"]                             # rows of lmato_fly_control's out_final
SENS_ROWS = ["Ft", "M0", "M_dot", "angle_doubledot_max"]      # lmato_sens_t
PARAM_ROWS = ["G", "M", "R0", "Ft", "M0", "M_dot", "fuel_mass", "angle_doubledot_max",
              "r_periapsis", "r_apoapsis", "final_time", "mass_scalar", "angle_ub", "u_bound"]
VAR_ROWS = ["y", "ydot", "ydoubledot", "x", "xdot", "xdoubledot", "angle", "angledot", "mass",
            "angledoubledot"]
STATUS_NAMES = {0: "converged", 1: "max_iter", 2: "linesearch_fail", 3: "inertia_fail", 4: "numerical",
                5: "stalled"}

KERNEL_IDS = {"auto": 0, "thread": 1, "coop": 2}     # lmato_kernel_t

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


class LmatoOptions(C.Structure):
    _fields_ = [("tol", C.c_double), ("mu_init", C.c_double), ("obj_scale", C.c_double),
                ("tf_guess", C.c_double), ("delta_c", C.c_double), ("mu_min_factor", C.c_double),
                ("max_iter", C.c_int32), ("max_ls", C.c_int32), ("n_polish", C.c_int32),
                ("warm_start", C.c_int32), ("mu_ref", C.c_double), ("dcost", C.c_double),
                ("kappa_eps", C.c_double), ("objective_nodes", C.c_int32), ("kernel", C.c_int32),
                ("coop_lanes", C.c_int32), ("reserved_", C.c_int32), ("otol", C.c_double), ("rtol", C.c_double)]


class LmatoError(RuntimeError):
    pass


LAST_BUILD = {"action": None, "seconds": 0.0}     # what the last build_library() call did: "compiled" | "reused"


def cuda_tool(name: str) -> str:
    """Path of a CUDA toolkit program (``nvcc``, ``cuobjdump``): from PATH, else from ``$CUDA_HOME/bin``,
    ``$CUDA_PATH/bin`` or ``/usr/local/cuda/bin``, so that a shell whose PATH lacks the toolkit still builds."""
    found = shutil.which(name)
    if found:
        return found
    for root in (os.environ.get("CUDA_HOME"), os.environ.get("CUDA_PATH"), "/usr/local/cuda"):
        if root and os.access(os.path.join(root, "bin", name), os.X_OK):
            return os.path.join(root, "bin", name)
    raise LmatoError(f"{name} not found on PATH, in $CUDA_HOME/bin, $CUDA_PATH/bin or /usr/local/cuda/bin")


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/ascent_cabi.cu for sm_100a into the in-tree shared library (or reuse it if it is newer than
    every source; ``LAST_BUILD`` says which)."""
    import time as _time
    srcs = [os.path.join(CSRC, f) for f in ("ascent_cabi.cu", "ascent_ipm.cuh", "ascent_ipm_dc.cuh", "ascent_coop.cuh", "ascent_colloc.cuh",
                                            "ascent_fly.cuh", "ascent_model.cuh", "ascent_result.cuh", "ascent_plan.h")]
    srcs.append(os.path.join(INCLUDE, "lmato_b200.h"))
    if not force and os.path.exists(LIB_PATH):
        if all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(s) for s in srcs):
            LAST_BUILD.update(action="reused", seconds=0.0)
            return LIB_PATH
    cmd = [cuda_tool("nvcc")] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", LIB_PATH, os.path.join(CSRC, "ascent_cabi.cu")]
    t0 = _time.time()
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise LmatoError("nvcc failed:\n" + r.stdout + r.stderr)
    LAST_BUILD.update(action="compiled", seconds=_time.time() - t0)
    if verbose:
        sys.stderr.write(r.stderr)
    return LIB_PATH


_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    """Load the CUDA library; raise loudly if it is missing (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LmatoError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built. "
            "Run `python -c 'import __graft_entry__ as g; g.build()'`. There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, dp, ip = C.c_void_p, C.c_int32, C.c_int64, C.POINTER(C.c_double), C.c_void_p
    L.lmato_last_error.restype = C.c_char_p
    L.lmato_version.restype = C.c_char_p
    L.lmato_default_options.argtypes = [C.POINTER(LmatoOptions)]
    L.lmato_default_options.restype = None
    L.lmato_create.argtypes = [C.POINTER(vp), i32, i32, vp, i32, i32]
    L.lmato_destroy.argtypes = [vp]
    L.lmato_set_options.argtypes = [vp, C.POINTER(LmatoOptions)]
    L.lmato_solve_batch.argtypes = [vp, vp, i64, vp, vp, vp, vp, vp, vp, vp]
    L.lmato_solve_batch_host.argtypes = [vp, vp, i64, vp, vp, vp, vp, vp, vp]
    L.lmato_workspace_bytes.argtypes = [vp, i64, C.POINTER(i64)]
    L.lmato_kernel_launches.argtypes = [vp, C.POINTER(i64)]
    L.lmato_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_double)]
    L.lmato_measure_fp64_peak.argtypes = [vp, C.POINTER(C.c_double)]
    L.lmato_selftest_math.argtypes = [vp, C.POINTER(C.c_double)]
    L.lmato_coast_orbit.argtypes = [vp, vp, i64, C.c_double, C.c_double, i64, vp, vp]
    L.lmato_fly_control.argtypes = [vp, vp, i64, vp, vp, i32, vp, vp, vp]
    L.lmato_set_sensitivity_output.argtypes = [vp, vp]
    L.lmato_set_param_sensitivity_output.argtypes = [vp, vp]
    L.lmato_set_initial_guess.argtypes = [vp, vp, vp]
    L.lmato_collocation_rule.argtypes = [i32, vp, vp]
    L.lmato_multi_create.argtypes = [C.POINTER(vp), C.POINTER(i32), i32, i32, vp, i32, i32]
    L.lmato_multi_destroy.argtypes = [vp]
    L.lmato_multi_set_options.argtypes = [vp, C.POINTER(LmatoOptions)]
    L.lmato_multi_device_count.argtypes = [vp, C.POINTER(i32)]
    L.lmato_multi_solve_host.argtypes = [vp, vp, i64, vp, vp, vp, vp, vp, vp]
    for name in ("lmato_create", "lmato_destroy", "lmato_set_options", "lmato_solve_batch",
                 "lmato_solve_batch_host", "lmato_workspace_bytes", "lmato_kernel_launches",
                 "lmato_last_kernel_ms", "lmato_measure_fp64_peak", "lmato_selftest_math", "lmato_coast_orbit",
                 "lmato_fly_control", "lmato_set_sensitivity_output", "lmato_set_param_sensitivity_output",
                 "lmato_set_initial_guess", "lmato_multi_create", "lmato_multi_destroy",
                 "lmato_multi_set_options", "lmato_multi_device_count", "lmato_multi_solve_host", "lmato_collocation_rule"):
        getattr(L, name).restype = C.c_int
    _lib = L
    return L


EXPORTED_SYMBOLS = ["lmato_default_options", "lmato_create", "lmato_destroy", "lmato_set_options",
                    "lmato_solve_batch", "lmato_solve_batch_host", "lmato_workspace_bytes",
                    "lmato_kernel_launches", "lmato_last_kernel_ms", "lmato_measure_fp64_peak",
                    "lmato_selftest_math", "lmato_coast_orbit", "lmato_fly_control", "lmato_set_sensitivity_output",
                    "lmato_set_param_sensitivity_output",
                    "lmato_set_initial_guess", "lmato_last_error",
                    "lmato_version", "lmato_multi_create", "lmato_multi_destroy", "lmato_multi_set_options",
                    "lmato_multi_device_count", "lmato_multi_solve_host", "lmato_collocation_rule"]


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().lmato_last_error().decode("utf-8", "replace")
        raise LmatoError(f"{what} failed (code {rc}): {msg}")
