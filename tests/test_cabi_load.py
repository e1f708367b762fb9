"""The C-ABI library builds for sm_100a, loads without a GPU, exports every symbol that
include/lmato_b200.h declares, and refuses to compute without a device (no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "lmato_b200.h")


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(lmato_[a-z0-9_]+)\s*\(", src)))


def test_header_functions_are_exported(built_lib):
    from lunar_module_ascent_trajectory_optimiser_b200 import _cabi
    fns = declared_functions()
    assert len(fns) >= 10
    L = C.CDLL(built_lib)
    for f in fns:
        assert hasattr(L, f), f
    assert sorted(_cabi.EXPORTED_SYMBOLS) == fns


def test_library_is_sm100a_and_has_no_torch_types(built_lib):
    from lunar_module_ascent_trajectory_optimiser_b200 import _cabi
    out = subprocess.run([_cabi.cuda_tool("cuobjdump"), "-lelf", built_lib], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out
    nm = subprocess.run(["nm", "-D", "--defined-only", built_lib], capture_output=True, text=True).stdout
    exported = [l.split()[-1] for l in nm.splitlines() if " T " in l]
    assert all(not s.startswith("_ZN2at") and "torch" not in s for s in exported)


def test_default_options_and_enums(built_lib):
    from lunar_module_ascent_trajectory_optimiser_b200 import _cabi
    L = _cabi.lib()
    o = _cabi.LmatoOptions()
    L.lmato_default_options(C.byref(o))
    assert o.tol == 1e-10 and o.mu_init == 0.1 and o.max_iter == 20000 and o.obj_scale == 10.0   # LO:28
    assert o.mu_min_factor == 1e-3 and o.n_polish == -1 and o.warm_start == 1 and o.mu_ref == 1e-3
    assert o.dcost == 1e-5 and o.objective_nodes == 0 and o.kappa_eps == 30.0                                             # LO:99
    src = open(HEADER).read()
    assert int(re.search(r"LMATO_NPARAM = (\d+)", src).group(1)) == _cabi.NPARAM == len(_cabi.PARAM_ROWS)
    assert int(re.search(r"LMATO_NVAR = (\d+)", src).group(1)) == _cabi.NVAR == len(_cabi.VAR_ROWS)
    assert L.lmato_version().decode().startswith("lmato_b200")


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_device_fails_loudly(built_lib):
    from lunar_module_ascent_trajectory_optimiser_b200 import _cabi
    import lunar_module_ascent_trajectory_optimiser_b200 as lm
    L = _cabi.lib()
    h = C.c_void_p()
    rc = L.lmato_create(C.byref(h), 0, 200, None, 2, 0)
    assert rc == 3 and not h.value                      # LMATO_ERR_NO_DEVICE
    assert b"no CPU fallback" in L.lmato_last_error()
    with pytest.raises(lm.LmatoError):
        lm.optimise()
    with pytest.raises(lm.LmatoError):
        lm.optimise_batch(lm.dispersed_params(4))


def test_argument_validation_without_gpu(built_lib):
    from lunar_module_ascent_trajectory_optimiser_b200 import _cabi
    L = _cabi.lib()
    h = C.c_void_p()
    assert L.lmato_create(None, 0, 200, None, 2, 0) == 1
    assert L.lmato_create(C.byref(h), 0, 1, None, 2, 0) == 1          # nt < 2
    assert L.lmato_create(C.byref(h), 0, 200, None, 7, 0) == 1        # NODES outside GEKKO's 2..6 (LO:25)
    assert L.lmato_create(C.byref(h), 0, 200, None, 3, 1) == 4        # NODES >= 3 with the circular model: unsupported
    assert L.lmato_create(C.byref(h), 0, 200, None, 2, 7) == 1        # unknown model
    assert L.lmato_solve_batch(None, None, 1, None, None, None, None, None, None, None) == 1
    assert L.lmato_solve_batch_host(None, None, 1, None, None, None, None, None, None) == 1
    assert L.lmato_multi_solve_host(None, None, 1, None, None, None, None, None, None) == 1
    assert b"lmato_multi_solve_host: NULL handle" in L.lmato_last_error()
    assert L.lmato_destroy(None) == 0
    if not torch.cuda.is_available():
        m = C.c_void_p()
        assert L.lmato_multi_create(C.byref(m), (C.c_int32 * 1)(0), 1, 200, None, 2, 0) == 3 and not m.value   # LMATO_ERR_NO_DEVICE


def test_product_does_not_import_oracle():
    """The product package must never route through the CPU oracle."""
    pkg = os.path.join(ROOT, "lunar_module_ascent_trajectory_optimiser_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                s = open(os.path.join(dp, f)).read()
                assert "import oracle" not in s and "from oracle" not in s, f
