"""Python API: ``optimise()`` / ``optimise_batch()``.

Drop-in for the model that ``Launch_Optimiser.py`` declares and solves (LO:19-202 of
/root/reference/Launch_Optimiser.py): the same physical parameters, mesh and options go
in; the same ``tf``, per-node state lists, control and final mass come out, in the same
scaled units the reference's ``.value`` lists use.

    reference                                   here
    ---------                                   ----
    G_py, M_py, R0_py            (LO:50-52)     AscentParams.G, .M, .R0
    Ft, M0, M_dot, fuel_mass     (LO:61-65)     AscentParams.Ft, .M0, .M_dot, .fuel_mass
    angle_doubledot_max          (LO:66)        AscentParams.angle_doubledot_max
    r_periapsis, r_apoapsis      (LO:70-71)     AscentParams.r_periapsis, .r_apoapsis
    final_time                   (LO:38)        AscentParams.final_time
    nt, m.time, m.options.NODES  (LO:20-25)     Mesh.nt, .time, .nodes
    m.options.MAX_ITER/OTOL/RTOL (LO:28-32)     SolverOptions.max_iter, .otol, .rtol
    m.solve()                    (LO:177)       optimise() / optimise_batch()
    tf.value[0]                  (LO:178)       solution.tf
    y.value, x.value, ...        (LO:188-202)   solution.states["y"], ...  ([B, nt])
    failure -> Exception         (LO:177)       optimise(): raises; optimise_batch(): status[b]
    (no counterpart)                            fly(): the solved control flown through LO:114-136

Host code is Python; all numerical work happens in hand-written sm_100a CUDA kernels
behind the C ABI of ``include/lmato_b200.h`` (ctypes).  PyTorch provides device memory,
streams and ``torch.distributed`` only.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import math
from typing import Callable, Dict, List, Optional, Sequence, Union

import torch

from . import _cabi

Scalar = Union[float, int, torch.Tensor]

G_ISP = 9.807   # reference PDF p.6:  M_dot = Ft / (Isp * 9.807)


@dataclasses.dataclass
class AscentParams:
    """Physical parameters, reference names and defaults.  Every field may be a python
    float (shared by the whole batch) or a float64 tensor of shape ``[B]``."""

    G: Scalar = 6.674e-11                 # LO:50
    M: Scalar = 7.346e22                  # LO:51
    R0: Scalar = 1738100.0                # LO:52
    Ft: Scalar = 15346.0                  # LO:61
    M0: Scalar = 4821.0                   # LO:62
    M_dot: Scalar = 5.053                 # LO:63 (the literal used in mflow, LO:65)
    fuel_mass: Scalar = 2376.0            # LO:64
    angle_doubledot_max: Scalar = 5e-4    # LO:66
    r_periapsis: Scalar = 17703.0         # LO:70
    r_apoapsis: Scalar = 88615.0          # LO:71
    final_time: Scalar = 470.0            # LO:38
    model: str = "elliptical"             # "elliptical" | "circular" (reference PDF p.26-28)
    Isp: Optional[Scalar] = None          # if given, M_dot = Ft/(Isp*9.807) (PDF p.6)
    mass_scalar: Optional[Scalar] = None  # LO:108 (= fuel_mass); 2576 in the PDF original
    angle_ub: Scalar = math.pi / 3        # LO:94
    u_bound: Scalar = 1.0                 # LO:96
    dcost: float = 1e-5                   # LO:99 angledoubledot.DCOST (0 = off)

    @staticmethod
    def circular() -> "AscentParams":
        """The 'original IB-document' model (reference PDF p.26 src 32-46, p.27 src 66-67)."""
        return AscentParams(r_periapsis=53108.4, r_apoapsis=53108.4, model="circular",
                            mass_scalar=2576.0)

    def batch_size(self) -> Optional[int]:
        B = None
        for f in dataclasses.fields(self):
            v = getattr(self, f.name)
            if isinstance(v, torch.Tensor) and v.dim() > 0:
                if v.dim() != 1:
                    raise ValueError(f"AscentParams.{f.name}: expected shape [B], got {tuple(v.shape)}")
                if B is not None and v.shape[0] != B:
                    raise ValueError(f"AscentParams.{f.name}: batch {v.shape[0]} != {B}")
                B = v.shape[0]
        return B

    def rows(self, B: Optional[int] = None, device: Union[str, torch.device] = "cpu") -> torch.Tensor:
        """Pack into the C ABI's ``[LMATO_NPARAM][B]`` struct-of-arrays block (float64)."""
        Bt = self.batch_size()
        if B is None:
            B = 1 if Bt is None else Bt
        elif Bt is not None and Bt != B:
            raise ValueError(f"batch size mismatch: tensors have {Bt}, requested {B}")
        vals = {}
        for name in _cabi.PARAM_ROWS:
            vals[name] = getattr(self, name)
        if self.Isp is not None:
            vals["M_dot"] = _t(self.Ft, device) / (_t(self.Isp, device) * G_ISP)
        if self.mass_scalar is None:
            vals["mass_scalar"] = self.fuel_mass
        out = torch.empty((_cabi.NPARAM, B), dtype=torch.float64, device=device)
        for i, name in enumerate(_cabi.PARAM_ROWS):
            out[i] = _t(vals[name], device)
        return out


def _t(v: Scalar, device) -> torch.Tensor:
    if isinstance(v, torch.Tensor):
        return v.to(device=device, dtype=torch.float64)
    return torch.tensor(float(v), dtype=torch.float64, device=device)


@dataclasses.dataclass
class Mesh:
    """LO:20-25: ``nt`` nodes on normalised time, GEKKO ``NODES`` per step."""
    nt: int = 200
    time: Optional[Sequence[float]] = None    # explicit m.time (overrides nt)
    nodes: int = 2

    def grid(self) -> torch.Tensor:
        if self.time is not None:
            t = torch.as_tensor(self.time, dtype=torch.float64).flatten().cpu()
            return t
        return torch.linspace(0.0, 1.0, self.nt, dtype=torch.float64)   # LO:21


@dataclasses.dataclass
class SolverOptions:
    """LO:26-33 plus solver-native knobs."""
    max_iter: int = 20000          # LO:28
    otol: float = 1e-3             # LO:31  } the solve runs to min(tol, otol, rtol): the reference's 1e-3 never loosens
    rtol: float = 1e-3             # LO:32  } the default tol, a tighter OTOL/RTOL tightens it (lmato_b200.h)
    tol: float = 1e-10             # scaled KKT error at which a problem counts as converged
    mu_init: float = 0.1
    obj_scale: float = 10.0
    tf_guess: float = 0.9
    delta_c: float = 1e-8
    max_ls: int = 40
    mu_min_factor: float = 1e-3    # barrier floor = mu_min_factor * tol
    n_polish: int = -1             # Newton iterations after tol is first met; -1 = 2 with DCOST, 4 without
    warm_start: int = 1            # 1: batches >= 512 start from the batch-mean problem's central path; 0: never; 2: always
    mu_ref: float = 1e-3           # barrier parameter at which that reference solve stops
    dcost: Optional[float] = None  # LO:99; None = take AscentParams.dcost (1e-5 in the reference)
    objective_nodes: int = 0       # APMonitor sums the objective over the horizon; 0 = nt-1
    kappa_eps: float = 30.0        # barrier sub-problem tolerance factor (IPOPT's default is 10)
    kernel: str = "auto"           # "auto" | "thread" (one problem per thread) | "coop" (eight lanes per problem)
    coop_lanes: int = 0            # coop kernel: lanes per problem in the stage-parallel phases (8 | 32; 0 = by batch size)


@dataclasses.dataclass
class AscentBatchSolution:
    tf: torch.Tensor                 # [B] scaled final time (tf.value[0], LO:178)
    tf_seconds: torch.Tensor         # [B] tf * final_time (LO:194)
    states: Dict[str, torch.Tensor]  # name -> [B, nt], reference `.value` lists, scaled units
    control: Optional[torch.Tensor]  # [B, nt] angledoubledot (node 0 = 0)
    final_mass: torch.Tensor         # [B] kg
    status: torch.Tensor             # [B] int32, 0 = converged
    iterations: torch.Tensor         # [B] int32
    kkt_error: torch.Tensor          # [B]
    time: torch.Tensor               # [nt] normalised mesh (m.time)
    # optional: d tf / d parameter, name -> [B] (scaled tf per unit of the raw parameter), for
    # Ft, M0, M_dot, angle_doubledot_max (NaN for the circular model, which has no such limit) with
    # ``sensitivities=True``, for every name of PARAM_ROWS with ``sensitivities="all"`` (the circular model: NaN for
    # angle_doubledot_max and u_bound, which it does not read).  Partial derivatives: one row of the parameter block
    # moves, the others stay (see optimise_batch).
    dtf_dparam: Optional[Dict[str, torch.Tensor]] = None
    # optional, ``sensitivities="all"`` only: d final_mass / d parameter, name -> [B] (kg per unit of the raw
    # parameter), the partial derivatives of final_mass = M0 - M_dot * final_time * tf
    dfinal_mass_dparam: Optional[Dict[str, torch.Tensor]] = None
    # which reference variable `control` is: the MV `angledoubledot` (LO:96) or, for the circular model, the MV
    # `angle` (PDF p.27 src 69-73)
    control_name: str = "angledoubledot"

    @property
    def converged(self) -> torch.Tensor:
        return self.status == 0

    def __len__(self) -> int:
        return int(self.tf.shape[0])


@dataclasses.dataclass
class AscentSolution:
    tf: float
    tf_seconds: float
    states: Dict[str, torch.Tensor]  # name -> [nt]
    control: torch.Tensor            # [nt]
    final_mass: float
    status: int
    iterations: int
    kkt_error: float
    time: torch.Tensor
    control_name: str = "angledoubledot"


def _empty(shape, dtype: torch.dtype, device: Optional[torch.device]) -> torch.Tensor:
    """A result array of a solve: on ``device``, or in pinned host memory when ``device`` is None."""
    kw = dict(device=device) if device is not None else dict(pin_memory=True)
    return torch.empty(shape, dtype=dtype, **kw)


def alloc_outputs(nt: int, B: int, trajectories: bool = True,
                  device: Optional[torch.device] = None) -> Dict[str, torch.Tensor]:
    """The result arrays of a solve of ``B`` problems on an ``nt``-node mesh (the output layout of
    ``include/lmato_b200.h``): on ``device``, or in pinned host memory when ``device`` is None."""
    return {
        "traj": _empty((_cabi.NVAR, nt, B), torch.float64, device) if trajectories else None,
        "tf": _empty(B, torch.float64, device),
        "final_mass": _empty(B, torch.float64, device),
        "status": _empty(B, torch.int32, device),
        "iterations": _empty(B, torch.int32, device),
        "kkt": _empty(B, torch.float64, device),
    }


class AscentSolver:
    """Owns one C-ABI handle: one device, one mesh, one model."""

    def __init__(self, mesh: Optional[Mesh] = None, options: Optional[SolverOptions] = None,
                 device: Union[int, str, torch.device, None] = None, model: str = "elliptical"):
        self.mesh = mesh or Mesh()
        self.options = options or SolverOptions()
        L = _cabi.lib()
        if not torch.cuda.is_available():
            raise _cabi.LmatoError("no CUDA device: the solver has no CPU fallback")
        if device is None:
            device = torch.cuda.current_device()
        dev = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
        self.device = torch.device("cuda", dev.index if dev.index is not None else torch.cuda.current_device())
        self.time = self.mesh.grid()
        self.nt = int(self.time.shape[0])
        self.model = model
        model_id = {"elliptical": 0, "circular": 1}.get(model)
        if model_id is None:
            raise ValueError(f"unknown model {model!r}")
        self._h = C.c_void_p()
        tbuf = (C.c_double * self.nt)(*self.time.tolist())
        _cabi.check(L.lmato_create(C.byref(self._h), self.device.index, self.nt,
                                   C.cast(tbuf, C.c_void_p), int(self.mesh.nodes), model_id), "lmato_create")
        self.set_options(self.options)

    def set_options(self, o: SolverOptions) -> None:
        co = _c_options(o)
        _cabi.check(_cabi.lib().lmato_set_options(self._h, C.byref(co)), "lmato_set_options")
        self.options = o

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            _cabi.lib().lmato_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- raw entry points ---------------------------------------------------------------
    def alloc_outputs(self, B: int, trajectories: bool = True, on_device: bool = True) -> Dict[str, torch.Tensor]:
        """Result buffers for ``solve_rows(..., out=...)`` (device memory or pinned host memory)."""
        return alloc_outputs(self.nt, B, trajectories, self.device if on_device else None)

    def solve_rows(self, rows: torch.Tensor, trajectories: bool = True,
                   out: Optional[Dict[str, torch.Tensor]] = None,
                   sensitivities: Union[bool, str] = False,
                   guess: Optional[Dict[str, torch.Tensor]] = None) -> Dict[str, torch.Tensor]:
        """``rows``: ``[NPARAM, B]`` float64.  CUDA tensor -> device entry point, results stay on
        the device (asynchronous on the current stream).  CPU tensor -> host entry point
        (H2D + solve + D2H, synchronous), results in pinned host memory.  ``out``: buffers from
        :meth:`alloc_outputs` to write into (avoids re-allocating ~1 GB of trajectories per call).
        ``sensitivities``: also return ``"dtf"`` ``[NSENS, B]`` = d tf / d (Ft, M0, M_dot,
        angle_doubledot_max) from the multipliers at the solution (``lmato_set_sensitivity_output``);
        ``sensitivities="all"``: instead ``"dtf_all"`` ``[NPARAM, B]`` = d tf / d every row of ``rows``
        (``lmato_set_param_sensitivity_output``).
        ``guess``: ``{"traj": [NVAR, nt, B], "tf": [B]}`` (e.g. a previous result of this method, same
        placement as ``rows``) to start from instead of the built-in start (``lmato_set_initial_guess``)."""
        L = _cabi.lib()
        sens_key = _sens_key(sensitivities)
        if rows.dtype != torch.float64 or rows.dim() != 2 or rows.shape[0] != _cabi.NPARAM:
            raise ValueError("rows must be float64 [NPARAM, B]")
        rows = rows.contiguous()
        B = int(rows.shape[1])
        on_dev = rows.is_cuda
        if on_dev and rows.device != self.device:
            raise ValueError(f"rows live on {rows.device}, solver on {self.device}")
        dev = self.device if on_dev else None
        if out is None:
            out = alloc_outputs(self.nt, B, trajectories, dev)
        else:
            if out["tf"].shape[0] != B or out["tf"].is_cuda != on_dev or (trajectories and out["traj"] is None):
                raise ValueError("out buffers do not match this call (batch size / placement / trajectories)")
            if not trajectories:
                out = dict(out, traj=None)
        if sens_key is not None:
            out = dict(out, **{sens_key: _empty((_SENS_OUT[sens_key][0], B), torch.float64, dev)})
        if B == 0:
            return out
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p()
        if guess is not None:
            gt, gf = guess["traj"], guess["tf"]
            if (gt is None or tuple(gt.shape) != (_cabi.NVAR, self.nt, B) or tuple(gf.shape) != (B,) or
                    gt.dtype != torch.float64 or gf.dtype != torch.float64 or gt.is_cuda != on_dev or gf.is_cuda != on_dev):
                raise ValueError("guess must be {'traj': float64 [NVAR, nt, B], 'tf': float64 [B]} placed like rows")
            gt, gf = gt.contiguous(), gf.contiguous()
            _cabi.check(L.lmato_set_initial_guess(self._h, ptr(gt), ptr(gf)), "lmato_set_initial_guess")
        if sens_key is not None:
            fn = _SENS_OUT[sens_key][1]
            _cabi.check(getattr(L, fn)(self._h, ptr(out[sens_key])), fn)
        try:
            self._solve_call(L, rows, B, out, on_dev, ptr)
            if guess is not None and on_dev:
                torch.cuda.current_stream(self.device).synchronize()    # the guess buffers may be temporaries
        finally:
            if sens_key is not None:
                getattr(L, _SENS_OUT[sens_key][1])(self._h, C.c_void_p())
            if guess is not None:
                L.lmato_set_initial_guess(self._h, C.c_void_p(), C.c_void_p())
        return out

    def _solve_call(self, L, rows, B, out, on_dev, ptr) -> None:
        if on_dev:
            with torch.cuda.device(self.device):
                stream = torch.cuda.current_stream(self.device).cuda_stream
                _cabi.check(L.lmato_solve_batch(self._h, ptr(rows), B, ptr(out["traj"]), ptr(out["tf"]),
                                                ptr(out["final_mass"]), ptr(out["status"]),
                                                ptr(out["iterations"]), ptr(out["kkt"]),
                                                C.c_void_p(stream)), "lmato_solve_batch")
        else:
            _cabi.check(L.lmato_solve_batch_host(self._h, ptr(rows), B, ptr(out["traj"]), ptr(out["tf"]),
                                                 ptr(out["final_mass"]), ptr(out["status"]),
                                                 ptr(out["iterations"]), ptr(out["kkt"])),
                        "lmato_solve_batch_host")

    def last_kernel_ms(self) -> float:
        ms = C.c_double()
        _cabi.check(_cabi.lib().lmato_last_kernel_ms(self._h, C.byref(ms)), "lmato_last_kernel_ms")
        return ms.value

    def kernel_launches(self) -> int:
        n = C.c_int64()
        _cabi.check(_cabi.lib().lmato_kernel_launches(self._h, C.byref(n)), "lmato_kernel_launches")
        return n.value

    def workspace_bytes(self, B: int) -> int:
        n = C.c_int64()
        _cabi.check(_cabi.lib().lmato_workspace_bytes(self._h, B, C.byref(n)), "lmato_workspace_bytes")
        return n.value

    def measure_fp64_peak(self) -> float:
        g = C.c_double()
        _cabi.check(_cabi.lib().lmato_measure_fp64_peak(self._h, C.byref(g)), "lmato_measure_fp64_peak")
        return g.value

    def coast_orbit(self, state: torch.Tensor, t_coast: float = 6600.0, dt: float = 1e-3,
                    gm: float = 6.67e-11 * 7.346e22) -> Dict[str, torch.Tensor]:
        """The reference PDF's post-solve orbit check (p.28-29 src 185-237), batched: explicit Euler coast of
        ``state`` ``[4, B]`` = x, y, vx, vy (SI, Moon-centred, CUDA float64) for ``t_coast`` seconds.  Returns the
        extreme radii seen and the final state."""
        if not state.is_cuda or state.dtype != torch.float64 or state.dim() != 2 or state.shape[0] != 4:
            raise ValueError("state must be a CUDA float64 tensor of shape [4, B]")
        state = state.contiguous()
        B = int(state.shape[1])
        out = torch.empty((6, B), dtype=torch.float64, device=self.device)
        nsteps = int(round(t_coast / dt))
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            _cabi.check(_cabi.lib().lmato_coast_orbit(self._h, C.c_void_p(state.data_ptr()), B, float(gm), float(dt),
                                                      nsteps, C.c_void_p(out.data_ptr()), C.c_void_p(stream)),
                        "lmato_coast_orbit")
        return {"r_min": out[0], "r_max": out[1], "final_state": out[2:6]}

    def fly_control(self, rows: torch.Tensor, traj: torch.Tensor, tf: torch.Tensor,
                    substeps: int, trajectories: bool = True) -> Dict[str, torch.Tensor]:
        """``lmato_fly_control``: fly the MV row of ``traj`` ``[NVAR, nt, B]`` (a solve's output on this handle's mesh)
        with final times ``tf`` ``[B]`` and parameters ``rows`` ``[NPARAM, B]`` through the continuous dynamics.  CUDA
        float64 tensors on this solver's device; asynchronous on the current stream.  Returns ``"final"``
        ``[NFLY, B]`` (rows ``_cabi.FLY_ROWS``) and ``"traj"`` ``[NVAR, nt, B]`` (None without ``trajectories``)."""
        B = int(tf.shape[0]) if tf.dim() == 1 else -1
        for name, t, shape in (("rows", rows, (_cabi.NPARAM, B)), ("traj", traj, (_cabi.NVAR, self.nt, B)),
                               ("tf", tf, (B,))):
            if t.device != self.device or t.dtype != torch.float64 or tuple(t.shape) != shape:
                raise ValueError(f"{name} must be a float64 tensor of shape {shape} on {self.device}")
        rows, traj, tf = rows.contiguous(), traj.contiguous(), tf.contiguous()
        out = {"final": torch.empty((_cabi.NFLY, B), dtype=torch.float64, device=self.device),
               "traj": torch.empty_like(traj) if trajectories else None}
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p()
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            _cabi.check(_cabi.lib().lmato_fly_control(self._h, ptr(rows), B, ptr(traj), ptr(tf), int(substeps),
                                                      ptr(out["final"]), ptr(out["traj"]), C.c_void_p(stream)),
                        "lmato_fly_control")
        return out

    def selftest_math(self):
        e = (C.c_double * 5)()
        _cabi.check(_cabi.lib().lmato_selftest_math(self._h, e), "lmato_selftest_math")
        return dict(zip(("rcp", "rsqrt", "log", "sin", "cos"), list(e)))

    # -- packaged result ----------------------------------------------------------------
    def solve(self, params: AscentParams, B: Optional[int] = None, trajectories: bool = True,
              on_device: bool = False) -> AscentBatchSolution:
        rows = params.rows(B, device=self.device if on_device else "cpu")
        if not on_device:
            rows = rows.pin_memory()
        raw = self.solve_rows(rows, trajectories)
        return package_solution(raw, rows, self.time, self.model)


class AscentMultiSolver:
    """Owns one ``lmato_multi`` handle of the C ABI: a device list driven by ONE host process
    (``lmato_multi_create`` / ``lmato_multi_solve_host``).  Host tensors in, pinned host tensors out."""

    def __init__(self, devices: Sequence[int], mesh: Optional[Mesh] = None, options: Optional[SolverOptions] = None,
                 model: str = "elliptical"):
        self.mesh = mesh or Mesh()
        self.options = options or SolverOptions()
        L = _cabi.lib()
        if not torch.cuda.is_available():
            raise _cabi.LmatoError("no CUDA device: the solver has no CPU fallback")
        self.devices = [int(d) for d in devices]
        if not self.devices:
            raise ValueError("`devices` is empty")
        self.time = self.mesh.grid()
        self.nt = int(self.time.shape[0])
        self.model = model
        model_id = {"elliptical": 0, "circular": 1}.get(model)
        if model_id is None:
            raise ValueError(f"unknown model {model!r}")
        self._h = C.c_void_p()
        tbuf = (C.c_double * self.nt)(*self.time.tolist())
        dbuf = (C.c_int32 * len(self.devices))(*self.devices)
        _cabi.check(L.lmato_multi_create(C.byref(self._h), dbuf, len(self.devices), self.nt, C.cast(tbuf, C.c_void_p),
                                         int(self.mesh.nodes), model_id), "lmato_multi_create")
        self.set_options(self.options)

    def set_options(self, o: SolverOptions) -> None:
        _cabi.check(_cabi.lib().lmato_multi_set_options(self._h, C.byref(_c_options(o))), "lmato_multi_set_options")
        self.options = o

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            _cabi.lib().lmato_multi_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def solve_rows(self, rows: torch.Tensor, trajectories: bool = True) -> Dict[str, torch.Tensor]:
        if rows.is_cuda or rows.dtype != torch.float64 or rows.dim() != 2 or rows.shape[0] != _cabi.NPARAM:
            raise ValueError("rows must be a CPU float64 tensor [NPARAM, B]")
        rows = rows.contiguous()
        B = int(rows.shape[1])
        out = alloc_outputs(self.nt, B, trajectories)
        if B == 0:
            return out
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p()
        _cabi.check(_cabi.lib().lmato_multi_solve_host(self._h, ptr(rows), B, ptr(out["traj"]), ptr(out["tf"]),
                                                       ptr(out["final_mass"]), ptr(out["status"]), ptr(out["iterations"]),
                                                       ptr(out["kkt"])), "lmato_multi_solve_host")
        return out


def _c_options(o: SolverOptions) -> "_cabi.LmatoOptions":
    return _cabi.LmatoOptions(tol=o.tol, mu_init=o.mu_init, obj_scale=o.obj_scale, tf_guess=o.tf_guess,
                              delta_c=o.delta_c, mu_min_factor=o.mu_min_factor, max_iter=int(o.max_iter),
                              max_ls=int(o.max_ls), n_polish=int(o.n_polish),
                              warm_start=int(o.warm_start), mu_ref=o.mu_ref,
                              dcost=float(1e-5 if o.dcost is None else o.dcost),
                              kappa_eps=float(o.kappa_eps), objective_nodes=int(o.objective_nodes),
                              kernel=_cabi.KERNEL_IDS[o.kernel], coop_lanes=int(o.coop_lanes), otol=float(o.otol),
                              rtol=float(o.rtol))


# the key of a solve_rows result and the C entry that registers it, per `sensitivities` setting
_SENS_OUT = {"dtf": (_cabi.NSENS, "lmato_set_sensitivity_output"),
             "dtf_all": (_cabi.NPARAM, "lmato_set_param_sensitivity_output")}


def _sens_key(sensitivities: Union[bool, str]) -> Optional[str]:
    if isinstance(sensitivities, str) and sensitivities != "all":
        raise ValueError(f"sensitivities must be False, True or 'all', not {sensitivities!r}")
    return "dtf_all" if sensitivities == "all" else "dtf" if sensitivities else None


def dfinal_mass_dparam(dtf: torch.Tensor, rows: torch.Tensor, tf: torch.Tensor) -> torch.Tensor:
    """``[NPARAM, B]`` partial derivatives of final_mass = M0 - M_dot * final_time * tf (the library's output,
    LO:123) with respect to every row of the parameter block, from ``dtf`` = d tf / d row (``[NPARAM, B]``)."""
    rows = rows.to(dtf.device)
    tf = tf.to(dtf.device)
    i = _cabi.PARAM_ROWS.index
    mdot, T = rows[i("M_dot")], rows[i("final_time")]
    out = -(mdot * T) * dtf
    out[i("M0")] += 1.0
    out[i("M_dot")] -= T * tf
    out[i("final_time")] -= mdot * tf
    return out


def package_solution(raw: Dict[str, torch.Tensor], rows: torch.Tensor, time: torch.Tensor,
                     model: str = "elliptical") -> AscentBatchSolution:
    traj = raw["traj"]
    states: Dict[str, torch.Tensor] = {}
    control = None
    if traj is not None:
        for i, name in enumerate(_cabi.VAR_ROWS):
            states[name] = traj[i].transpose(0, 1)      # [B, nt] view
        if model == "circular":
            # PDF p.27 src 54-73: the Vars are y, ydot, ydoubledot, x, xdot, xdoubledot, mass and the
            # MV is `angle`; angledot / angledoubledot do not exist in that model
            states.pop("angledot"); states.pop("angledoubledot")
            control = states.pop("angle")
        else:
            control = states.pop("angledoubledot")
    T = rows[_cabi.PARAM_ROWS.index("final_time")]
    dtf, dtf_all = raw.get("dtf"), raw.get("dtf_all")
    dtf_dparam = dfm_dparam = None
    if dtf is not None:
        dtf_dparam = {n: dtf[i] for i, n in enumerate(_cabi.SENS_ROWS)}
    elif dtf_all is not None:
        dtf_dparam = {n: dtf_all[i] for i, n in enumerate(_cabi.PARAM_ROWS)}
        dfm = dfinal_mass_dparam(dtf_all, rows, raw["tf"])
        dfm_dparam = {n: dfm[i] for i, n in enumerate(_cabi.PARAM_ROWS)}
    return AscentBatchSolution(tf=raw["tf"], tf_seconds=raw["tf"] * T.to(raw["tf"].device), states=states,
                               control=control, final_mass=raw["final_mass"], status=raw["status"],
                               iterations=raw["iterations"], kkt_error=raw["kkt"], time=time,
                               dtf_dparam=dtf_dparam, dfinal_mass_dparam=dfm_dparam,
                               control_name="angle" if model == "circular" else "angledoubledot")


# ---------------------------------------------------------------------------------------
# index-partitioned multi-GPU solve: problem i -> rank floor(i*G/B); ONE allgather at the end
# ---------------------------------------------------------------------------------------
def shard_bounds(B: int, world: int, rank: int):
    """Contiguous index ranges, sizes differ by at most one."""
    lo = (B * rank) // world
    hi = (B * (rank + 1)) // world
    return lo, hi


def sharded_solve(rows: torch.Tensor, solve_fn: Callable[[torch.Tensor], Dict[str, torch.Tensor]],
                  group=None, gather: bool = True, gather_traj: bool = True) -> Dict[str, torch.Tensor]:
    """Every rank holds the full ``rows`` block; rank r solves its contiguous shard with
    ``solve_fn`` and a single ``all_gather`` (NCCL over NVLink on GPUs, gloo in the CPU tests)
    reassembles the per-problem results on every rank.  No per-iteration collectives: the
    problems are independent.  ``gather_traj=False`` gathers the per-problem scalars only (tf, final mass,
    status, iterations, KKT error: 40 B per problem) and returns the rank's own trajectory shard under
    ``"traj"`` together with its index range ``"shard"`` (SURVEY 8e: the trajectories are optional)."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    B = int(rows.shape[1])
    lo, hi = shard_bounds(B, world, rank)
    local = solve_fn(rows[:, lo:hi].contiguous())
    if not gather:
        return local
    per = (B + world - 1) // world
    keys = [k for k, v in local.items() if v is not None and (gather_traj or k != "traj")]
    # pack every result into one float64 buffer [per, width] so that one collective suffices
    cols = []
    for k in keys:
        v = local[k]
        if k == "traj":
            v = v.permute(2, 0, 1).reshape(hi - lo, -1)
        else:
            v = v.reshape(hi - lo, 1)
        cols.append(v.to(torch.float64))
    packed = torch.cat(cols, dim=1)
    width = packed.shape[1]
    send = torch.zeros((per, width), dtype=torch.float64, device=packed.device)
    send[: hi - lo] = packed
    recv = torch.empty((world * per, width), dtype=torch.float64, device=packed.device)
    dist.all_gather_into_tensor(recv, send, group=group)
    pieces = []
    for r in range(world):
        l, h = shard_bounds(B, world, r)
        pieces.append(recv[r * per: r * per + (h - l)])
    full = torch.cat(pieces, dim=0)
    out: Dict[str, torch.Tensor] = {k: None for k in local}
    c = 0
    for k in keys:
        v = local[k]
        if k == "traj":
            w = v.shape[0] * v.shape[1]
            out[k] = full[:, c: c + w].reshape(B, v.shape[0], v.shape[1]).permute(1, 2, 0).contiguous()
        else:
            w = 1
            out[k] = full[:, c].to(v.dtype)
        c += w
    if not gather_traj:
        out["traj"] = local.get("traj")
        out["shard"] = (lo, hi)
    return out


def multi_device_solve(rows: torch.Tensor, solvers: List["AscentSolver"], trajectories: bool = True,
                       out_device: Union[str, torch.device, None] = None,
                       sensitivities: Union[bool, str] = False) -> Dict[str, torch.Tensor]:
    """One host process, several GPUs (no torchrun): problem i goes to GPU ``floor(i*G/B)`` (the same
    contiguous index partition as :func:`sharded_solve`).  The device entry point is asynchronous, so
    all launches are issued first and every GPU solves its shard concurrently; the shards are then
    copied into one result block on ``out_device`` (default: the first solver's device; peer copies
    over NVLink) or into pinned host memory (``"cpu"``)."""
    G = len(solvers)
    B = int(rows.shape[1])
    # distribute ALL shards first: a peer copy is ordered behind whatever its source device has queued, so
    # copying shard g+1 after launching solve g would make every other GPU wait for the first one's kernel
    shards = []
    for g, solver in enumerate(solvers):
        lo, hi = shard_bounds(B, G, g)
        shards.append(rows[:, lo:hi].to(solver.device, non_blocking=True).contiguous())
    if rows.is_cuda:
        torch.cuda.synchronize(rows.device)
    parts = []
    for g, solver in enumerate(solvers):
        with torch.cuda.device(solver.device):
            parts.append(solver.solve_rows(shards[g], trajectories, sensitivities=sensitivities)
                         if shards[g].shape[1] > 0 else None)
    # Assemble on the first solver's device: each shard travels as ONE contiguous peer copy (NVLink) and is
    # placed into its strided slot of the [.., B] block by a local copy kernel; a host result is then a single
    # contiguous transfer into pinned memory.
    hub = solvers[0].device
    ref = next(p for p in parts if p is not None)
    keys = [k for k, v in ref.items() if v is not None]
    out: Dict[str, Optional[torch.Tensor]] = {k: None for k in ref}
    for solver in solvers:
        torch.cuda.synchronize(solver.device)
    with torch.cuda.device(hub):
        for k in keys:
            shape = list(ref[k].shape)
            shape[-1] = B
            out[k] = torch.empty(shape, dtype=ref[k].dtype, device=hub)
        for g, part in enumerate(parts):
            if part is None:
                continue
            lo, hi = shard_bounds(B, G, g)
            for k in keys:
                out[k][..., lo:hi] = part[k].to(hub, non_blocking=True)
        torch.cuda.synchronize(hub)
        dst = torch.device(out_device) if out_device is not None else hub
        if dst.type == "cpu":
            for k in keys:
                host = torch.empty(out[k].shape, dtype=out[k].dtype, pin_memory=True)
                host.copy_(out[k], non_blocking=True)
                out[k] = host
            torch.cuda.synchronize(hub)
        elif dst != hub:
            out = {k: (v.to(dst) if v is not None else None) for k, v in out.items()}
    return out


def final_state_si(sol: AscentBatchSolution, params: AscentParams) -> torch.Tensor:
    """Final ascent state in the PDF's plotting frame (src 189-192): ``[4, B]`` = (-x*S, y*S+R0, -xdot*S, ydot*S)."""
    B = len(sol)
    rows = params.rows(B, device=sol.tf.device)
    S, R0 = rows[_cabi.PARAM_ROWS.index("r_periapsis")], rows[_cabi.PARAM_ROWS.index("R0")]
    st = sol.states
    return torch.stack([-st["x"][:, -1] * S, st["y"][:, -1] * S + R0, -st["xdot"][:, -1] * S, st["ydot"][:, -1] * S])


# ---------------------------------------------------------------------------------------
# post-solve flight: the solved control flown through the continuous dynamics
# ---------------------------------------------------------------------------------------
# Length of one RK4 sub-step in normalised time: 16 sub-steps per step of the reference's nt = 200 mesh.
FLY_SUBSTEP = 1.0 / (16 * 199)


def default_fly_substeps(time: torch.Tensor) -> int:
    """RK4 sub-steps per mesh step that :func:`fly` takes by default: the smallest power of two that keeps every
    sub-step of the mesh ``time`` no longer than ``FLY_SUBSTEP``.

    On the reference mesh (nt = 200) that is 16: the smallest power of two for which multiplying the count by 4
    changes the flown end state by less than 1e-10 relative (measured on the host build against the oracle fixtures:
    16 -> 64 changes it by 1.4e-11, 8 -> 32 by 2.5e-10).  RK4's error is set by the sub-step length, so a coarser mesh
    gets more sub-steps per step; on every fixture mesh (nt 20 ... 200, uniform and non-uniform, both models) the
    count this gives changes the end state by at most 1.0e-11 when it is multiplied by 4
    (``tests/test_fly_on_host.py``)."""
    hmax = float(torch.diff(time.to(torch.float64).cpu()).max())
    n = 1
    while hmax > n * FLY_SUBSTEP * (1 + 1e-9):       # (a uniform mesh's steps differ from 1/(nt-1) by rounding)
        n *= 2
    return n


@dataclasses.dataclass
class FlownAscent:
    """A solved control flown through the continuous dynamics (:func:`fly`).  ``B`` = 1 for an :class:`AscentSolution`."""
    states: Dict[str, torch.Tensor]   # name -> [B, nt], the names of the solution's states, scaled units
    final_state: Dict[str, torch.Tensor]   # y, ydot, x, xdot, angle, angledot, mass at tf -> [B], scaled
    radius_miss_m: torch.Tensor       # [B] flown radius at tf minus the target radius R0 + r_periapsis (LO:161)
    speed_miss_mps: torch.Tensor      # [B] flown speed at tf minus the target speed (LO:75, 169)
    flight_path_angle_rad: torch.Tensor   # [B] asin(r.v / (|r| |v|)) at tf; the target is 0 (LO:173)
    substeps: int                     # RK4 sub-steps per mesh step
    S: torch.Tensor                   # [B] distance scale r_periapsis (LO:73)
    R0: torch.Tensor                  # [B] lunar radius

    def final_state_si(self) -> torch.Tensor:
        """Flown insertion state in the frame of :func:`final_state_si`: ``[4, B]`` = (-x*S, y*S+R0, -xdot*S, ydot*S),
        the start state :meth:`AscentSolver.coast_orbit` takes."""
        f, S = self.final_state, self.S
        return torch.stack([-f["x"] * S, f["y"] * S + self.R0, -f["xdot"] * S, f["ydot"] * S])


def fly(solution: Union[AscentBatchSolution, AscentSolution], params: AscentParams,
        substeps: Optional[int] = None) -> FlownAscent:
    """Fly the solved control of ``solution`` through the continuous ascent dynamics (LO:114-136) on the GPU and
    report each problem's insertion miss.

    A solve returns the optimum of the transcribed problem; this shows how far the vehicle ends up from the target
    orbit when it flies that control.  Classical RK4 with ``substeps`` sub-steps per mesh step (default:
    :func:`default_fly_substeps`), the MV of node k held on (t_{k-1}, t_k] as both transcriptions hold it, so the
    flight does not depend on NODES.  ``params`` are the solve's parameters.  ``solution`` needs its trajectories
    and may live on the CPU or a GPU; the results follow its placement, as :func:`optimise_batch` does.  Problems that
    did not converge are flown as given (check ``solution.status``)."""
    if solution.control is None or not solution.states:
        raise ValueError("fly() needs a solution with trajectories")
    model = "circular" if solution.control_name == "angle" else "elliptical"
    if params.model != model:
        raise ValueError(f"params are of the {params.model} model, the solution of the {model} model")
    single = isinstance(solution, AscentSolution)
    expand = (lambda t: t.unsqueeze(0)) if single else (lambda t: t)
    src = solution.control.device
    dev = src if src.type == "cuda" else torch.device("cuda", torch.cuda.current_device())
    solver = _get_solver(Mesh(time=solution.time.tolist()), SolverOptions(), dev, model)
    control = expand(solution.control)
    B, nt = int(control.shape[0]), int(control.shape[1])
    if nt != solver.nt:
        raise ValueError(f"the solution has {nt} nodes, its time grid {solver.nt}")
    cols = []
    for name in _cabi.VAR_ROWS:
        if name == solution.control_name:
            cols.append(control)
        elif name in solution.states:
            cols.append(expand(solution.states[name]))
        else:
            cols.append(torch.zeros_like(control))
    traj = torch.stack([c.to(dev, torch.float64).transpose(0, 1) for c in cols])      # [NVAR, nt, B]
    tf = torch.as_tensor(solution.tf, dtype=torch.float64).reshape(-1).to(dev)
    rows = params.rows(B, device=dev)
    n = default_fly_substeps(solution.time) if substeps is None else int(substeps)
    out = solver.fly_control(rows, traj, tf, n)
    if src.type != "cuda":
        out = {k: v.cpu() for k, v in out.items()}
        rows = rows.cpu()
    fin = out["final"]
    states = {name: out["traj"][i].transpose(0, 1) for i, name in enumerate(_cabi.VAR_ROWS) if name in solution.states}
    return FlownAscent(states=states, final_state={n_: fin[i] for i, n_ in enumerate(_cabi.FLY_ROWS[:7])},
                       radius_miss_m=fin[7], speed_miss_mps=fin[8], flight_path_angle_rad=fin[9], substeps=n,
                       S=rows[_cabi.PARAM_ROWS.index("r_periapsis")], R0=rows[_cabi.PARAM_ROWS.index("R0")])


# ---------------------------------------------------------------------------------------
# public functions
# ---------------------------------------------------------------------------------------
_solver_cache: Dict[tuple, AscentSolver] = {}


def _get_solver(mesh: Mesh, options: SolverOptions, device, model: str) -> AscentSolver:
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    dev = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
    key = (dev.index or 0, tuple(mesh.grid().tolist()), mesh.nodes, model)
    s = _solver_cache.get(key)
    if s is None:
        s = AscentSolver(mesh, options, dev, model)
        _solver_cache[key] = s
    else:
        s.set_options(options)
    return s


def optimise_batch(params: AscentParams, mesh: Optional[Mesh] = None,
                   options: Optional[SolverOptions] = None, device=None, batch: Optional[int] = None,
                   trajectories: bool = True, group=None,
                   devices: Optional[Sequence[int]] = None, sensitivities: Union[bool, str] = False,
                   guess: Optional[AscentBatchSolution] = None) -> AscentBatchSolution:
    """Solve a batch of ascent problems (one per entry of the ``[B]`` parameter tensors).

    Results follow the placement of the inputs: CPU parameter tensors (or plain floats) give
    pinned CPU result tensors (host->device and device->host copies are part of the call);
    CUDA parameter tensors give CUDA results without any host transfer.

    ``group``: a ``torch.distributed`` process group (or ``True`` for the default group).  Every
    rank passes the same full batch; rank r solves the contiguous index shard
    ``[B*r/G, B*(r+1)/G)`` on its own GPU and one allgather returns the full result everywhere.

    ``devices``: GPU indices to shard over from THIS process (same partition, no process group, no
    collective: the shards are copied into one result block, see :func:`multi_device_solve`).

    ``sensitivities``: also return ``dtf_dparam`` (d tf / d Ft, M0, M_dot, angle_doubledot_max per
    problem; SURVEY 8f.4).  ``sensitivities="all"``: ``dtf_dparam`` for every name of ``PARAM_ROWS`` and
    ``dfinal_mass_dparam`` (d final_mass / d the same rows).  Not available together with ``group``.
    These are partial derivatives with respect to rows of the parameter block (``params.rows()``), each row moved
    with the others held.  Where a field of ``params`` sets more than one row, the total derivative is the sum over
    those rows: ``mass_scalar=None`` follows ``fuel_mass``, so the derivative with respect to the reference's tied
    fuel mass is ``dtf_dparam["fuel_mass"] + dtf_dparam["mass_scalar"]``; with ``Isp`` given, ``M_dot`` is derived
    from ``Ft`` and ``Isp`` and the ``Ft`` row holds thrust at fixed ``M_dot``.

    ``guess``: a previous :class:`AscentBatchSolution` of the same batch size and mesh (elliptical
    model) to start from -- the counterpart of the ``value=`` arguments at LO:39, 83-96.  Single
    device only.
    """
    mesh = mesh or Mesh()
    options = options or SolverOptions()
    _sens_key(sensitivities)
    if options.dcost is None:          # the move-suppression weight travels with the model parameters
        options = dataclasses.replace(options, dcost=float(params.dcost))
    on_dev = any(isinstance(getattr(params, f.name), torch.Tensor) and getattr(params, f.name).is_cuda
                 for f in dataclasses.fields(params))
    if guess is not None and (devices is not None or group is not None):
        raise ValueError("`guess` is supported on a single device only")
    if devices is not None:
        if group is not None:
            raise ValueError("pass either `group` (one process per GPU) or `devices` (one process), not both")
        if len(devices) == 0:
            raise ValueError("`devices` is empty")
        nB = batch if batch is not None else (params.batch_size() or 1)
        if options.warm_start == 1 and nB >= 512:
            # the shards belong to one batch: they keep the batch warm start even if a shard alone is small
            options = dataclasses.replace(options, warm_start=2)
        if not on_dev and not sensitivities:
            # host tensors: the C ABI's own device-list entry (lmato_multi_solve_host)
            key = ("multi", tuple(int(d) for d in devices), tuple(mesh.grid().tolist()), mesh.nodes, params.model)
            ms = _solver_cache.get(key)
            if ms is None:
                ms = _solver_cache[key] = AscentMultiSolver(devices, mesh, options, params.model)
            else:
                ms.set_options(options)
            rows = params.rows(batch).pin_memory()
            return package_solution(ms.solve_rows(rows, trajectories), rows, ms.time, params.model)
        solvers = [_get_solver(mesh, options, d, params.model) for d in devices]
        rows = params.rows(batch, device=solvers[0].device if on_dev else "cpu")
        if not on_dev:
            rows = rows.pin_memory()
        raw = multi_device_solve(rows, solvers, trajectories, out_device=None if on_dev else "cpu",
                                 sensitivities=sensitivities)
        return package_solution(raw, rows, solvers[0].time, params.model)
    solver = _get_solver(mesh, options, device, params.model)
    rows = params.rows(batch, device=solver.device if on_dev else "cpu")
    if group is not None:
        if sensitivities:
            raise ValueError("sensitivities are not gathered across a process group; use `devices=` or one GPU")
        import torch.distributed as dist
        g = None if group is True else group
        dev_rows = rows.to(solver.device)
        raw = sharded_solve(dev_rows, lambda r: solver.solve_rows(r, trajectories), g)
        if not on_dev:
            raw = {k: (v.cpu() if v is not None else None) for k, v in raw.items()}
        return package_solution(raw, rows, solver.time, params.model)
    if not on_dev:
        rows = rows.pin_memory()
    g = None
    if guess is not None:
        if params.model != "elliptical" or guess.control is None or "angledot" not in guess.states:
            raise ValueError("`guess` must be a solution of the elliptical model with trajectories")
        cols = [guess.control if n == "angledoubledot" else guess.states[n] for n in _cabi.VAR_ROWS]
        gt = torch.stack([c.transpose(0, 1) for c in cols]).to(rows.device)        # [NVAR, nt, B]
        gf = guess.tf.to(rows.device)
        if not on_dev:
            gt, gf = gt.pin_memory(), gf.pin_memory()
        g = {"traj": gt, "tf": gf}
    raw = solver.solve_rows(rows, trajectories, sensitivities=sensitivities, guess=g)
    return package_solution(raw, rows, solver.time, params.model)


def optimise(params: Optional[AscentParams] = None, mesh: Optional[Mesh] = None,
             options: Optional[SolverOptions] = None, device=None) -> AscentSolution:
    """Solve one ascent problem; the single-instance twin of the reference script.
    Raises ``LmatoError`` if the solver does not converge (the reference raises a bare
    ``Exception`` from ``m.solve``, LO:177)."""
    params = params or AscentParams()
    sol = optimise_batch(params, mesh, options, device, batch=1)
    st = int(sol.status[0])
    if st != 0:
        raise _cabi.LmatoError(f"@error: Solution Not Found (status {st}: {_cabi.STATUS_NAMES.get(st, '?')}, "
                               f"kkt error {float(sol.kkt_error[0]):.3e} after {int(sol.iterations[0])} iterations)")
    return AscentSolution(tf=float(sol.tf[0]), tf_seconds=float(sol.tf_seconds[0]),
                          states={k: v[0].clone() for k, v in sol.states.items()},
                          control=sol.control[0].clone(), final_mass=float(sol.final_mass[0]), status=st,
                          iterations=int(sol.iterations[0]), kkt_error=float(sol.kkt_error[0]), time=sol.time,
                          control_name=sol.control_name)
