"""CPU oracle, part 1: the ascent NLP exactly as the reference states it.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is imported by the product
package; only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs may use it, and only as the checker.

PARITY UNPINNED (by the letter of the rule): the reference delegates all arithmetic
to GEKKO + the closed-source ``apm`` binary + IPOPT, none of which exist in this
container or in ``/root/reference``, and the reference has no tests.  The only pins
are two screenshots of program output (``Numerical_results.png`` and PDF p.30), which
this restatement reproduces to 2e-5 / 3e-6 in ``tf`` (tests/test_oracle_golden.py).

What is restated here, literally (``LO:n`` = /root/reference/Launch_Optimiser.py:n,
``PDF p.N src a-b`` = code screenshot on page N of the reference PDF):

* variables and bounds ......... LO:39, LO:83-100   (circular: PDF p.26-27 src 50-73)
* constants and scales ......... LO:38, LO:50-75, LO:107-109
* differential equations ....... LO:114-123         (circular: PDF p.27 src 76-83)
* algebraic dynamics ........... LO:127-136         (circular: PDF p.27 src 87-96)
* initial conditions ........... LO:145-151 (+ GEKKO pins every variable at node 0)
* terminal constraints ......... LO:158-173         (circular: PDF p.27 src 112-126)
* objective .................... LO:176 (+ DCOST LO:99, see ``dcost`` below)
* transcription ................ GEKKO IMODE=6 orthogonal collocation on the mesh
  LO:20-21 with NODES (LO:25) Lobatto points per step; NODES=2 is backward Euler.

The variable set is kept *literal* (all 9 GEKKO Vars + the MV per node, one global
``tf``, two terminal slacks) on purpose: the CUDA product eliminates ``ydoubledot``,
``xdoubledot`` and ``mass`` and carries ``tf`` as a stage state, so agreement between
the two is a meaningful check of both.  Derivatives here come from sympy, the product's
are hand-derived.
"""
from __future__ import annotations

import dataclasses
import functools
import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import scipy.sparse as sp
import sympy as sy


# --------------------------------------------------------------------------------------
# Parameters (names follow the reference script)
# --------------------------------------------------------------------------------------
@dataclasses.dataclass
class AscentParams:
    """Physical parameters; defaults are the literals of Launch_Optimiser.py."""

    G: float = 6.674e-11            # LO:50
    M: float = 7.346e22             # LO:51
    R0: float = 1738100.0           # LO:52
    Ft: float = 15346.0             # LO:61
    M0: float = 4821.0              # LO:62
    M_dot: float = 5.053            # LO:63 / numerator of mflow LO:65
    fuel_mass: float = 2376.0       # LO:64
    angle_doubledot_max: float = 5e-4   # LO:66
    r_periapsis: float = 17703.0    # LO:70
    r_apoapsis: float = 88615.0     # LO:71
    final_time: float = 470.0       # LO:38
    model: str = "elliptical"       # "elliptical" (script) | "circular" (PDF p.26-28)
    mass_scalar: Optional[float] = None  # LO:108 = fuel_mass; PDF p.27 src 67 = 2576
    angle_ub: float = math.pi / 3   # LO:94
    u_bound: float = 1.0            # LO:96
    dcost: float = 0.0              # LO:99 is 1e-5; 0 = without the move-suppression term (DESIGN.md 7)

    @staticmethod
    def circular() -> "AscentParams":
        """The 'original IB-document' model: PDF p.26 src 32-46, p.27 src 66-67."""
        return AscentParams(r_periapsis=53108.4, r_apoapsis=53108.4,
                            model="circular", mass_scalar=2576.0)

    # derived (LO:65, 72-75, 107-109)
    @property
    def GM(self) -> float:
        return self.G * self.M

    @property
    def S(self) -> float:           # distance scale = Rfmin = r_periapsis  (LO:73, 107)
        return self.r_periapsis

    @property
    def mscale(self) -> float:
        return self.fuel_mass if self.mass_scalar is None else self.mass_scalar

    @property
    def mflow(self) -> float:       # LO:65
        return self.M_dot / self.fuel_mass

    @property
    def asc(self) -> float:         # LO:109
        return self.angle_doubledot_max / 3.0

    @property
    def v_target(self) -> float:    # LO:75 (circular speed at the mean radius)
        r_avg = 0.5 * (self.r_periapsis + self.r_apoapsis)
        return math.sqrt(self.GM / (self.R0 + r_avg))


PARAM_SYMS = ["GM", "R0", "Ft", "M0", "S", "mscale", "mflow", "asc", "T"]


def _param_vector(p: AscentParams) -> np.ndarray:
    return np.array([p.GM, p.R0, p.Ft, p.M0, p.S, p.mscale, p.mflow, p.asc,
                     p.final_time], dtype=np.float64)


# --------------------------------------------------------------------------------------
# Symbolic model (one mesh node) -> numpy callables
# --------------------------------------------------------------------------------------
@dataclasses.dataclass
class _NodeModel:
    names: List[str]            # per-node variable names, GEKKO order
    ndiff: int                  # number of differential rows
    diff_idx: List[int]         # index in `names` of each differential variable
    lb: np.ndarray
    ub: np.ndarray
    rhs: callable               # (v[nv,K], tf, P) -> [ndiff, K]   d/dtau right-hand sides
    rhs_jac: callable           # -> dense [ndiff, nv+1, K] (last column: d/dtf)
    rhs_hess: callable          # (v, tf, P, w[ndiff,K]) -> [nv+1, nv+1, K]
    alg: callable               # (v, P) -> [nalg, K]
    alg_jac: callable           # -> [nalg, nv, K]
    alg_hess: callable          # (v, P, w[nalg,K]) -> [nv, nv, K]
    nalg: int


def _accel_expr(y, x, a, m, P):
    """LO:127-136 verbatim structure (same for the circular model, PDF p.27 src 87-96)."""
    GM, R0, Ft, M0, S, mscale = P["GM"], P["R0"], P["Ft"], P["M0"], P["S"], P["mscale"]
    X = x * S
    Y = y * S + R0
    r2 = X ** 2 + Y ** 2
    k = Ft / ((M0 - mscale * m) * sy.sqrt(r2))
    ydd = (k * (Y * sy.cos(3 * a) + X * sy.sin(3 * a)) - Y * (GM / r2 ** sy.Rational(3, 2))) / S
    xdd = (k * (X * sy.cos(3 * a) - Y * sy.sin(3 * a)) - X * (GM / r2 ** sy.Rational(3, 2))) / S
    return ydd, xdd


@functools.lru_cache(maxsize=None)
def _build_node_model(model: str) -> _NodeModel:
    P = {n: sy.Symbol(n, real=True) for n in PARAM_SYMS}
    tf = sy.Symbol("tf", real=True)
    if model == "elliptical":
        names = ["y", "ydot", "ydoubledot", "x", "xdot", "xdoubledot",
                 "angle", "angledot", "mass", "angledoubledot"]          # LO:83-96
    elif model == "circular":
        names = ["y", "ydot", "ydoubledot", "x", "xdot", "xdoubledot",
                 "mass", "angle"]                                        # PDF src 54-69
    else:
        raise ValueError(f"unknown model {model!r}")
    V = {n: sy.Symbol(n, real=True) for n in names}
    T = P["T"]
    if model == "elliptical":
        diff = ["y", "ydot", "x", "xdot", "angle", "angledot", "mass"]
        rhs = [tf * V["ydot"] * T,                     # LO:114
               tf * V["ydoubledot"] * T,               # LO:115
               tf * V["xdot"] * T,                     # LO:117
               tf * V["xdoubledot"] * T,               # LO:118
               tf * V["angledot"] * T,                 # LO:120
               tf * V["angledoubledot"] * T * P["asc"],  # LO:121
               P["mflow"] * T * tf]                    # LO:123
    else:
        diff = ["y", "ydot", "x", "xdot", "mass"]
        rhs = [tf * V["ydot"] * T, tf * V["ydoubledot"] * T,             # PDF src 76-77
               tf * V["xdot"] * T, tf * V["xdoubledot"] * T,             # PDF src 80-81
               P["mflow"] * T * tf]                                      # PDF src 83
    ydd, xdd = _accel_expr(V["y"], V["x"], V["angle"], V["mass"], P)
    alg = [V["ydoubledot"] - ydd, V["xdoubledot"] - xdd]                 # LO:127-136

    vs = [V[n] for n in names]
    ps = [P[n] for n in PARAM_SYMS]
    nv = len(vs)

    def lam(args, exprs):
        return sy.lambdify(args, exprs, modules="numpy", cse=True)

    rhs_f = lam(vs + [tf] + ps, rhs)
    rhs_J = lam(vs + [tf] + ps, [[sy.diff(e, s) for s in vs + [tf]] for e in rhs])
    w_r = [sy.Symbol(f"wr{i}", real=True) for i in range(len(rhs))]
    Lr = sum(w * e for w, e in zip(w_r, rhs))
    rhs_H = lam(vs + [tf] + ps + w_r, [[sy.diff(Lr, s1, s2) for s2 in vs + [tf]] for s1 in vs + [tf]])
    alg_f = lam(vs + ps, alg)
    alg_J = lam(vs + ps, [[sy.diff(e, s) for s in vs] for e in alg])
    w_a = [sy.Symbol(f"wa{i}", real=True) for i in range(len(alg))]
    La = sum(w * e for w, e in zip(w_a, alg))
    alg_H = lam(vs + ps + w_a, [[sy.diff(La, s1, s2) for s2 in vs] for s1 in vs])

    def _stack(out, K):
        nested = isinstance(out[0], (list, tuple))
        a = np.empty((len(out),) + ((len(out[0]),) if nested else ()) + (K,))
        if nested:
            for i, row in enumerate(out):
                for j, e in enumerate(row):
                    a[i, j, :] = e
        else:
            for i, e in enumerate(out):
                a[i, :] = e
        return a

    def f_rhs(v, tfv, Pv):
        return _stack(rhs_f(*v, tfv, *Pv), v.shape[1])

    def f_rhs_jac(v, tfv, Pv):
        return _stack(rhs_J(*v, tfv, *Pv), v.shape[1])

    def f_rhs_hess(v, tfv, Pv, w):
        return _stack(rhs_H(*v, tfv, *Pv, *w), v.shape[1])

    def f_alg(v, Pv):
        return _stack(alg_f(*v, *Pv), v.shape[1])

    def f_alg_jac(v, Pv):
        return _stack(alg_J(*v, *Pv), v.shape[1])

    def f_alg_hess(v, Pv, w):
        return _stack(alg_H(*v, *Pv, *w), v.shape[1])

    lb = np.full(nv, -np.inf)
    ub = np.full(nv, np.inf)
    lb[names.index("mass")], ub[names.index("mass")] = 0.0, 1.0          # LO:83
    # angle / control bounds are filled per-instance (angle_ub, u_bound) in AscentNLP
    return _NodeModel(names=names, ndiff=len(diff), diff_idx=[names.index(d) for d in diff],
                      lb=lb, ub=ub, rhs=f_rhs, rhs_jac=f_rhs_jac, rhs_hess=f_rhs_hess,
                      alg=f_alg, alg_jac=f_alg_jac, alg_hess=f_alg_hess, nalg=len(alg))


# --------------------------------------------------------------------------------------
# Collocation matrices (SURVEY Appendix B.2): Lobatto points on [0,1], derivative
# interpolated on the non-initial points and integrated.
# --------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def collocation_matrix(nodes: int) -> Tuple[np.ndarray, np.ndarray]:
    """Return (tau[nodes], N[(nodes-1),(nodes-1)]) with  h*N*xdot_{1..} = x_{1..} - x_0."""
    if nodes < 2 or nodes > 6:
        raise ValueError("NODES must be 2..6 (GEKKO's range)")
    if nodes == 2:
        return np.array([0.0, 1.0]), np.array([[1.0]])
    s = sy.Symbol("s")
    # Gauss-Lobatto points on [-1,1]: +-1 and the roots of P'_{n-1}
    roots = sy.Poly(sy.diff(sy.legendre(nodes - 1, s), s), s).nroots(n=30)
    pts = sorted([-1.0] + [float(r) for r in roots] + [1.0])
    tau = [(p + 1) / 2 for p in pts]
    tq = [sy.nsimplify(t, rational=False) for t in tau]
    n1 = nodes - 1
    N = np.zeros((n1, n1))
    for j in range(n1):
        ell = sy.Integer(1)
        for m in range(n1):
            if m != j:
                ell *= (s - tau[m + 1]) / (tau[j + 1] - tau[m + 1])
        I = sy.integrate(sy.expand(ell), s)
        for i in range(n1):
            N[i, j] = float(I.subs(s, tau[i + 1]) - I.subs(s, 0))
    return np.array(tau), N


# --------------------------------------------------------------------------------------
# The transcribed NLP:  min f(x)  s.t.  c(x) = 0,  lb <= x <= ub
# --------------------------------------------------------------------------------------
class AscentNLP:
    """GEKKO IMODE=6 transcription of the ascent problem on a normalised time mesh.

    Unknown vector ``x`` = [v_1 .. v_K (nv each, K collocation points, node 0 pinned
    and therefore absent), tf, s_radius, s_speed].  For NODES=2, K = nt-1 and point k is
    mesh node k.  For NODES>2 each of the nt-1 steps carries (NODES-1) points, the last
    of which is the mesh node; the MV is held constant over a step (MV_TYPE=0, LO:29).
    """

    def __init__(self, params: AscentParams, nt: int = 200, nodes: int = 2,
                 time: Optional[Sequence[float]] = None, obj_scale: float = 1.0,
                 objective_nodes: Optional[int] = None):
        self.p = params
        self.nm = _build_node_model(params.model)
        self.time = np.linspace(0.0, 1.0, nt) if time is None else np.asarray(time, float)  # LO:20-21
        self.nt = len(self.time)
        self.nodes = nodes
        self.tau, self.Ncol = collocation_matrix(nodes)
        self.nsteps = self.nt - 1
        self.npts = nodes - 1                      # collocation points per step (excl. left end)
        self.K = self.nsteps * self.npts
        self.nv = len(self.nm.names)
        self.P = _param_vector(params)
        self.obj_scale = obj_scale
        nm = self.nm
        # index helpers
        self.i_tf = self.K * self.nv
        self.i_s1 = self.i_tf + 1
        self.i_s2 = self.i_tf + 2
        self.n = self.i_tf + 3
        # DCOST (LO:99): l1 penalty dcost*|MV_k - MV_{k-1}| per step, written with non-negative
        # slack pairs  MV_k - MV_{k-1} = p_k - n_k  (SURVEY B.3).  APMonitor sums the objective over
        # the horizon (`objective_nodes` copies of tf, default nt-1), so relative to obj_scale*tf
        # the weight per unit of move is obj_scale*dcost/objective_nodes.
        self.dcost = float(params.dcost) if nodes == 2 else 0.0
        self.objective_nodes = (self.nt - 1) if objective_nodes is None else objective_nodes
        self.w_dcost = obj_scale * self.dcost / self.objective_nodes
        self.i_p = self.n
        self.i_n = self.n + (self.K if self.dcost > 0 else 0)
        if self.dcost > 0:
            self.n += 2 * self.K
        self.is_mv = np.zeros(self.nv, bool)
        self.mv_name = "angledoubledot" if params.model == "elliptical" else "angle"
        self.i_mv = nm.names.index(self.mv_name)
        # constraints: per point ndiff + nalg; MV hold rows for NODES>2; 3 terminal
        self.rows_per_pt = nm.ndiff + nm.nalg
        self.m_hold = self.nsteps * (self.npts - 1)
        self.m = self.K * self.rows_per_pt + self.m_hold + 3 + (self.K if self.dcost > 0 else 0)
        # bounds
        lb = np.tile(nm.lb, self.K)
        ub = np.tile(nm.ub, self.K)
        ia = nm.names.index("angle")
        lb[ia::self.nv] = 0.0
        ub[ia::self.nv] = params.angle_ub                                  # LO:94
        if params.model == "elliptical":
            lb[self.i_mv::self.nv] = -params.u_bound                       # LO:96
            ub[self.i_mv::self.nv] = params.u_bound
        self.lb = np.concatenate([lb, [0.0, 0.0, 0.0]])                    # tf LO:39; slacks >= 0
        self.ub = np.concatenate([ub, [1.0, np.inf, np.inf]])
        if self.dcost > 0:
            self.lb = np.concatenate([self.lb, np.zeros(2 * self.K)])
            self.ub = np.concatenate([self.ub, np.full(2 * self.K, np.inf)])
        # step widths per collocation point
        self.h = np.repeat(np.diff(self.time), self.npts)                  # [K]
        self._build_structure()

    # -- helpers ------------------------------------------------------------------------
    def split(self, x):
        v = x[: self.i_tf].reshape(self.K, self.nv).T                      # [nv, K]
        return v, x[self.i_tf], x[self.i_s1], x[self.i_s2]

    def node_values(self, x) -> Dict[str, np.ndarray]:
        """GEKKO-style ``.value`` lists: one value per mesh node (length nt), node 0 = 0."""
        v, tf, _, _ = self.split(x)
        out = {}
        for i, n in enumerate(self.nm.names):
            out[n] = np.concatenate([[0.0], v[i, self.npts - 1:: self.npts]])
        out["tf"] = float(tf)
        return out

    def _build_structure(self):
        nm, K, nv = self.nm, self.K, self.nv
        npts = self.npts
        # predecessor ("x_0" of the step) for each collocation point: index of the point
        # that is the previous mesh node, or -1 for node 0.
        step = np.arange(K) // npts
        self.prev = np.where(step == 0, -1, step * npts - 1)
        self.step = step
        self.within = np.arange(K) % npts

    # -- objective ----------------------------------------------------------------------
    def f(self, x):
        f = self.obj_scale * x[self.i_tf]                                   # LO:176
        if self.dcost > 0:
            f += self.w_dcost * x[self.i_p:].sum()                          # LO:99
        return f

    def grad(self, x):
        g = np.zeros(self.n)
        g[self.i_tf] = self.obj_scale
        if self.dcost > 0:
            g[self.i_p:] = self.w_dcost
        return g

    # -- constraints --------------------------------------------------------------------
    def _terminal(self, v):
        nm, p = self.nm, self.p
        names = nm.names
        y = v[names.index("y"), -1]
        x = v[names.index("x"), -1]
        yd = v[names.index("ydot"), -1]
        xd = v[names.index("xdot"), -1]
        return y, x, yd, xd

    def c(self, x):
        nm, K, nv = self.nm, self.K, self.nv
        v, tf, s1, s2 = self.split(x)
        F = nm.rhs(v, tf, self.P)                                          # [ndiff, K]
        A = nm.alg(v, self.P)                                              # [nalg, K]
        vd = v[nm.diff_idx, :]                                             # [ndiff, K]
        v0 = np.where(self.prev[None, :] >= 0, vd[:, np.maximum(self.prev, 0)], 0.0)
        # collocation rows:  x_i - x_0 - h * sum_j N_ij f_j = 0   (i within the same step)
        Fs = F.reshape(nm.ndiff, self.nsteps, self.npts)
        NF = np.einsum("ij,dsj->dsi", self.Ncol, Fs).reshape(nm.ndiff, K)
        defect = vd - v0 - self.h[None, :] * NF
        rows = np.concatenate([defect, A], axis=0).T.reshape(-1)          # point-major
        out = [rows]
        if self.m_hold:
            mv = v[self.i_mv].reshape(self.nsteps, self.npts)
            out.append((mv[:, :-1] - mv[:, -1:]).reshape(-1))             # ZOH over the step
        p = self.p
        y, xx, yd, xd = self._terminal(v)
        S, R0 = p.S, p.R0
        t1 = math.sqrt((y + R0 / S) ** 2 + xx ** 2) - (R0 + S) / S - s1    # LO:161 (>= -> slack)
        t2 = xd ** 2 + yd ** 2 - (p.v_target / S) ** 2 - s2                # LO:169
        t3 = (y + R0 / S) * yd + xx * xd                                   # LO:173 divided by S^2
        out.append(np.array([t1, t2, t3]))
        if self.dcost > 0:
            mv = v[self.i_mv]
            dmv = np.diff(np.concatenate([[0.0], mv]))                     # MV(0) = 0 (pinned)
            out.append(dmv - x[self.i_p:self.i_p + K] + x[self.i_n:self.i_n + K])
        return np.concatenate(out)

    def jac(self, x) -> sp.csr_matrix:
        nm, K, nv = self.nm, self.K, self.nv
        nd, na, rp = nm.ndiff, nm.nalg, self.rows_per_pt
        v, tf, s1, s2 = self.split(x)
        FJ = nm.rhs_jac(v, tf, self.P)                                     # [nd, nv+1, K]
        AJ = nm.alg_jac(v, self.P)                                         # [na, nv, K]
        rows, cols, vals = [], [], []
        k = np.arange(K)
        # d defect_i(point k) / d v(point k') for k' in same step: -h N[w(k), w(k')] * FJ(k')
        for wi in range(self.npts):
            for wj in range(self.npts):
                kk = k[self.within == wi]                                  # row points
                kj = kk - wi + wj                                          # column points
                coef = -self.h[kk] * self.Ncol[wi, wj]
                for d in range(nd):
                    for j in range(nv):
                        rows.append(kk * rp + d)
                        cols.append(kj * nv + j)
                        vals.append(coef * FJ[d, j, kj])
                    rows.append(kk * rp + d)
                    cols.append(np.full(len(kk), self.i_tf))
                    vals.append(coef * FJ[d, nv, kj])
        for d in range(nd):
            rows.append(k * rp + d)
            cols.append(k * nv + nm.diff_idx[d])
            vals.append(np.ones(K))
            has = self.prev >= 0
            rows.append(k[has] * rp + d)
            cols.append(self.prev[has] * nv + nm.diff_idx[d])
            vals.append(-np.ones(has.sum()))
        for a in range(na):
            for j in range(nv):
                rows.append(k * rp + nd + a)
                cols.append(k * nv + j)
                vals.append(AJ[a, j, :])
        r0 = K * rp
        if self.m_hold:
            idx = 0
            for s in range(self.nsteps):
                for w in range(self.npts - 1):
                    rows.append(np.array([r0 + idx, r0 + idx]))
                    cols.append(np.array([(s * self.npts + w) * nv + self.i_mv,
                                          (s * self.npts + self.npts - 1) * nv + self.i_mv]))
                    vals.append(np.array([1.0, -1.0]))
                    idx += 1
            r0 += self.m_hold
        p = self.p
        names = nm.names
        last = (K - 1) * nv
        iy, ix, iyd, ixd = (last + names.index(n) for n in ("y", "x", "ydot", "xdot"))
        y, xx, yd, xd = self._terminal(v)
        Yb = y + p.R0 / p.S
        r = math.sqrt(Yb ** 2 + xx ** 2)
        trip = [(r0, iy, Yb / r), (r0, ix, xx / r), (r0, self.i_s1, -1.0),
                (r0 + 1, iyd, 2 * yd), (r0 + 1, ixd, 2 * xd), (r0 + 1, self.i_s2, -1.0),
                (r0 + 2, iy, yd), (r0 + 2, iyd, Yb), (r0 + 2, ix, xd), (r0 + 2, ixd, xx)]
        for (r_, c_, v_) in trip:
            rows.append(np.array([r_]))
            cols.append(np.array([c_]))
            vals.append(np.array([v_]))
        if self.dcost > 0:
            rd = r0 + 3 + k
            rows += [rd, rd[1:], rd, rd]
            cols += [k * nv + self.i_mv, k[:-1] * nv + self.i_mv, self.i_p + k, self.i_n + k]
            vals += [np.ones(K), -np.ones(K - 1), -np.ones(K), np.ones(K)]
        R = np.concatenate([np.asarray(a).ravel() for a in rows])
        C = np.concatenate([np.asarray(a).ravel() for a in cols])
        Vv = np.concatenate([np.asarray(a, float).ravel() for a in vals])
        return sp.csr_matrix((Vv, (R, C)), shape=(self.m, self.n))

    def hess(self, x, lam) -> sp.csr_matrix:
        """Hessian of  f + lam^T c  (objective is linear, so only constraints contribute)."""
        nm, K, nv = self.nm, self.K, self.nv
        nd, na, rp = nm.ndiff, nm.nalg, self.rows_per_pt
        v, tf, s1, s2 = self.split(x)
        L = lam[: K * rp].reshape(K, rp).T                                 # [rp, K]
        Ld = L[:nd].reshape(nd, self.nsteps, self.npts)
        # weight on F(point j) = -h * sum_i N[i,j] * lam_i   (same step)
        Wr = (-np.einsum("ij,dsi->dsj", self.Ncol, Ld)).reshape(nd, K) * self.h[None, :]
        HR = nm.rhs_hess(v, tf, self.P, Wr)                                # [nv+1, nv+1, K]
        HA = nm.alg_hess(v, self.P, L[nd:])                                # [nv, nv, K]
        rows, cols, vals = [], [], []
        k = np.arange(K)
        for i in range(nv):
            for j in range(nv):
                rows.append(k * nv + i)
                cols.append(k * nv + j)
                vals.append(HR[i, j] + HA[i, j])
            rows.append(k * nv + i)
            cols.append(np.full(K, self.i_tf))
            vals.append(HR[i, nv])
            rows.append(np.full(K, self.i_tf))
            cols.append(k * nv + i)
            vals.append(HR[nv, i])
        rows.append(np.full(K, self.i_tf))
        cols.append(np.full(K, self.i_tf))
        vals.append(HR[nv, nv])
        # terminal rows
        p, names = self.p, nm.names
        r0 = K * rp + self.m_hold
        l1, l2, l3 = lam[r0], lam[r0 + 1], lam[r0 + 2]
        last = (K - 1) * nv
        iy, ix, iyd, ixd = (last + names.index(n) for n in ("y", "x", "ydot", "xdot"))
        y, xx, yd, xd = self._terminal(v)
        Yb = y + p.R0 / p.S
        r = math.sqrt(Yb ** 2 + xx ** 2)
        trip = [(iy, iy, l1 * xx * xx / r ** 3), (ix, ix, l1 * Yb * Yb / r ** 3),
                (iy, ix, -l1 * Yb * xx / r ** 3), (ix, iy, -l1 * Yb * xx / r ** 3),
                (iyd, iyd, 2 * l2), (ixd, ixd, 2 * l2),
                (iy, iyd, l3), (iyd, iy, l3), (ix, ixd, l3), (ixd, ix, l3)]
        for (r_, c_, v_) in trip:
            rows.append(np.array([r_]))
            cols.append(np.array([c_]))
            vals.append(np.array([v_]))
        R = np.concatenate([np.asarray(a).ravel() for a in rows])
        C = np.concatenate([np.asarray(a).ravel() for a in cols])
        Vv = np.concatenate([np.asarray(a, float).ravel() for a in vals])
        return sp.csr_matrix((Vv, (R, C)), shape=(self.n, self.n))

    # -- initial guess ------------------------------------------------------------------
    def initial_guess(self, tf0: float = 0.9) -> np.ndarray:
        """Start point.  ``tf0=None`` gives the reference's all-zero cold start (LO:39,
        83-96), which needs IPOPT's full restoration phase.  Otherwise: a dynamically
        consistent roll-out of a bang-bang pitch-acceleration profile (+0.9 until t1, -0.9
        until t1+t2, then 0), the shape of Angle_vs_Time.png.  The product builds the same
        start on the device (csrc/ascent_ipm.cuh: start_rollout) -- restated here, not shared."""
        nm, p, K, nv = self.nm, self.p, self.K, self.nv
        x = np.zeros(self.n)
        if tf0 is None:
            return x
        tf0 = min(max(tf0, 1e-2), 0.99)
        names = nm.names
        tau_pts = np.empty(K)
        for k in range(K):
            s, w = divmod(k, self.npts)
            tau_pts[k] = self.time[s] + (self.time[s + 1] - self.time[s]) * self.tau[w + 1]
        t = np.concatenate([[0.0], tau_pts]) * tf0 * p.final_time
        v = np.zeros((nv, K))
        if p.model == "elliptical":
            a_tgt = min(0.40, 0.8 * p.angle_ub)
            w_rem = 3.5e-4
            ulev = 0.9 * p.u_bound
            ueff = ulev * p.asc
            t1 = math.sqrt(a_tgt / ueff)
            t2 = max(t1 - w_rem / ueff, 0.0)
        a = w = 0.0
        y = yd = xx = xd = 0.0
        a_lo, a_hi = 1e-2 * p.angle_ub, 0.99 * p.angle_ub
        for k in range(1, K + 1):
            dt = t[k] - t[k - 1]
            tm = 0.5 * (t[k] + t[k - 1])
            if p.model == "elliptical":
                u = ulev if tm < t1 else (-ulev if tm < t1 + t2 else 0.0)
                w += dt * p.asc * u
                a += dt * w
            else:   # circular: the pitch itself is the MV; ramp to ~35 deg then rise linearly
                a = (0.2 + 0.45 * t[k] / t[-1])
            ac = min(max(a, a_lo), a_hi)
            m = p.mflow * t[k]
            yn, xn, ydn, xdn = y + dt * yd, xx + dt * xd, yd, xd
            for _ in range(3):
                ydd, xdd = _accel_numeric(p, yn, xn, ac, m)
                ydn, xdn = yd + dt * ydd, xd + dt * xdd
                yn, xn = y + dt * ydn, xx + dt * xdn
            y, yd, xx, xd = yn, ydn, xn, xdn
            col = k - 1
            v[names.index("y"), col] = y
            v[names.index("ydot"), col] = yd
            v[names.index("x"), col] = xx
            v[names.index("xdot"), col] = xd
            v[names.index("ydoubledot"), col] = ydd
            v[names.index("xdoubledot"), col] = xdd
            v[names.index("mass"), col] = min(m, 0.99)
            v[names.index("angle"), col] = ac
            if p.model == "elliptical":
                v[names.index("angledot"), col] = w
                v[names.index("angledoubledot"), col] = u
        x[: self.i_tf] = v.T.reshape(-1)
        x[self.i_tf] = tf0
        x[self.i_s1] = 1e-2
        x[self.i_s2] = 1e-2
        if self.dcost > 0:
            mv = v[self.i_mv]
            dmv = np.diff(np.concatenate([[0.0], mv]))
            x[self.i_p:self.i_p + K] = np.maximum(dmv, 0.0) + 1e-2
            x[self.i_n:self.i_n + K] = np.maximum(-dmv, 0.0) + 1e-2
        return x


def _accel_numeric(p: AscentParams, y, x, a, m):
    """LO:127-136 evaluated numerically (scaled units)."""
    S, R0, GM = p.S, p.R0, p.GM
    X, Y = x * S, y * S + R0
    r = math.hypot(X, Y)
    kk = p.Ft / ((p.M0 - p.mscale * m) * r)
    c3, s3 = math.cos(3 * a), math.sin(3 * a)
    ydd = (kk * (Y * c3 + X * s3) - Y * GM / r ** 3) / S
    xdd = (kk * (X * c3 - Y * s3) - X * GM / r ** 3) / S
    return ydd, xdd
