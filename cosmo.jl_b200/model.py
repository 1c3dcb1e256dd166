"""Host-side mirror of COSMO.jl's native API for the accelerated path.

Same names, argument meaning and error behaviour as the reference's
``COSMO.Model`` / ``COSMO.Constraint`` / ``assemble!`` / ``optimize!`` /
``warm_start_*!`` / ``update!`` (src/interface.jl, src/constraint.jl,
src/solver.jl:78-203), so that parity tests read like the reference's own.
Everything here is model building and the `setup!` / `reverse_scaling!` glue
that stays on the host in the reference too; the ADMM loop itself is
``cosmo_b200_solve`` in the CUDA library (engine.py).  Julia is not available in
this image, which is why this mirror is Python: INTEGRATION.md shows the
~100-line Julia shim that replaces it in a real deployment.
"""
from __future__ import annotations

import math
import time
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Union

import os

import numpy as np
import scipy.sparse as sp

from . import engine as _eng


# ---------------------------------------------------------------------------
# convex sets (src/convexset.jl)
# ---------------------------------------------------------------------------
class AbstractConvexSet:
    dim: int


class ZeroSet(AbstractConvexSet):
    """COSMO.ZeroSet(dim), convexset.jl:16-23."""
    code = _eng.ZERO

    def __init__(self, dim):
        if dim < 0:
            raise ValueError("dimension must be nonnegative")
        self.dim = int(dim)


class Nonnegatives(AbstractConvexSet):
    """COSMO.Nonnegatives(dim), convexset.jl:52-60."""
    code = _eng.NONNEG

    def __init__(self, dim):
        if dim < 0:
            raise ValueError("dimension must be nonnegative")
        self.dim = int(dim)


class Box(AbstractConvexSet):
    """COSMO.Box(l, u), convexset.jl:803-830."""
    code = _eng.BOX

    def __init__(self, l, u):
        self.l = np.array(l, dtype=np.float64).ravel()
        self.u = np.array(u, dtype=np.float64).ravel()
        if self.l.shape != self.u.shape:
            raise ValueError("bounds must be same length")
        bad = np.nonzero(self.l > self.u)[0]
        if bad.size:
            i = int(bad[0])
            raise ValueError("Box set: inconsistent lower/upper bounds specified at index i = %d: l[i] = %g, u[i] = %g"
                             % (i + 1, self.l[i], self.u[i]))
        self.dim = self.l.shape[0]


class SecondOrderCone(AbstractConvexSet):
    """COSMO.SecondOrderCone(dim), convexset.jl:92-98."""
    code = _eng.SOC

    def __init__(self, dim):
        if dim < 0:
            raise ValueError("dimension must be nonnegative")
        self.dim = int(dim)


class PsdCone(AbstractConvexSet):
    """COSMO.PsdCone(dim): vec of a square matrix, convexset.jl:271-284."""
    code = _eng.PSD_SQUARE

    def __init__(self, dim):
        if dim < 0:
            raise ValueError("dimension must be nonnegative")
        r = math.isqrt(dim)
        if r * r != dim:
            raise ValueError("dimension must be a square")
        self.dim, self.sqrt_dim = int(dim), r


class PsdConeTriangle(AbstractConvexSet):
    """COSMO.PsdConeTriangle(dim): scaled upper triangle, convexset.jl:362-377."""
    code = _eng.PSD_TRIANGLE

    def __init__(self, dim):
        if dim < 0:
            raise ValueError("dimension must be nonnegative")
        self.dim = int(dim)
        self.sqrt_dim = (math.isqrt(1 + 8 * dim) - 1) // 2
        if self.sqrt_dim * (self.sqrt_dim + 1) // 2 != dim:
            raise ValueError("dimension must be N(N+1)/2")


class ComplexPsdConeTriangle(AbstractConvexSet):
    """COSMO.PsdConeTriangle{T, Complex{T}}(dim), dim = N^2: Hermitian PSD matrices, real upper triangle (sqrt 2 scaled
    off the diagonal) followed by the imaginary parts of the strict upper triangle (convexset.jl:344-360)."""
    code = _eng.PSD_TRIANGLE_COMPLEX

    def __init__(self, dim):
        if dim < 0:
            raise ValueError("dimension must be nonnegative")
        self.dim = int(dim)
        self.sqrt_dim = math.isqrt(self.dim)
        if self.sqrt_dim * self.sqrt_dim != self.dim:
            raise ValueError("dimension must be a square")


class ExponentialCone(AbstractConvexSet):
    """COSMO.ExponentialCone(): cl{(x,y,z) | y > 0, y e^(x/y) <= z}, convexset.jl:497-507."""
    code = _eng.EXP
    dim = 3

    def __init__(self, dim=3, MAX_ITERS=100, EXP_TOL=1e-8):
        self.MAX_ITER, self.TOL = int(MAX_ITERS), float(EXP_TOL)


class DualExponentialCone(ExponentialCone):
    """COSMO.DualExponentialCone(), convexset.jl:749-758."""
    code = _eng.DUAL_EXP


class PowerCone(AbstractConvexSet):
    """COSMO.PowerCone(alpha): {(x,y,z) | x^a y^(1-a) >= |z|, x, y >= 0}, convexset.jl:625-636."""
    code = _eng.POW
    dim = 3

    def __init__(self, alpha, MAX_ITERS=20, POW_TOL=1e-8):
        if alpha <= 0 or alpha >= 1:
            raise ValueError("The exponent alpha of the power cone has to be in (0, 1).")
        self.alpha, self.MAX_ITER, self.TOL = float(alpha), int(MAX_ITERS), float(POW_TOL)


class DualPowerCone(PowerCone):
    """COSMO.DualPowerCone(alpha), convexset.jl:765-775."""
    code = _eng.DUAL_POW


# cones whose rows may only be scaled by one common factor (rectify_scaling!, convexset.jl:955-957)
SCALAR_SCALED_CONES = (SecondOrderCone, PsdCone, PsdConeTriangle, ComplexPsdConeTriangle, ExponentialCone, PowerCone)
# cones that cannot be split across ranks
ATOMIC_CONES = SCALAR_SCALED_CONES


def set_tuple(S):
    """The (type, dim, l, u[, params]) tuple `engine.Engine` marshals into a cosmo_b200_set."""
    if isinstance(S, (ExponentialCone, PowerCone)):
        return (S.code, 3, None, None, {"alpha": getattr(S, "alpha", 0.0), "max_iter": S.MAX_ITER, "tol": S.TOL})
    return (S.code, S.dim, getattr(S, "l", None), getattr(S, "u", None))


_SORT = (ZeroSet, Nonnegatives, Box, SecondOrderCone, PsdCone, PsdConeTriangle)


def _sort_sets(C) -> int:
    """sort_sets, interface.jl:466-475."""
    for k, T in enumerate(_SORT):
        if isinstance(C, T):
            return k + 1
    return 6


# ---------------------------------------------------------------------------
# Constraint (src/constraint.jl:47-108)
# ---------------------------------------------------------------------------
class Constraint:
    """``COSMO.Constraint(A, b, convex_set, dim=0, indices=None)``: A x + b in convex_set."""

    def __init__(self, A, b, convex_set, dim: int = 0, indices=None):
        if not sp.issparse(A):
            A = np.asarray(A, dtype=np.float64)
            if A.ndim == 0:
                A = A.reshape(1, 1)
            elif A.ndim == 1:
                A = A.reshape(-1, 1)
        A = sp.csr_matrix(A, dtype=np.float64)
        b = np.atleast_1d(np.asarray(b, dtype=np.float64)).ravel()
        if isinstance(convex_set, type):  # set passed as a type, constraint.jl:84-108
            if issubclass(convex_set, Box):
                raise ValueError("You can't create a constraint by passing the convex set as a type, if your "
                                 "convex set is a Box. Please pass an object.")
            convex_set = convex_set(A.shape[0])
        if A.shape[0] != b.shape[0]:
            raise ValueError("The dimensions of matrix A and vector b don't match.")
        if A.shape[0] != convex_set.dim:
            raise ValueError("The row dimension of A doesn't match the dimension of the constraint set.")
        if indices is not None:  # constraint.jl:66-72; (start, stop) 1-based inclusive like Julia's start:stop
            start, stop = int(indices[0]), int(indices[-1])
            if start < 1 or stop < start:
                raise ValueError("The index range for x has to be increasing and nonnegative.")
            if dim < stop:
                raise ValueError("The dimension of x must be equal or higher than the stop value of indices.")
            Ac = sp.lil_matrix((A.shape[0], dim))
            Ac[:, start - 1:stop] = A
            A = sp.csr_matrix(Ac)
        self.A, self.b, self.convex_set = A, b, convex_set


# ---------------------------------------------------------------------------
# Settings (src/settings.jl:61-155) and results (src/types.jl:26-112)
# ---------------------------------------------------------------------------
@dataclass
class Settings:
    rho: float = 0.1
    sigma: float = 1e-6
    alpha: float = 1.6
    eps_abs: float = 1e-5
    eps_rel: float = 1e-5
    eps_prim_inf: float = 1e-4
    eps_dual_inf: float = 1e-4
    max_iter: int = 5000
    verbose: bool = False
    verbose_timing: bool = False             # settings.jl:43: here it forces the device phase timers (proj_time, kkt_time)
    kkt_solver: str = "CGIndirectKKTSolver"   # the indirect family, or "DirectReducedKKTSolver" (dense device Cholesky)
    check_termination: int = 25
    check_infeasibility: int = 40
    scaling: int = 10
    MIN_SCALING: float = 1e-4
    MAX_SCALING: float = 1e4
    adaptive_rho: bool = True
    adaptive_rho_interval: int = 40           # 0: automatic (a fraction of the setup time, solver.jl:244-256)
    adaptive_rho_fraction: float = 0.4
    adaptive_rho_tolerance: float = 5.0
    adaptive_rho_max_adaptions: int = 2 ** 62
    RHO_MIN: float = 1e-6
    RHO_MAX: float = 1e6
    RHO_TOL: float = 1e-4
    RHO_EQ_OVER_RHO_INEQ: float = 1e3
    COSMO_INFTY: float = 1e20
    time_limit: float = 0.0
    obj_true: float = float("nan")            # residuals.jl:132-137: |obj_true - cost| <= obj_true_tol joins the convergence test
    obj_true_tol: float = 1e-3
    nearly_ratio: float = 100.0               # only read by is_primal/dual_nearly_feasible (the MOI layer, residuals.jl:119-125)
    tol_constant: float = 1.0
    tol_exponent: float = 1.5
    psd_max_sweeps: int = 30
    # "EmptyAccelerator" | "AndersonAccelerator" (= AndersonAccelerator{T, Type2{QRDecomp}, RestartedMemory,
    # NoRegularizer} with ImmediateActivation, the reference's default family, settings.jl:136-138)
    accelerator: str = "EmptyAccelerator"
    accelerator_mem: int = 15
    accelerator_min_mem: int = 3
    safeguard: bool = True
    safeguard_tol: float = 2.0
    # chordal decomposition of PsdConeTriangle constraints (settings.jl:50-53,129-135; host side, chordal.py).
    # The reference defaults to decompose = true with CliqueGraphMerge; here it is opt-in.
    decompose: bool = False
    merge_strategy: str = "CliqueGraphMerge"   # "NoMerge" | "ParentChildMerge" | "CliqueGraphMerge"
    complete_dual: bool = False
    compact_transformation: bool = True         # the only transformation restated

    _KKT = {"CGIndirectKKTSolver": _eng.KKT_CG, "MINRESIndirectKKTSolver": _eng.KKT_MINRES,
            "IndirectReducedKKTSolver:MINRES": _eng.KKT_MINRES_REDUCED, "DirectReducedKKTSolver": _eng.KKT_DIRECT}

    def to_struct(self) -> "_eng.SettingsStruct":
        if self.kkt_solver not in self._KKT:
            raise _eng.EngineError(_eng.ERR_UNSUPPORTED,
                                   "kkt_solver %r is a direct CPU factorisation; the B200 engine implements "
                                   "CGIndirectKKTSolver / MINRESIndirectKKTSolver, and DirectReducedKKTSolver for an "
                                   "exact solve on the device" % self.kkt_solver)
        if self.accelerator not in ("EmptyAccelerator", "AndersonAccelerator"):
            raise _eng.EngineError(_eng.ERR_UNSUPPORTED,
                                   "accelerator %r: the engine implements EmptyAccelerator and AndersonAccelerator"
                                   "{T, Type2{QRDecomp}, RestartedMemory, NoRegularizer}" % self.accelerator)
        if self.accelerator == "AndersonAccelerator":
            if self.accelerator_mem <= 2:
                raise ValueError("Memory has to be bigger than two.")      # AndersonAccelerator ctor (DomainError)
            if self.accelerator_mem > 32:
                raise _eng.EngineError(_eng.ERR_UNSUPPORTED, "accelerator_mem > 32 is not supported by the device accelerator")
        s = _eng.default_settings()
        for name in ("rho", "sigma", "alpha", "eps_abs", "eps_rel", "eps_prim_inf", "eps_dual_inf", "max_iter",
                     "check_termination", "check_infeasibility", "scaling", "adaptive_rho_interval",
                     "adaptive_rho_tolerance", "adaptive_rho_max_adaptions", "RHO_MIN", "RHO_MAX", "RHO_TOL",
                     "RHO_EQ_OVER_RHO_INEQ", "COSMO_INFTY", "MIN_SCALING", "time_limit", "tol_constant",
                     "tol_exponent", "psd_max_sweeps", "accelerator_mem", "accelerator_min_mem", "safeguard_tol",
                     "adaptive_rho_fraction", "MAX_SCALING", "obj_true", "obj_true_tol"):
            setattr(s, name, getattr(self, name))
        s.adaptive_rho = int(self.adaptive_rho)
        s.verbose = int(bool(self.verbose)) | (2 if self.verbose_timing else 0)
        s.kkt_solver = self._KKT[self.kkt_solver]
        s.accelerator = _eng.ACC_ANDERSON if self.accelerator == "AndersonAccelerator" else _eng.ACC_EMPTY
        s.safeguard = int(self.safeguard)
        return s


@dataclass
class ResultInfo:
    r_prim: float
    r_dual: float
    max_norm_prim: float
    max_norm_dual: float
    rho_updates: List[float]


@dataclass
class Result:
    x: np.ndarray
    y: np.ndarray
    s: np.ndarray
    obj_val: float
    iter: int
    safeguarding_iter: int
    status: str
    info: ResultInfo
    times: dict
    kkt_inner_iterations: int = 0
    kernel_launches: int = 0


# ---------------------------------------------------------------------------
# Ruiz equilibration (src/scaling.jl:21-116) -- host-side setup!, runs once
# ---------------------------------------------------------------------------
def _col_absmax(M: sp.csc_matrix, out: np.ndarray):
    if M.nnz:
        nz = np.diff(M.indptr) > 0
        mx = np.maximum.reduceat(np.abs(M.data), M.indptr[:-1][nz])
        out[nz] = np.maximum(out[nz], mx)
    return out


def _row_absmax(M: sp.csc_matrix, out: np.ndarray):
    if M.nnz:
        np.maximum.at(out, M.indices, np.abs(M.data))
    return out


def _limit(v, lo, hi):
    """limit_scaling!: clip(s, MIN, MAX, one, MAX) (scaling.jl:10-18, algebra.jl:5-7)."""
    return np.where(v < lo, 1.0, np.where(v > hi, hi, v))


def ruiz_equilibrate(P, q, A, b, sets, st: Settings):
    """scale_ruiz! on CSC arrays in place; returns (P, q, A, b, sets, D, E, c)."""
    P = sp.csc_matrix(P, dtype=np.float64, copy=True)
    A = sp.csc_matrix(A, dtype=np.float64, copy=True)
    q = np.array(q, dtype=np.float64)
    b = np.array(b, dtype=np.float64)
    m, n = A.shape
    D, E, c = np.ones(n), np.ones(m), 1.0
    colA = np.repeat(np.arange(n), np.diff(A.indptr))
    colP = np.repeat(np.arange(n), np.diff(P.indptr))

    def scale_data(Ds, Es):
        nonlocal q, b
        P.data *= Ds[P.indices] * Ds[colP]
        A.data *= Es[A.indices] * Ds[colA]
        q = Ds * q
        b = Es * b

    for _ in range(st.scaling):
        Dw = _col_absmax(A, _col_absmax(P, np.zeros(n)))
        Ew = _row_absmax(A, np.zeros(m))
        Dw = 1.0 / np.sqrt(_limit(Dw, st.MIN_SCALING, st.MAX_SCALING))
        Ew = 1.0 / np.sqrt(_limit(Ew, st.MIN_SCALING, st.MAX_SCALING))
        scale_data(Dw, Ew)
        D *= Dw
        E *= Ew
        mean_col_norm_P = float(np.mean(_col_absmax(P, np.zeros(n)))) if n else 0.0
        inf_norm_q = float(np.max(np.abs(q))) if n else 0.0
        if mean_col_norm_P != 0.0 and inf_norm_q != 0.0:
            inf_norm_q = float(_limit(inf_norm_q, st.MIN_SCALING, st.MAX_SCALING))
            scale_cost = float(_limit(max(inf_norm_q, mean_col_norm_P), st.MIN_SCALING, st.MAX_SCALING))
            ctmp = 1.0 / scale_cost
            P.data *= ctmp
            q = q * ctmp
            c *= ctmp
    # cones that only admit a scalar scaling (convexset.jl:905-958, 978-982)
    Ew = np.ones(m)
    changed = False
    off = 0
    for S in sets:
        if isinstance(S, SCALAR_SCALED_CONES) and S.dim > 0:
            seg = slice(off, off + S.dim)
            Ew[seg] = np.mean(E[seg]) / E[seg]
            changed = True
        off += S.dim
    if changed:
        scale_data(np.ones(n), Ew)
        E *= Ew
    new_sets, off = [], 0
    for S in sets:  # scale!(box, e), convexset.jl:863-867
        if isinstance(S, Box):
            e = E[off:off + S.dim]
            new_sets.append(Box(S.l * e, S.u * e))
        else:
            new_sets.append(S)
        off += S.dim
    return P, q, A, b, new_sets, D, E, c


# ---------------------------------------------------------------------------
# Model (COSMO.Model = Workspace, src/types.jl:348-403)
# ---------------------------------------------------------------------------
class Model:
    def __init__(self, dtype=np.float64, device: int = 0):
        self.dtype = np.dtype(dtype)
        self.device = device
        self.is_assembled = False
        self.is_scaled = False
        self.engine: Optional[_eng.Engine] = None
        self.settings = Settings()
        self.times = {}
        self._dec = None          # chordal DecompositionInfo of the problem the engine holds (settings.decompose)
        self._x2 = None           # iterates of the decomposed problem (None: restart from self.x)

    # assemble!(model, P, q, constraints; settings, x0, y0), interface.jl:30-77
    def assemble(self, P, q, constraints: Union[Constraint, Sequence[Constraint]], settings: Optional[Settings] = None,
                 x0=None, y0=None):
        if isinstance(constraints, Constraint):
            constraints = [constraints]
        cons = list(constraints)
        n = int(np.atleast_1d(np.asarray(q)).size)
        # merge_constraints!, interface.jl:411-460
        for T in (ZeroSet, Nonnegatives):
            idx = [i for i, c in enumerate(cons) if type(c.convex_set) is T]
            if len(idx) > 1:
                A = sp.vstack([cons[i].A for i in idx], format="csr")
                b = np.concatenate([cons[i].b for i in idx])
                cons = [c for i, c in enumerate(cons) if i not in idx] + [Constraint(A, b, T(A.shape[0]))]
        cons.sort(key=lambda c: _sort_sets(c.convex_set))
        for c in cons:  # check_A_dim
            if c.A.shape[1] != n:
                raise ValueError("The dimensions of a matrix A (m x %d) in one of the constraints is inconsistent "
                                 "with the dimension of P (%d)." % (c.A.shape[1], n))
        P = sp.csc_matrix(P, dtype=np.float64) if sp.issparse(P) else sp.csc_matrix(np.atleast_2d(np.asarray(P, dtype=np.float64)))
        if P.shape != (n, n):
            raise ValueError("Dimensions of P and q are inconsistent.")
        A = sp.vstack([-c.A for c in cons], format="csc") if cons else sp.csc_matrix((0, n))
        b = np.concatenate([c.b for c in cons]) if cons else np.zeros(0)
        self.set(P, np.asarray(q, dtype=np.float64).ravel(), A, b, [c.convex_set for c in cons], settings)
        if x0 is not None:
            self.warm_start_primal(x0)
        if y0 is not None:
            self.warm_start_dual(y0)

    # set!(model, P, q, A, b, convex_sets, settings), interface.jl:218-250: model form A x + s = b
    def set(self, P, q, A, b, convex_sets: Sequence[AbstractConvexSet], settings: Optional[Settings] = None):
        A = sp.csc_matrix(A, dtype=np.float64)
        P = sp.csc_matrix(P, dtype=np.float64)
        m, n = A.shape
        if sum(S.dim for S in convex_sets) != m:
            raise ValueError("set dimension is not m")
        if P.shape != (n, n) or len(q) != n or len(b) != m:
            raise ValueError("Dimensions of P, q, A, b are inconsistent.")
        self.P0, self.q0, self.A0, self.b0 = P, np.array(q, dtype=np.float64), A, np.array(b, dtype=np.float64)
        self.sets0 = list(convex_sets)
        self.m, self.n = m, n
        if settings is not None:
            self.settings = settings
        self.x = np.zeros(n)
        self.s = np.zeros(m)
        self.mu = np.zeros(m)
        self.is_assembled = True
        self.is_scaled = False
        self._dec = None
        self._x2 = None
        if self.engine is not None:
            self.engine.close()
            self.engine = None

    # warm starts in unscaled coordinates, interface.jl:117-179
    def warm_start_primal(self, x0):
        x0 = np.asarray(x0, dtype=np.float64)
        if x0.shape != (self.n,):
            raise ValueError("Dimension of warm starting vector doesn't match the length of index range ind.")
        self.x[:] = x0
        self.s[:] = self.b0 - self.A0 @ self.x   # s0 = b - A x0 (interface.jl:131-147)
        self._x2 = None                           # a decomposed model restarts from this point (see _setup)

    def warm_start_slack(self, s0):
        self.s[:] = s0
        self._x2 = None

    def warm_start_dual(self, y0):
        y0 = np.asarray(y0, dtype=np.float64)
        if y0.shape != (self.m,):
            raise ValueError("Dimension of warm starting vector doesn't match the length of index range ind.")
        self.mu[:] = -y0
        self._x2 = None

    # update!(model; q, b), interface.jl:187-211
    def update(self, q=None, b=None):
        if not self.is_assembled:
            raise RuntimeError("Model has to be assembled once before one can start updating q or b.")
        if q is not None:
            q = np.asarray(q, dtype=np.float64)
            if q.shape != (self.n,):
                raise ValueError("The dimension of q, does not agree with the model dimension, n.")
            self.q0 = q.copy()
        if b is not None:
            b = np.asarray(b, dtype=np.float64)
            if b.shape != (self.m,):
                raise ValueError("The dimension of b, does not agree with the model dimension, m.")
            self.b0 = b.copy()
        if self.engine is not None and getattr(self, "_dec", None) is not None:
            # the row map of b into the clique blocks is rebuilt with the decomposition at the next optimize! (rho and
            # the iterates of the decomposed problem restart; the reference refuses: "can not be updated if the model
            # has been chordally decomposed before", interface.jl:192,204)
            self._x2 = None
            self.engine.close()
            self.engine = None
        elif self.engine is not None:
            qs = (self.D * self.q0) * self.c if q is not None else None
            bs = self.E * self.b0 if b is not None else None
            self.engine.update_qb(qs, bs)

    # setup! (setup.jl:18-64): scaling + engine creation (the KKT "factorisation" analogue)
    def _setup(self):
        st = self.settings
        t0 = time.perf_counter()
        if self.engine is None:
            # chordal_decomposition!(ws), chordal_decomposition.jl:1-30 (before setup!, solver.jl:88-93)
            self._dec = None
            P0, q0, A0, b0, sets0 = self.P0, self.q0, self.A0, self.b0, self.sets0
            if st.decompose:
                from . import chordal as _chordal
                if not st.compact_transformation:
                    raise _eng.EngineError(_eng.ERR_UNSUPPORTED, "only compact_transformation = true is implemented")
                merge = {"NoMerge": "none", "ParentChildMerge": "parent_child_reference",
                         "CliqueGraphMerge": "clique_graph"}.get(st.merge_strategy)
                if merge is None:
                    raise ValueError("unknown merge_strategy %r" % (st.merge_strategy,))
                P2, q2, A2, b2, sets2, info = _chordal.decompose(P0, q0, A0, b0, sets0, merge=merge)
                if info.blocks:                   # at least one cone was decomposed
                    self._dec = info
                    P0, q0, A0, b0, sets0 = P2, q2, A2, b2, sets2
                    self._x2 = np.concatenate([self.x, np.zeros(A2.shape[1] - self.n)])
                    self._s2, self._mu2 = np.zeros(A2.shape[0]), np.zeros(A2.shape[0])
            m2, n2 = A0.shape
            host_ruiz = os.environ.get("COSMO_B200_HOST_RUIZ") == "1"
            if st.scaling != 0 and host_ruiz:      # the NumPy restatement (kept for the sharded path and as a cross-check)
                P, q, A, b, sets, D, E, c = ruiz_equilibrate(P0, q0, A0, b0, sets0, st)
                self.engine = _eng.Engine(P, q, A, b, [set_tuple(S) for S in sets], st.to_struct(), D=D, E=E, c=c,
                                          dtype=self.dtype, device=self.device)
            else:
                # scale_ruiz! runs on the device (csrc/ruiz.cuh): the engine ingests the unscaled data and hands D, E, c back
                self.engine = _eng.Engine(P0, q0, A0, b0, [set_tuple(S) for S in sets0], st.to_struct(),
                                          dtype=self.dtype, device=self.device, equilibrate=(st.scaling != 0))
                D, E, c = self.engine.scaling() if st.scaling != 0 else (np.ones(n2), np.ones(m2), 1.0)
            self.D, self.E, self.c = D, E, c
        else:
            self.engine.update_settings(st.to_struct())
        # scale_variables! (scaling.jl:118-123)
        if self._dec is not None:
            # The decomposed problem keeps its own iterates between solves.  A warm start given in the ORIGINAL
            # coordinates enters through x only (the clique copies of s and mu start from zero): the reference
            # re-allocates all variables after the decomposition (pre_allocate_variables!, chordal_decomposition.jl:29),
            # i.e. drops the warm start altogether, and cannot re-solve a decomposed model.
            if getattr(self, "_x2", None) is None:
                n2, m2 = len(self.D), len(self.E)
                self._x2 = np.concatenate([self.x, np.zeros(n2 - self.n)])
                self._s2, self._mu2 = np.zeros(m2), np.zeros(m2)
            self.engine.warm_start(self._x2 / self.D, self.E * self._s2, (self._mu2 / self.E) * self.c)
        else:
            self.engine.warm_start(self.x / self.D, self.E * self.s, (self.mu / self.E) * self.c)
        return time.perf_counter() - t0

    # optimize!(model), solver.jl:78-203
    def optimize(self) -> Result:
        if not self.is_assembled:
            raise RuntimeError("The model has to be assembled! / set! before optimize!() can be called.")
        t0 = time.perf_counter()
        setup_time = self._setup()
        if self.settings.time_limit != 0 or (self.settings.adaptive_rho and self.settings.adaptive_rho_interval == 0):
            st = self.settings.to_struct()           # both rules count setup! (solver.jl:119,244-256,349)
            st.setup_time = setup_time
            self.engine.update_settings(st)
        out = self.engine.solve()
        # reverse_scaling! (scaling.jl:170-179)
        x = self.D * out.x.astype(np.float64)
        s = out.s.astype(np.float64) / self.E
        mu = self.E * out.mu.astype(np.float64) / self.c
        if self._dec is not None:   # reverse_decomposition! (+ psd_completion!), chordal_decomposition.jl:129-151
            from . import chordal as _chordal
            self._x2, self._s2, self._mu2 = x.copy(), s.copy(), mu.copy()
            x, s, mu = _chordal.reverse(self._dec, x, s, mu, complete_dual=self.settings.complete_dual)
        self.x, self.s, self.mu = x.copy(), s.copy(), mu.copy()
        times = dict(out.times)
        if self.settings.kkt_solver == "DirectReducedKKTSolver":
            fs = self.engine.kkt_factor_stats()
            times["init_factor_time"], times["factor_update_time"] = fs["init_factor_time"], fs["factor_update_time"]
        times["setup_time"] = setup_time
        times["solver_time"] = time.perf_counter() - t0
        info = ResultInfo(out.r_prim, out.r_dual, out.max_norm_prim, out.max_norm_dual, list(out.rho_updates))
        return Result(x, -mu, s, out.obj_val, out.iter, out.safeguarding_iter, out.status, info, times,
                      kkt_inner_iterations=out.kkt_inner_iterations, kernel_launches=out.kernel_launches)

    def empty_model(self):  # empty_model!, interface.jl:84-100
        if self.engine is not None:
            self.engine.close()
        self.__init__(self.dtype, self.device)


def assemble(model: Model, P, q, constraints, settings: Optional[Settings] = None, x0=None, y0=None):
    """``assemble!(model, P, q, constraints; settings, x0, y0)``."""
    model.assemble(P, q, constraints, settings, x0, y0)


def optimize(model: Model) -> Result:
    """``COSMO.optimize!(model)``."""
    return model.optimize()
