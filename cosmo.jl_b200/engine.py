"""ctypes binding of libcosmo_b200.so (include/cosmo_b200.h).

This is the stub a maintainer would write for any host language: plain
pointers and sizes, no torch types.  The Julia equivalent (``ccall``) is shown
in INTEGRATION.md.  There is no CPU fallback here: if the shared library is
missing or no CUDA device is present every call raises ``EngineError``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import numpy as np

from . import build as _build

OK = 0
ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA, ERR_ALLOC, ERR_NCCL, ERR_NUMERICAL = -1, -2, -3, -4, -5, -6
F64, F32 = 0, 1
ZERO, NONNEG, BOX, SOC, PSD_SQUARE, PSD_TRIANGLE, EXP, DUAL_EXP, POW, DUAL_POW, PSD_TRIANGLE_COMPLEX = range(11)
STATUS = {0: "Undetermined", 1: "Solved", 2: "Max_iter_reached", 3: "Time_limit_reached",
          4: "Primal_infeasible", 5: "Dual_infeasible", 6: "Unsolved"}
KKT_CG, KKT_MINRES_REDUCED, KKT_MINRES, KKT_DIRECT = 0, 1, 2, 3
ACC_EMPTY, ACC_ANDERSON = 0, 1


class EngineError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("cosmo_b200 error %d: %s" % (code, msg))
        self.code = code


class CscStruct(C.Structure):
    _fields_ = [("nrows", C.c_int64), ("ncols", C.c_int64), ("colptr", C.c_void_p), ("rowval", C.c_void_p),
                ("nzval", C.c_void_p)]


class SetStruct(C.Structure):
    _fields_ = [("type", C.c_int32), ("max_iter", C.c_int32), ("dim", C.c_int64), ("l", C.c_void_p), ("u", C.c_void_p),
                ("alpha", C.c_double), ("tol", C.c_double)]


class ProblemStruct(C.Structure):
    _fields_ = [("dtype", C.c_int32), ("index_base", C.c_int32), ("device", C.c_int32), ("flags", C.c_int32),
                ("m", C.c_int64), ("n", C.c_int64), ("P", CscStruct), ("A", CscStruct),
                ("q", C.c_void_p), ("b", C.c_void_p), ("n_sets", C.c_int64), ("sets", C.c_void_p),
                ("D", C.c_void_p), ("Dinv", C.c_void_p), ("E", C.c_void_p), ("Einv", C.c_void_p), ("c", C.c_double)]


class SettingsStruct(C.Structure):
    _fields_ = [("rho", C.c_double), ("sigma", C.c_double), ("alpha", C.c_double),
                ("eps_abs", C.c_double), ("eps_rel", C.c_double), ("eps_prim_inf", C.c_double),
                ("eps_dual_inf", C.c_double),
                ("max_iter", C.c_int64), ("check_termination", C.c_int32), ("check_infeasibility", C.c_int32),
                ("scaling", C.c_int32), ("adaptive_rho", C.c_int32), ("adaptive_rho_interval", C.c_int32),
                ("kkt_solver", C.c_int32),
                ("adaptive_rho_tolerance", C.c_double), ("adaptive_rho_max_adaptions", C.c_int64),
                ("RHO_MIN", C.c_double), ("RHO_MAX", C.c_double), ("RHO_TOL", C.c_double),
                ("RHO_EQ_OVER_RHO_INEQ", C.c_double), ("COSMO_INFTY", C.c_double), ("MIN_SCALING", C.c_double),
                ("time_limit", C.c_double), ("tol_constant", C.c_double), ("tol_exponent", C.c_double),
                ("verbose", C.c_int32), ("psd_max_sweeps", C.c_int32),
                ("accelerator", C.c_int32), ("accelerator_mem", C.c_int32), ("accelerator_min_mem", C.c_int32),
                ("safeguard", C.c_int32), ("safeguard_tol", C.c_double),
                ("adaptive_rho_fraction", C.c_double), ("setup_time", C.c_double), ("MAX_SCALING", C.c_double),
                ("obj_true", C.c_double), ("obj_true_tol", C.c_double)]


class ResultStruct(C.Structure):
    _fields_ = [("x", C.c_void_p), ("s", C.c_void_p), ("mu", C.c_void_p),
                ("obj_val", C.c_double), ("iter", C.c_int64), ("safeguarding_iter", C.c_int64),
                ("status", C.c_int32), ("_pad", C.c_int32),
                ("r_prim", C.c_double), ("r_dual", C.c_double), ("max_norm_prim", C.c_double),
                ("max_norm_dual", C.c_double), ("rho", C.c_double),
                ("rho_updates", C.c_void_p), ("rho_updates_cap", C.c_int64), ("n_rho_updates", C.c_int64),
                ("solver_time", C.c_double), ("setup_time", C.c_double), ("iter_time", C.c_double),
                ("proj_time", C.c_double), ("kkt_time", C.c_double), ("res_time", C.c_double),
                ("iter_time_device", C.c_double),
                ("kkt_inner_iterations", C.c_int64), ("kkt_multiplications", C.c_int64),
                ("kernel_launches", C.c_int64)]


EXPORTS = [
    "cosmo_b200_abi_version", "cosmo_b200_default_settings", "cosmo_b200_create", "cosmo_b200_destroy",
    "cosmo_b200_last_error", "cosmo_b200_update_settings", "cosmo_b200_warm_start", "cosmo_b200_update_qb",
    "cosmo_b200_update_rho", "cosmo_b200_reset", "cosmo_b200_solve", "cosmo_b200_project", "cosmo_b200_kkt_solve",
    "cosmo_b200_residuals", "cosmo_b200_spmv", "cosmo_b200_spmv_bench", "cosmo_b200_get_rho_vec", "cosmo_b200_get_w",
    "cosmo_b200_comm_unique_id", "cosmo_b200_comm_init", "cosmo_b200_comm_p2p_export", "cosmo_b200_comm_p2p_attach",
    "cosmo_b200_tc_gemm_test", "cosmo_b200_psd_stats", "cosmo_b200_get_scaling", "cosmo_b200_kkt_factor_stats",
    "cosmo_b200_kkt_symbolic",
]

_lib = None


def lib_path():
    return _build.LIB


def load_library(rebuild_if_stale=True):
    """dlopen the in-tree shared library (building it with nvcc when stale)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if rebuild_if_stale and (not os.path.exists(path)):
        _build.build()
    if not os.path.exists(path):
        raise EngineError(ERR_CUDA, "libcosmo_b200.so is missing (run `python -c 'import __graft_entry__ as g; g.build()'`)")
    lib = C.CDLL(path)
    vp = C.c_void_p
    lib.cosmo_b200_abi_version.restype = C.c_int
    lib.cosmo_b200_default_settings.argtypes = [C.POINTER(SettingsStruct)]
    lib.cosmo_b200_create.argtypes = [C.POINTER(vp), C.POINTER(ProblemStruct), C.POINTER(SettingsStruct)]
    lib.cosmo_b200_destroy.argtypes = [vp]
    lib.cosmo_b200_destroy.restype = None
    lib.cosmo_b200_last_error.argtypes = [vp]
    lib.cosmo_b200_last_error.restype = C.c_char_p
    lib.cosmo_b200_update_settings.argtypes = [vp, C.POINTER(SettingsStruct)]
    lib.cosmo_b200_warm_start.argtypes = [vp, vp, vp, vp]
    lib.cosmo_b200_update_qb.argtypes = [vp, vp, vp]
    lib.cosmo_b200_update_rho.argtypes = [vp, vp, C.c_double]
    lib.cosmo_b200_reset.argtypes = [vp]
    lib.cosmo_b200_solve.argtypes = [vp, C.POINTER(ResultStruct)]
    lib.cosmo_b200_project.argtypes = [vp, vp, vp]
    lib.cosmo_b200_kkt_solve.argtypes = [vp, vp, vp, C.POINTER(C.c_int64)]
    lib.cosmo_b200_residuals.argtypes = [vp, vp, vp, vp, C.c_int32, C.POINTER(C.c_double)]
    lib.cosmo_b200_spmv.argtypes = [vp, C.c_int32, vp, vp]
    lib.cosmo_b200_spmv_bench.argtypes = [vp, C.c_int32, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.cosmo_b200_get_rho_vec.argtypes = [vp, vp]
    lib.cosmo_b200_get_w.argtypes = [vp, vp]
    lib.cosmo_b200_comm_unique_id.argtypes = [vp]
    lib.cosmo_b200_comm_init.argtypes = [vp, C.c_int32, C.c_int32, vp]
    lib.cosmo_b200_comm_p2p_export.argtypes = [vp, vp]
    lib.cosmo_b200_comm_p2p_attach.argtypes = [vp, vp, C.c_int32]
    lib.cosmo_b200_psd_stats.argtypes = [vp, C.POINTER(C.c_int64)]
    lib.cosmo_b200_get_scaling.argtypes = [vp, vp, vp, C.POINTER(C.c_double)]
    lib.cosmo_b200_kkt_factor_stats.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_double)]
    lib.cosmo_b200_kkt_symbolic.argtypes = [C.POINTER(ProblemStruct), vp, C.POINTER(C.c_int64)]
    lib.cosmo_b200_tc_gemm_test.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, C.c_int32,
                                            C.POINTER(C.c_double), C.POINTER(C.c_double)]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name not in ("cosmo_b200_destroy", "cosmo_b200_last_error"):
            fn.restype = C.c_int
    _lib = lib
    return lib


def default_settings() -> SettingsStruct:
    s = SettingsStruct()
    rc = load_library().cosmo_b200_default_settings(C.byref(s))
    if rc != OK:
        raise EngineError(rc, "default_settings failed")
    return s


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def nccl_unique_id() -> bytes:
    buf = (C.c_char * 128)()
    lib = load_library()
    rc = lib.cosmo_b200_comm_unique_id(C.cast(buf, C.c_void_p))
    if rc != OK:
        raise EngineError(rc, (lib.cosmo_b200_last_error(None) or b"").decode())
    return bytes(buf)


class SolveOutput:
    __slots__ = ("x", "s", "mu", "obj_val", "iter", "safeguarding_iter", "status", "r_prim", "r_dual", "max_norm_prim", "max_norm_dual",
                 "rho", "rho_updates", "times", "kkt_inner_iterations", "kkt_multiplications", "kernel_launches")


class Engine:
    """Owns one ``cosmo_b200_handle`` (one problem resident in HBM on one GPU).

    ``P`` and ``A`` are SciPy CSC matrices (the same three arrays Julia's
    SparseMatrixCSC holds); ``sets`` is a list of ``(type, dim, l, u)`` or, for the
    exponential / power cones, ``(type, 3, None, None, {"alpha": a, "max_iter": k, "tol": t})``.
    """

    def __init__(self, P, q, A, b, sets: Sequence[tuple], settings: Optional[SettingsStruct] = None,
                 D=None, E=None, c: float = 1.0, dtype=np.float64, device: int = 0, julia_indexing: bool = True,
                 equilibrate: bool = False):
        """equilibrate=True: the data are unscaled and settings.scaling != 0 -- the engine runs scale_ruiz! on the
        device (COSMO_B200_PROBLEM_EQUILIBRATE); read D, E, c back with scaling()."""
        import scipy.sparse as sp
        self._lib = load_library()
        self.dtype = np.dtype(dtype)
        if self.dtype not in (np.dtype(np.float64), np.dtype(np.float32)):
            raise EngineError(ERR_UNSUPPORTED, "dtype must be float64 or float32")
        T = self.dtype
        P = sp.csc_matrix(P)
        A = sp.csc_matrix(A)
        P.sort_indices()
        A.sort_indices()
        self.m, self.n = A.shape
        base = 1 if julia_indexing else 0
        keep = []  # keep host arrays alive during create

        def csc(M):
            colptr = np.ascontiguousarray(M.indptr, dtype=np.int64) + base
            rowval = np.ascontiguousarray(M.indices, dtype=np.int64) + base
            nz = np.ascontiguousarray(M.data, dtype=T)
            keep.extend([colptr, rowval, nz])
            return CscStruct(M.shape[0], M.shape[1], _ptr(colptr), _ptr(rowval), _ptr(nz))

        set_arr = (SetStruct * max(len(sets), 1))()
        for i, (typ, dim, l, u, *extra) in enumerate(sets):
            set_arr[i].type = int(typ)
            set_arr[i].dim = int(dim)
            if extra and extra[0]:
                set_arr[i].alpha = float(extra[0].get("alpha", 0.0))
                set_arr[i].max_iter = int(extra[0].get("max_iter", 0))
                set_arr[i].tol = float(extra[0].get("tol", 0.0))
            if l is not None:
                la = np.ascontiguousarray(l, dtype=T)
                ua = np.ascontiguousarray(u, dtype=T)
                keep.extend([la, ua])
                set_arr[i].l = _ptr(la)
                set_arr[i].u = _ptr(ua)
        prob = ProblemStruct()
        prob.dtype = F64 if T == np.float64 else F32
        prob.index_base = base
        prob.device = device
        prob.flags = 1 if equilibrate else 0
        prob.m, prob.n = self.m, self.n
        prob.P, prob.A = csc(P), csc(A)
        qa = np.ascontiguousarray(q, dtype=T)
        ba = np.ascontiguousarray(b, dtype=T)
        keep.extend([qa, ba])
        prob.q, prob.b = _ptr(qa), _ptr(ba)
        prob.n_sets = len(sets)
        prob.sets = C.cast(set_arr, C.c_void_p)
        if D is not None and E is not None:
            Da = np.ascontiguousarray(D, dtype=T)
            Ea = np.ascontiguousarray(E, dtype=T)
            Di = np.ascontiguousarray(1.0 / np.asarray(D, dtype=np.float64), dtype=T)
            Ei = np.ascontiguousarray(1.0 / np.asarray(E, dtype=np.float64), dtype=T)
            keep.extend([Da, Ea, Di, Ei])
            prob.D, prob.Dinv, prob.E, prob.Einv = _ptr(Da), _ptr(Di), _ptr(Ea), _ptr(Ei)
        prob.c = float(c)
        self.settings = settings if settings is not None else default_settings()
        h = C.c_void_p()
        rc = self._lib.cosmo_b200_create(C.byref(h), C.byref(prob), C.byref(self.settings))
        if rc != OK:
            raise EngineError(rc, (self._lib.cosmo_b200_last_error(None) or b"").decode())
        self._h = h
        del keep

    # ---- lifecycle --------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._lib.cosmo_b200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != OK:
            raise EngineError(rc, (self._lib.cosmo_b200_last_error(self._h) or b"").decode())

    def _vec(self, a, size):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dtype=self.dtype)
        if a.shape != (size,):
            raise EngineError(ERR_INVALID, "vector has wrong length")
        return a

    # ---- updates ------------------------------------------------------------
    def update_settings(self, settings: SettingsStruct):
        self.settings = settings
        self._check(self._lib.cosmo_b200_update_settings(self._h, C.byref(settings)))

    def warm_start(self, x=None, s=None, mu=None):
        x, s, mu = self._vec(x, self.n), self._vec(s, self.m), self._vec(mu, self.m)
        self._check(self._lib.cosmo_b200_warm_start(self._h, _ptr(x), _ptr(s), _ptr(mu)))

    def update_qb(self, q=None, b=None):
        q, b = self._vec(q, self.n), self._vec(b, self.m)
        self._check(self._lib.cosmo_b200_update_qb(self._h, _ptr(q), _ptr(b)))

    def update_rho(self, rho_vec, rho):
        rv = self._vec(rho_vec, self.m)
        self._check(self._lib.cosmo_b200_update_rho(self._h, _ptr(rv), float(rho)))

    def reset(self):
        self._check(self._lib.cosmo_b200_reset(self._h))

    def comm_init(self, nranks, rank, unique_id: Optional[bytes]):
        buf = C.create_string_buffer(unique_id, 128) if unique_id is not None else None
        self._check(self._lib.cosmo_b200_comm_init(self._h, nranks, rank, C.cast(buf, C.c_void_p) if buf else None))

    def p2p_export(self) -> bytes:
        buf = (C.c_char * 128)()
        self._check(self._lib.cosmo_b200_comm_p2p_export(self._h, C.cast(buf, C.c_void_p)))
        return bytes(buf)

    def p2p_attach(self, blobs: bytes, nranks: int):
        buf = C.create_string_buffer(blobs, len(blobs))
        self._check(self._lib.cosmo_b200_comm_p2p_attach(self._h, C.cast(buf, C.c_void_p), nranks))

    # ---- the hot loop ----------------------------------------------------------
    def solve(self, out_x=None, out_s=None, out_mu=None) -> SolveOutput:
        """cosmo_b200_solve.  Output buffers may be caller-provided (e.g. pinned)."""
        T = self.dtype
        x = out_x if out_x is not None else np.empty(self.n, dtype=T)
        s = out_s if out_s is not None else np.empty(self.m, dtype=T)
        mu = out_mu if out_mu is not None else np.empty(self.m, dtype=T)
        rho_updates = np.zeros(256, dtype=np.float64)
        r = ResultStruct()
        r.x, r.s, r.mu = _ptr(x), _ptr(s), _ptr(mu)
        r.rho_updates = _ptr(rho_updates)
        r.rho_updates_cap = rho_updates.shape[0]
        self._check(self._lib.cosmo_b200_solve(self._h, C.byref(r)))
        o = SolveOutput()
        o.x, o.s, o.mu = x, s, mu
        o.obj_val, o.iter, o.status = r.obj_val, r.iter, STATUS[r.status]
        o.safeguarding_iter = r.safeguarding_iter
        o.r_prim, o.r_dual, o.max_norm_prim, o.max_norm_dual = r.r_prim, r.r_dual, r.max_norm_prim, r.max_norm_dual
        o.rho = r.rho
        o.rho_updates = rho_updates[:min(r.n_rho_updates, rho_updates.shape[0])].copy()
        o.times = {"solver_time": r.solver_time, "setup_time": r.setup_time, "iter_time": r.iter_time,
                   "proj_time": r.proj_time, "kkt_time": r.kkt_time, "res_time": r.res_time,
                   "iter_time_device": r.iter_time_device}
        o.kkt_inner_iterations, o.kkt_multiplications = r.kkt_inner_iterations, r.kkt_multiplications
        o.kernel_launches = r.kernel_launches
        return o

    # ---- plugin-granularity entry points ------------------------------------
    def project(self, w_s):
        w_s = self._vec(w_s, self.m)
        out = np.empty(self.m, dtype=self.dtype)
        self._check(self._lib.cosmo_b200_project(self._h, _ptr(w_s), _ptr(out)))
        return out

    def kkt_solve(self, rhs):
        rhs = self._vec(rhs, self.n + self.m)
        sol = np.empty(self.n + self.m, dtype=self.dtype)
        inner = C.c_int64(0)
        self._check(self._lib.cosmo_b200_kkt_solve(self._h, _ptr(rhs), _ptr(sol), C.byref(inner)))
        return sol, inner.value

    def residuals(self, x, s, mu, ignore_scaling=False):
        x, s, mu = self._vec(x, self.n), self._vec(s, self.m), self._vec(mu, self.m)
        out = (C.c_double * 5)()
        self._check(self._lib.cosmo_b200_residuals(self._h, _ptr(x), _ptr(s), _ptr(mu), int(ignore_scaling), out))
        return tuple(out)

    def spmv(self, which, x):
        size_in = self.m if which == 1 else self.n
        size_out = self.m if which == 0 else self.n
        x = self._vec(x, size_in)
        y = np.empty(size_out, dtype=self.dtype)
        self._check(self._lib.cosmo_b200_spmv(self._h, which, _ptr(x), _ptr(y)))
        return y

    def spmv_bench(self, which, reps=20):
        ms, nbytes = C.c_double(0), C.c_double(0)
        self._check(self._lib.cosmo_b200_spmv_bench(self._h, which, reps, C.byref(ms), C.byref(nbytes)))
        return ms.value, nbytes.value

    def rho_vec(self):
        out = np.empty(self.m, dtype=self.dtype)
        self._check(self._lib.cosmo_b200_get_rho_vec(self._h, _ptr(out)))
        return out

    def w(self):
        out = np.empty(self.n + self.m, dtype=self.dtype)
        self._check(self._lib.cosmo_b200_get_w(self._h, _ptr(out)))
        return out

    def scaling(self):
        """(D, E, c) as used by the engine (cosmo_b200_get_scaling)."""
        D = np.empty(self.n, dtype=self.dtype)
        E = np.empty(self.m, dtype=self.dtype)
        c = C.c_double(1.0)
        self._check(self._lib.cosmo_b200_get_scaling(self._h, _ptr(D), _ptr(E), C.byref(c)))
        return D.astype(np.float64), E.astype(np.float64), float(c.value)

    def psd_stats(self):
        """Which path projected the large PSD cones so far (cosmo_b200_psd_stats)."""
        out = (C.c_int64 * 8)()
        self._check(self._lib.cosmo_b200_psd_stats(self._h, out))
        keys = ("tc_projections", "tc_fallbacks", "tc_last_steps", "tc_last_checks", "sign_projections", "sign_fallbacks",
                "jacobi_last_sweeps", "tc_slices")
        return dict(zip(keys, [int(v) for v in out]))

    def kkt_factor_stats(self):
        """Factorisations of the direct KKT solver (cosmo_b200_kkt_factor_stats): their count, the device seconds of the
        initial one (init_factor_time) and of all later ones (factor_update_time); zeros on an indirect solver."""
        cnt = C.c_int64(0)
        sec = (C.c_double * 2)()
        self._check(self._lib.cosmo_b200_kkt_factor_stats(self._h, C.byref(cnt), sec))
        return {"factorizations": int(cnt.value), "init_factor_time": float(sec[0]), "factor_update_time": float(sec[1])}


SYMBOLIC_INFO = ("nnz_L", "supernodes", "height", "widest", "largest_front", "factor_bytes", "workspace_bytes", "dense")


def kkt_symbolic(P, A):
    """Symbolic analysis of the full KKT matrix [P + sigma I, A'; A, -R^-1] (cosmo_b200_kkt_symbolic, host only).

    Returns (perm, info): the 0-based elimination order of the n + m nodes (x first, then the rows of A) and a dict
    with the keys of SYMBOLIC_INFO."""
    import scipy.sparse as sp
    lib = load_library()
    P = sp.csc_matrix(P)
    A = sp.csc_matrix(A)
    m, n = A.shape
    keep = []

    def csc(M):
        colptr = np.ascontiguousarray(M.indptr, dtype=np.int64)
        rowval = np.ascontiguousarray(M.indices, dtype=np.int64)
        keep.extend([colptr, rowval])
        return CscStruct(M.shape[0], M.shape[1], _ptr(colptr), _ptr(rowval), None)

    prob = ProblemStruct()
    prob.dtype, prob.index_base, prob.m, prob.n = F64, 0, m, n
    prob.P, prob.A = csc(P), csc(A)
    perm = np.empty(n + m, dtype=np.int64)
    info = (C.c_int64 * 8)()
    rc = lib.cosmo_b200_kkt_symbolic(C.byref(prob), _ptr(perm), info)
    if rc != OK:
        raise EngineError(rc, (lib.cosmo_b200_last_error(None) or b"").decode())
    return perm, dict(zip(SYMBOLIC_INFO, [int(v) for v in info]))


def tc_gemm(A, B, slices=8, groups=0, reps=0):
    """C = A @ B for symmetric commuting fp64 matrices through the int8-sliced tcgen05 product kernel
    (diagnostic entry `cosmo_b200_tc_gemm_test`).  Returns (C, ms_per_product, (|C|_F^2, |I - C|_F^2))."""
    lib = load_library()
    A = np.asfortranarray(A, dtype=np.float64)
    B = np.asfortranarray(B, dtype=np.float64)
    N = A.shape[0]
    assert A.shape == (N, N) and B.shape == (N, N)
    Cm = np.zeros((N, N), dtype=np.float64, order="F")
    ms = C.c_double(0.0)
    fr = (C.c_double * 2)()
    rc = lib.cosmo_b200_tc_gemm_test(N, slices, groups, 0, A.ctypes.data, B.ctypes.data, Cm.ctypes.data, reps,
                                     C.byref(ms), fr)
    if rc != 0:
        raise EngineError(rc, (lib.cosmo_b200_last_error(None) or b"").decode())
    return Cm, ms.value, (fr[0], fr[1])
