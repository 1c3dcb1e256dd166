"""The direct KKT solver (csrc/direct.cuh) on the BASELINE configs C1, C3 (full size) and C2: factor size, assembly and
factorisation time, the KKT phase per ADMM iteration, ADMM iterations/s of the direct and the CG path measured in the
same process (alternated), and parity of w after the same iterations against an exact host solve of the same reduced
system.  One JSON line per config.  Usage: python tests/run_direct_kkt.py [c1] [c3] [c2]"""
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import scipy.linalg as la
import scipy.sparse as sp

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cosmo_b200
from oracle import cosmo_oracle as O
from oracle.bridge import to_oracle_cones

NB = 64


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def create_model(P, q, A, b, sets, st):
    """Model with its engine created; the engine's '[direct]' stderr line (COSMO_B200_SETUP_DEBUG) carries the
    event-timed assembly and factorisation of the initial factorisation."""
    model = cosmo_b200.Model()
    model.set(P, q, A, b, sets, st)
    os.environ["COSMO_B200_SETUP_DEBUG"] = "1"
    saved = os.dup(2)
    with tempfile.TemporaryFile() as f:
        os.dup2(f.fileno(), 2)
        try:
            model._setup()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["COSMO_B200_SETUP_DEBUG"]
        f.seek(0)
        log = f.read().decode(errors="replace")
    m = re.search(r"\[direct\] .*assembly ([0-9.]+) ms factorisation ([0-9.]+) ms", log)
    return model, (float(m.group(1)), float(m.group(2))) if m else (None, None)


def run_iters(model):
    model.engine.reset()
    model.engine.warm_start(np.zeros(model.n), np.zeros(model.m), np.zeros(model.m))
    if model.settings.kkt_solver == "DirectReducedKKTSolver":
        model.engine.kkt_solve(np.zeros(model.n + model.m))   # the reset marked the factor stale: refactor outside the timing
    out = model.engine.solve()
    return out


class DenseCholKKT:
    """Exact host solve of the reduced system through LAPACK (cho_factor of the dense M = P + sigma I + A'RA), for sizes
    where the oracle's sparse LU of the full KKT matrix is impractical."""

    def __init__(self, P, A, sigma, rho):
        self.P, self.A, self.sigma = sp.csr_matrix(P), sp.csr_matrix(A), sigma
        self.m, self.n = A.shape
        self.multiplications = []
        self.update_rho(rho)

    def update_rho(self, rho):
        self.rho = np.broadcast_to(np.asarray(rho, dtype=float), (self.m,)).copy()
        nnz = np.diff(self.A.indptr)
        dense = (nnz >= 64) & (8 * nnz >= self.n)
        Gd = (np.sqrt(self.rho[dense])[:, None] * self.A[dense].toarray())
        As = self.A[~dense]
        M = Gd.T @ Gd
        M += (As.T @ sp.diags(self.rho[~dense]) @ As + self.P).toarray()
        M[np.diag_indices(self.n)] += self.sigma
        self.c = la.cho_factor(M, lower=True, overwrite_a=True)

    def solve(self, rhs):
        x1, x2 = rhs[:self.n], rhs[self.n:]
        y1 = la.cho_solve(self.c, x1 + self.A.T @ (self.rho * x2))
        return np.concatenate([y1, self.rho * (self.A @ y1 - x2)])


def measure(name, P, q, A, b, sets, iters, reps, parity_iters, host_kkt):
    n, m = A.shape[1], A.shape[0]
    NT = -(-n // NB)
    base = dict(scaling=0, adaptive_rho=False, eps_abs=0.0, eps_rel=0.0, max_iter=iters, verbose_timing=True)
    line = {"config": name, "gpu": gpu_info(), "n": n, "m": m, "nnz_A": int(A.nnz), "factor_bytes": NT * (NT + 1) // 2 * NB * NB * 8}
    try:
        direct, (asm_ms, fac_ms) = create_model(P, q, A, b, sets, cosmo_b200.Settings(kkt_solver="DirectReducedKKTSolver", **base))
    except cosmo_b200.EngineError as e:
        line["direct"] = "refused: %s" % e
        print(json.dumps(line), flush=True)
        return
    cg, _ = create_model(P, q, A, b, sets, cosmo_b200.Settings(**base))
    line.update({"assembly_ms": asm_ms, "factorization_ms": fac_ms,
                 "factorization_tflops": (n ** 3 / 3.0) / (fac_ms * 1e-3) / 1e12 if fac_ms else None})
    rates = {"direct": [], "cg": []}
    kkt_ms = []
    for _ in range(reps):                         # alternated in the same process
        for key, model in (("direct", direct), ("cg", cg)):
            out = run_iters(model)
            rates[key].append(out.iter / out.times["iter_time_device"])
            if key == "direct":
                kkt_ms.append(1e3 * out.times["kkt_time"] / out.iter)
    line["direct_iter_per_s"] = rates["direct"]
    line["cg_iter_per_s"] = rates["cg"]
    line["speedup_direct_over_cg"] = float(np.median(rates["direct"]) / np.median(rates["cg"]))
    # kkt_time covers the rhs SpMV, both sweeps and the fused ADMM tail: an upper bound of the solve's time, so the rate
    # below is a lower bound of the sweeps' achieved bandwidth (they read the factor twice)
    line["kkt_phase_ms_per_iter"] = float(np.median(kkt_ms))
    line["sweeps_gbs_lower_bound"] = 2 * line["factor_bytes"] / (line["kkt_phase_ms_per_iter"] * 1e-3) / 1e9
    line["factor_stats"] = direct.engine.kkt_factor_stats()
    if host_kkt is not None:
        st = cosmo_b200.Settings(kkt_solver="DirectReducedKKTSolver", **dict(base, max_iter=parity_iters)).to_struct()
        direct.engine.update_settings(st)
        run_iters(direct)
        w = direct.engine.w()
        ost = dict(scaling=0, adaptive_rho=False, eps_abs=0.0, eps_rel=0.0, max_iter=parity_iters)
        saved = O.make_kkt_solver
        if host_kkt == "dense_cholesky":
            O.make_kkt_solver = lambda kind, P_, A_, sigma, rho, st_: DenseCholKKT(P_, A_, sigma, rho)
        try:
            ref = O.solve(P, q, A, b, to_oracle_cones(sets), O.Settings(**ost))
        finally:
            O.make_kkt_solver = saved
        line["parity_iters"] = parity_iters
        line["parity_host_solver"] = "oracle DirectKKT (sparse LU)" if host_kkt == "oracle" else "LAPACK cho_factor of dense M"
        line["parity_w_rel"] = float(np.max(np.abs(w - ref.w)) / max(np.max(np.abs(ref.w)), 1e-300))
    print(json.dumps(line), flush=True)
    direct.engine.close()
    cg.engine.close()


def main():
    which = sys.argv[1:] or ["c1", "c3", "c2"]
    pr = cosmo_b200.problems
    if "c1" in which:
        P = sp.csc_matrix(np.array([[4.0, 1.0], [1.0, 2.0]]))
        q = np.array([1.0, 1.0])
        Am = np.array([[1.0, 1.0], [1.0, 0.0], [0.0, 1.0]])
        A = sp.csc_matrix(np.vstack([Am, -Am]))          # model form of examples/qp.jl:19-21 (A = -Aa)
        b = np.array([1.0, 0.7, 0.7, -1.0, 0.0, 0.0])
        measure("C1 examples/qp.jl (n=2, m=6)", P, q, A, b, [cosmo_b200.Nonnegatives(6)], 2000, 3, 375, "oracle")
    if "c3" in which:
        P, q, A, b, sets = pr.portfolio_socp(n=20_000, k=2_000, seed=1)
        measure("C3 portfolio SOCP n=20000 k=2000", P, q, A, b, sets, 50, 3, 20, "dense_cholesky")
    if "c2" in which:
        P, q, A, b, sets = pr.random_sparse_qp(n=50_000, m=100_000, density=0.01, seed=2)
        measure("C2 random sparse QP n=50000 m=100000", P, q, A, b, sets, 20, 2, 0, None)


if __name__ == "__main__":
    main()
