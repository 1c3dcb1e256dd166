"""CPU checks of the direct KKT solver: the settings mapping, the C header's enum value, and a NumPy model of the device
algorithm of csrc/direct.cuh (tile order, padding, assembly split, right-looking tile Cholesky, both sweeps) against
LAPACK on random SPD problems with ragged n."""
import os
import re

import numpy as np
import pytest
import scipy.linalg as la
import scipy.sparse as sp

import cosmo_b200
from cosmo_b200 import engine as E

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NB = 64


def test_settings_mapping_and_header_enum():
    st = cosmo_b200.Settings(kkt_solver="DirectReducedKKTSolver").to_struct()
    assert st.kkt_solver == E.KKT_DIRECT == 3
    src = open(os.path.join(ROOT, "include", "cosmo_b200.h")).read()
    assert int(re.search(r"COSMO_B200_KKT_DIRECT\s*=\s*(\d+)", src).group(1)) == E.KKT_DIRECT
    assert "cosmo_b200_kkt_factor_stats" in E.EXPORTS
    with pytest.raises(E.EngineError) as ei:     # the CPU plugins' names stay refused and point to the device solver
        cosmo_b200.Settings(kkt_solver="CholmodKKTSolver").to_struct()
    assert "DirectReducedKKTSolver" in str(ei.value)


# ---- NumPy restatement of direct.cuh ------------------------------------------------------------------------------
def dense_row(nnz_row, n):
    return nnz_row >= 64 and 8 * nnz_row >= n


class TileFactor:
    """Lower tiles (I, J), I >= J, of side NB; n padded with a unit diagonal."""

    def __init__(self, n):
        self.n = n
        self.NT = max(1, -(-n // NB))
        self.t = {(I, J): np.zeros((NB, NB)) for I in range(self.NT) for J in range(I + 1)}

    def add(self, r, c, v):
        self.t[(r // NB, c // NB)][r % NB, c % NB] += v

    def dense_lower(self):
        N = self.NT * NB
        L = np.zeros((N, N))
        for (I, J), T in self.t.items():
            L[I * NB:(I + 1) * NB, J * NB:(J + 1) * NB] = T
        return np.tril(L)


def assemble(P, A, rho, sigma):
    """assemble_sparse_kernel + gather_dense_kernel + tile_update_kernel<true>."""
    m, n = A.shape
    Ar, Atr, Pr = sp.csr_matrix(A), sp.csr_matrix(A.T), sp.csr_matrix(P)
    for M in (Ar, Atr, Pr):
        M.sort_indices()
    F = TileFactor(n)
    dense = np.array([dense_row(Ar.indptr[i + 1] - Ar.indptr[i], n) for i in range(m)], dtype=bool)
    for r in range(F.NT * NB):
        if r >= n:
            F.add(r, r, 1.0)
            continue
        F.add(r, r, sigma)
        for k in range(Pr.indptr[r], Pr.indptr[r + 1]):
            if Pr.indices[k] <= r:
                F.add(r, Pr.indices[k], Pr.data[k])
        for k in range(Atr.indptr[r], Atr.indptr[r + 1]):        # rows i of A in ascending order
            i = Atr.indices[k]
            if dense[i]:
                continue
            w = rho[i] * Atr.data[k]
            for kk in range(Ar.indptr[i], Ar.indptr[i + 1]):
                if Ar.indices[kk] > r:
                    break
                F.add(r, Ar.indices[kk], w * Ar.data[kk])
    rows = np.nonzero(dense)[0]
    if rows.size:
        ldg = -(-rows.size // NB) * NB
        Gt = np.zeros((F.NT * NB, ldg))
        Gt[:n, :rows.size] = (np.sqrt(rho[rows])[:, None] * Ar[rows].toarray()).T
        for I in range(F.NT):
            for J in range(I + 1):
                F.t[(I, J)] += sum(Gt[I * NB:(I + 1) * NB, k:k + NB] @ Gt[J * NB:(J + 1) * NB, k:k + NB].T
                                   for k in range(0, ldg, NB))
    return F, int(rows.size)


def factor(F):
    """panel_kernel (POTRF + TRSM) and tile_update_kernel<false>, tile column by tile column."""
    for K in range(F.NT):
        D = F.t[(K, K)]
        if np.any(np.linalg.eigvalsh(np.tril(D) + np.tril(D, -1).T) <= 0):
            raise ValueError("Objective function is not convex.")
        Lkk = np.linalg.cholesky(np.tril(D) + np.tril(D, -1).T)
        F.t[(K, K)] = Lkk
        for I in range(K + 1, F.NT):
            F.t[(I, K)] = la.solve_triangular(Lkk, F.t[(I, K)].T, lower=True).T
        for I in range(K + 1, F.NT):
            for J in range(K + 1, I + 1):
                F.t[(I, J)] -= F.t[(I, K)] @ F.t[(J, K)].T
    return F


def sweeps(F, b):
    """trsv_persistent_kernel: forward by tile rows, backward by tile columns."""
    NT, n = F.NT, F.n
    acc = np.zeros(NT * NB)
    acc[:n] = b
    acc = acc.reshape(NT, NB)
    y = np.zeros_like(acc)
    for J in range(NT):
        y[J] = la.solve_triangular(F.t[(J, J)], acc[J], lower=True)
        for I in range(J + 1, NT):
            acc[I] -= F.t[(I, J)] @ y[J]
    acc = y.copy()
    x = np.zeros_like(acc)
    for I in range(NT - 1, -1, -1):
        x[I] = la.solve_triangular(F.t[(I, I)], acc[I], lower=True, trans="T")
        for J in range(I):
            acc[J] -= F.t[(I, J)].T @ x[I]
    return x.ravel()[:n]


def _problem(n, seed):
    rng = np.random.default_rng(seed)
    m = n + 7
    rows = []
    for i in range(m):
        k = min(n, [0, 1, 3, n, n // 2 + 1, 2][i % 6])
        row = np.zeros(n)
        row[rng.choice(n, size=k, replace=False)] = rng.standard_normal(k)
        rows.append(row)
    A = sp.csc_matrix(np.array(rows))
    B = sp.random(n, n, density=min(1.0, 3.0 / n), random_state=rng)
    P = ((B + B.T) * 0.1 + sp.identity(n)).tocsc()
    rho = rng.choice([0.1, 100.0, 1e-6], size=m)
    return P, A, rho


@pytest.mark.parametrize("n", [1, 2, NB - 1, NB, NB + 1, 2 * NB + 7, 4 * NB + 3])
def test_tile_cholesky_model_matches_lapack(n):
    P, A, rho = _problem(n, seed=n)
    sigma = 1e-6
    F, nd = assemble(P, A, rho, sigma)
    M = (P + sigma * sp.identity(n) + A.T @ sp.diags(rho) @ A).toarray()
    N = F.NT * NB
    Mpad = np.eye(N)
    Mpad[:n, :n] = M
    assert np.max(np.abs(F.dense_lower() - np.tril(Mpad))) <= 1e-13 * np.abs(Mpad).max()   # summation order only
    if n >= 64:
        assert nd > 0                     # the dense-row panel path ran
    factor(F)
    Lref = la.cho_factor(M, lower=True)[0]
    L = F.dense_lower()
    assert np.max(np.abs(L[:n, :n] - np.tril(Lref))) <= 1e-12 * np.abs(Lref).max()   # measured <= 1e-13 relative
    assert np.allclose(L[n:, n:], np.eye(N - n)) and not np.any(L[n:, :n])
    b = np.random.default_rng(1).standard_normal(n)
    x = sweeps(F, b)
    assert np.linalg.norm(x - la.cho_solve((Lref, True), b)) <= 1e-10 * (1 + np.linalg.norm(x))


def test_not_positive_definite_is_detected():
    P = sp.csc_matrix(np.diag([1.0, -1.0]))
    A = sp.csc_matrix(np.array([[1.0, 0.0]]))
    F, _ = assemble(P, A, np.array([0.1]), 1e-6)
    with pytest.raises(ValueError, match="not convex"):
        factor(F)


def _sweep_schedule(NT, G):
    """The tile-row ownership arithmetic of trsv_persistent_kernel, in C integer division (every operand is >= 0):
    for each CTA g, the (step, row) updates of the forward and the backward sweep in program order, with the acc slot each
    one writes, and the slot each step's owner solves."""
    fwd, bwd, owner_slots = [], [], []
    for g in range(G):
        nrows = (NT - g + G - 1) // G                           # tile rows I = g + G r, r < nrows
        for J in range(NT):
            r0 = (J + 1 - g + G - 1) // G if J + 1 > g else 0   # first owned row > J
            if J % G == g:
                owner_slots.append((J, g, J // G))
            for r in range(r0, nrows):
                fwd.append((g, J, g + G * r, r))                # acc_I -= L(I, J) y_J
        for I in range(NT - 1, -1, -1):
            rl = (I - 1 - g) // G if I - 1 >= g else -1         # last owned row < I
            if I % G == g:
                owner_slots.append((I, g, I // G))
            for r in range(rl, -1, -1):
                bwd.append((g, I, g + G * r, r))                # acc_J -= L(I, J)' x_I
    return fwd, bwd, owner_slots


def test_sweep_ownership_visits_every_tile_once_in_the_order_of_one_row_per_cta():
    """Every sum of the sweeps runs in an order that does not depend on the grid size G: for each tile row the forward
    sweep subtracts L(I, J) y_J for J ascending and the backward sweep L(I, J)' x_I for I descending, whichever CTA owns
    the row and whatever else it owns.  This is why a solve is bitwise the same for every G
    (tests/test_gpu_direct_kkt_edges.py checks that on the device)."""
    for NT in range(1, 61):
        pairs = {(I, J) for I in range(NT) for J in range(I)}
        for G in range(1, NT + 1):
            R = -(-NT // G)                                          # acc slots per CTA (trsv_smem_bytes)
            fwd, bwd, owner_slots = _sweep_schedule(NT, G)
            # each owned row is the CTA's own row of its slot, and the slot fits in acc
            for g, J, I, r in fwd + bwd:
                assert I % G == g and g + G * r == I and 0 <= r < R
            for step, g, slot in owner_slots:
                assert g + G * slot == step and slot < R
            assert sorted(s for s, _, _ in owner_slots) == sorted(list(range(NT)) * 2)   # one owner per step and sweep
            # forward: pairs (row I, column J), J < I; backward: pairs (row J, column I), J < I -- each exactly once
            f = [(I, J) for _, J, I, _ in fwd]
            b = [(I, J) for _, I, J, _ in bwd]
            assert len(f) == len(set(f)) and set(f) == pairs, (NT, G)
            assert len(b) == len(set(b)) and set(b) == pairs, (NT, G)
            # per row: the forward updates in ascending J, the backward ones in descending I
            f_row, b_row = {r: [] for r in range(NT)}, {r: [] for r in range(NT)}
            for I, J in f:
                f_row[I].append(J)
            for I, J in b:
                b_row[J].append(I)
            for row in range(NT):
                assert f_row[row] == list(range(row)) and b_row[row] == list(range(NT - 1, row, -1)), (NT, G, row)
            # the forward prefetch (tile (I0, J), I0 = g + G r0) is the first row of step J the update loop visits, and the
            # backward one (tile (I, J0), J0 = g + G rl) the first of step I
            first_f, first_b = {}, {}
            for g, J, I, _ in fwd:
                first_f.setdefault((g, J), I)
            for g, I, J, _ in bwd:
                first_b.setdefault((g, I), J)
            for g in range(G):
                for step in range(NT):
                    r0 = (step + 1 - g + G - 1) // G if step + 1 > g else 0
                    rl = (step - 1 - g) // G if step - 1 >= g else -1
                    assert first_f.get((g, step), g + G * r0) == g + G * r0
                    assert first_b.get((g, step), g + G * rl) == g + G * rl


def test_dense_row_rule():
    # the portfolio problem's 2000 rows of F' (10 000 entries) and all-ones row go through the panel product at
    # n = 20 000; its identity and diagonal rows, and rows of a few hundred entries at n = 50 000, stay sparse
    assert dense_row(10_000, 20_000) and dense_row(20_000, 20_000)
    assert not dense_row(1, 20_000) and not dense_row(500, 50_000) and not dense_row(63, 64)
