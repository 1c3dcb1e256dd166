"""The direct KKT solver (csrc/direct.cuh) where tests/test_gpu_direct_kkt.py does not reach: sweeps in which one CTA owns
several tile rows (capped grids through COSMO_B200_DIRECT_CTAS, and the natural grid at n > 64 * 2 * SMs), the fp32
model, Ruiz-scaled data, the edges of the assembly split, pivot failures after the first tile column and after a rho
update, duplicate entries, and switching solvers.

Every sum of the sweeps runs in an order that does not depend on the grid size G (tests/test_direct_kkt_cpu.py checks
the ownership arithmetic), so a solve must be bitwise the same for every G: the oracle for the multi-row paths."""
import re

import numpy as np
import pytest
import scipy.linalg as la
import scipy.sparse as sp
import torch

import cosmo_b200
from cosmo_b200 import engine as E
from cosmo_b200 import model as M
from oracle import cosmo_oracle as O
from tests.test_gpu_direct_kkt import DIRECT, NB, _engine, _kkt, _ragged_problem

pytestmark = pytest.mark.gpu

SIGMA = 1e-6
CAP_ENV = "COSMO_B200_DIRECT_CTAS"


def _cap(monkeypatch, cap):
    """The sweep grid of the next engine created: at most `cap` CTAs (None: the engine's own choice)."""
    if cap is None:
        monkeypatch.delenv(CAP_ENV, raising=False)
    else:
        monkeypatch.setenv(CAP_ENV, str(cap))


def _errors(P, A, rho, sols, rhss, ref=None):
    """Worst forward error against the oracle's direct solve (when given) and worst normwise backward error against the
    sparse KKT matrix."""
    K = _kkt(P, A, SIGMA, rho)
    normK = abs(K).sum(axis=1).max()
    fwd = bwd = 0.0
    for sol, rhs in zip(sols, rhss):
        if ref is not None:
            want = ref.solve(rhs)
            fwd = max(fwd, np.linalg.norm(sol - want) / (1 + np.linalg.norm(want)))
        bwd = max(bwd, np.abs(K @ sol - rhs).max() / (normK * np.abs(sol).max() + np.abs(rhs).max()))
    return fwd, bwd


def _solve_all(eng, rhss):
    out = []
    for rhs in rhss:
        sol, inner = eng.kkt_solve(rhs)
        assert inner == 0
        out.append(sol)
    return out


def _check(P, A, eng, rhss, label, ref=None):
    """Solve every rhs; forward error <= 1e-10 against the oracle, backward error <= 1e-13."""
    rho = eng.rho_vec().astype(np.float64)
    sols = _solve_all(eng, rhss)
    fwd, bwd = _errors(P, A, rho, sols, rhss, ref if ref is not None else O.DirectKKT(P, A, SIGMA, rho))
    print("%s: forward %.2e backward %.2e" % (label, fwd, bwd))
    assert fwd <= 1e-10 and bwd <= 1e-13, (label, fwd, bwd)
    return sols


def _rhss(n, m, seed, k=3):
    rng = np.random.default_rng(seed)
    return [rng.standard_normal(n + m) for _ in range(k)]


# ---- grid invariance ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [NB + 1, 3 * NB + 5, 1500, 64 * 37 + 3])
def test_sweeps_are_bitwise_equal_for_every_grid_size(n, monkeypatch):
    NT = -(-n // NB)
    P, q, A, b, sets = _ragged_problem(n, seed=n)
    m = A.shape[0]
    rhss = _rhss(n, m, 200 + n)
    rv = np.random.default_rng(n).uniform(0.01, 10.0, m)
    _cap(monkeypatch, None)
    eng = _engine(P, q, A, b, sets, scaling=0)
    rho0 = eng.rho_vec()
    ref0, ref1 = O.DirectKKT(P, A, SIGMA, rho0), O.DirectKKT(P, A, SIGMA, rv)
    base0 = _check(P, A, eng, rhss, "n=%d uncapped" % n, ref0)
    eng.update_rho(rv, 1.0)
    base1 = _check(P, A, eng, rhss, "n=%d uncapped after update_rho" % n, ref1)
    eng.close()
    for cap in sorted({1, 2, 3, 5, max(1, NT - 1)}):
        _cap(monkeypatch, cap)
        eng = _engine(P, q, A, b, sets, scaling=0)
        for sol, want in zip(_solve_all(eng, rhss), base0):
            assert np.array_equal(sol, want), (n, cap, np.abs(sol - want).max())
        eng.update_rho(rv, 1.0)                                       # the refactor under the capped grid
        sols = _solve_all(eng, rhss)
        for sol, want in zip(sols, base1):
            assert np.array_equal(sol, want), (n, cap, "after update_rho", np.abs(sol - want).max())
        assert eng.kkt_factor_stats()["factorizations"] == 2
        eng.close()


def test_no_solve_reads_the_blocks_or_flags_of_the_previous_one(monkeypatch):
    # 24 tile columns on 3 CTAs: every CTA owns 8 rows; the ready flags carry the solve's epoch and are never reset
    n = 1500
    P, q, A, b, sets = _ragged_problem(n, seed=11)
    m = A.shape[0]
    r1, r2 = _rhss(n, m, 12, k=2)
    _cap(monkeypatch, 3)
    eng = _engine(P, q, A, b, sets, scaling=0)
    first = {}
    for k in range(20):
        which = k % 2
        sol, _ = eng.kkt_solve((r1, r2)[which])
        if which not in first:
            first[which] = sol
        assert np.array_equal(sol, first[which]), (k, np.abs(sol - first[which]).max())
    _check(P, A, eng, [r1, r2], "epochs n=1500 cap 3")
    eng.close()


# ---- the natural multi-row grid at full size -----------------------------------------------------------------------
def _large_problem(n, seed):
    """Sparse rows of 0-5 entries (one per column and then some), 17 dense rows (the panel path) and a sparse SPD P."""
    rng = np.random.default_rng(seed)
    ms = n + n // 4
    k = rng.integers(0, 6, ms)
    rows = np.repeat(np.arange(ms), k)
    cols = rng.integers(0, n, rows.size)
    As = sp.csr_matrix((rng.standard_normal(rows.size), (rows, cols)), shape=(ms, n))   # duplicates summed
    nd = 17
    Ad = np.zeros((nd, n))
    for i in range(nd):
        c = rng.choice(n, size=n if i == 0 else min(n, n // 4 + 37 * i), replace=False)
        Ad[i, c] = rng.standard_normal(c.size)
    A = sp.vstack([As, sp.csr_matrix(Ad)]).tocsc()
    B = sp.random(n, n, density=4.0 / n, random_state=rng, data_rvs=rng.standard_normal)
    S = (B + B.T) * 0.1
    P = (S + sp.diags(np.asarray(abs(S).sum(axis=1)).ravel() + rng.uniform(0.5, 1.5, n))).tocsc()
    m = A.shape[0]
    mz = ms // 3
    sets = [cosmo_b200.ZeroSet(mz), cosmo_b200.Nonnegatives(m - mz)]
    return P, rng.standard_normal(n), A, rng.standard_normal(m), sets


def _dense_cholesky_solve(P, A, rho, rhss):
    """Exact host solves through LAPACK: cho_factor of the dense M = P + sigma I + A'RA (one n x n array)."""
    m, n = A.shape
    Ar = sp.csr_matrix(A)
    nnz = np.diff(Ar.indptr)
    dense = (nnz >= 64) & (8 * nnz >= n)
    Gd = np.sqrt(rho[dense])[:, None] * Ar[dense].toarray()
    Mh = Gd.T @ Gd
    S = (Ar[~dense].T @ sp.diags(rho[~dense]) @ Ar[~dense] + P).tocoo()
    S.sum_duplicates()
    Mh[S.row, S.col] += S.data
    Mh[np.diag_indices(n)] += SIGMA
    c = la.cho_factor(Mh.T, lower=True, overwrite_a=True, check_finite=False)   # Mh.T: Fortran order, factored in place
    out = []
    for rhs in rhss:
        x1, x2 = rhs[:n], rhs[n:]
        y1 = la.cho_solve(c, x1 + Ar.T @ (rho * x2), check_finite=False)
        out.append(np.concatenate([y1, rho * (Ar @ y1 - x2)]))
    return out


def test_the_natural_grid_with_several_rows_per_cta_at_full_size(monkeypatch):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = NB * (2 * sms + 9) + 17                    # NT = 2 SMs + 10 > every grid the engine can choose (<= 2 SMs)
    NT = -(-n // NB)
    P, q, A, b, sets = _large_problem(n, seed=3)
    m = A.shape[0]
    rhss = _rhss(n, m, 4, k=2)
    _cap(monkeypatch, None)
    eng = _engine(P, q, A, b, sets, scaling=0)
    rho = eng.rho_vec()
    sols = _solve_all(eng, rhss)
    eng.close()
    _, bwd = _errors(P, A, rho, sols, rhss)
    _cap(monkeypatch, 37)                          # R = ceil(NT / 37) rows per CTA
    eng = _engine(P, q, A, b, sets, scaling=0)
    for sol, want in zip(_solve_all(eng, rhss), sols):
        assert np.array_equal(sol, want), np.abs(sol - want).max()
    eng.close()
    fwd = 0.0
    for sol, want in zip(sols, _dense_cholesky_solve(P, A, rho, rhss)):
        fwd = max(fwd, np.linalg.norm(sol - want) / (1 + np.linalg.norm(want)))
    print("n=%d NT=%d (%d SMs): forward %.2e (LAPACK) backward %.2e" % (n, NT, sms, fwd, bwd))
    assert fwd <= 1e-10 and bwd <= 1e-13, (fwd, bwd)


# ---- solve level ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("accelerator", ["EmptyAccelerator", "AndersonAccelerator"])
def test_solve_is_bitwise_equal_under_a_capped_grid(accelerator, monkeypatch):
    P, q, A, b, sets = cosmo_b200.problems.portfolio_socp(n=700, k=70, seed=4)   # NT = 11; cap 3: 4 rows per CTA
    out = []
    for cap in (None, 3):
        _cap(monkeypatch, cap)
        model = cosmo_b200.Model()
        model.set(P, q, A, b, sets, cosmo_b200.Settings(kkt_solver=DIRECT, max_iter=300, accelerator=accelerator))
        res = model.optimize()
        out.append((res.iter, res.x.copy(), res.s.copy(), res.y.copy()))
        model.engine.close()
    assert out[0][0] == out[1][0]
    for a, c in zip(out[0][1:], out[1][1:]):
        assert np.array_equal(a, c)


# ---- fp32 model -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [NB - 1, NB + 1, 1500])
def test_float32_kkt_solve(n, monkeypatch):
    # the factor is fp64 for both model types: the fp32 roundings are the rhs SpMV x1 + A'(rho x2), the cast of y1 and
    # y2 = rho (A y1 - x2), so the backward error is measured against K of the float32-rounded data
    P, q, A, b, sets = _ragged_problem(n, seed=n)
    m = A.shape[0]
    P32, A32 = (sp.csc_matrix(X.astype(np.float32).astype(np.float64)) for X in (P, A))
    rhss = [r.astype(np.float32) for r in _rhss(n, m, 300 + n)]
    out = []
    for cap in (None, 2):
        _cap(monkeypatch, cap)
        eng = _engine(P, q, A, b, sets, dtype=np.float32, scaling=0)
        rho = eng.rho_vec().astype(np.float64)
        sols = _solve_all(eng, rhss)
        assert all(s.dtype == np.float32 for s in sols)
        out.append(sols)
        eng.close()
    for a, c in zip(*out):
        assert np.array_equal(a, c)
    _, bwd = _errors(P32, A32, rho, [s.astype(np.float64) for s in out[0]], [r.astype(np.float64) for r in rhss])
    print("fp32 n=%d: backward %.2e" % (n, bwd))
    assert bwd <= 1e-5, bwd


# ---- scaled data ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [NB + 1, 1500])
def test_kkt_solve_on_ruiz_scaled_data(n):
    # kkt_solve runs on the resident (scaled) data: both forms compare against the scaled matrices
    P, q, A, b, sets = _ragged_problem(n, seed=n)
    m = A.shape[0]
    st = cosmo_b200.Settings(kkt_solver=DIRECT, scaling=10)
    rhss = _rhss(n, m, 400 + n)
    # host Ruiz (model.py with COSMO_B200_HOST_RUIZ=1): scaled data handed over with D, E, c
    Ps, qs, As, bs, setss, D, Ev, c = M.ruiz_equilibrate(P, q, A, b, sets, st)
    eng = E.Engine(Ps, qs, As, bs, [M.set_tuple(S) for S in setss], st.to_struct(), D=D, E=Ev, c=c)
    _check(Ps, As, eng, rhss, "n=%d host Ruiz" % n)
    eng.close()
    # device Ruiz: unscaled data, the engine equilibrates them and hands D, E, c back
    eng = E.Engine(P, q, A, b, [M.set_tuple(S) for S in sets], st.to_struct(), equilibrate=True)
    D, Ev, c = eng.scaling()
    assert not np.allclose(D, 1.0)
    Dm, Em = sp.diags(D), sp.diags(Ev)
    _check(sp.csc_matrix(c * (Dm @ P @ Dm)), sp.csc_matrix(Em @ A @ Dm), eng, rhss, "n=%d device Ruiz" % n)
    eng.close()


# ---- assembly split ---------------------------------------------------------------------------------------------------
def _spd_p(n, rng, zero=False):
    if zero:
        return sp.csc_matrix((n, n))
    B = sp.random(n, n, density=min(1.0, 4.0 / n), random_state=rng, data_rvs=rng.standard_normal)
    S = (B + B.T) * 0.1
    return (S + sp.diags(np.asarray(abs(S).sum(axis=1)).ravel() + rng.uniform(0.5, 1.5, n))).tocsc()


def _row(n, cols, rng):
    r = np.zeros(n)
    r[cols] = rng.standard_normal(len(cols))
    return r


def _split_case(name, n, seed):
    """(P, A, expected number of dense rows) of one assembly edge."""
    rng = np.random.default_rng(seed)
    sparse = [_row(n, rng.choice(n, size=rng.integers(1, 4), replace=False), rng) for _ in range(n + 5)]
    P = _spd_p(n, rng)
    if name in ("nnz64_n512", "nnz64_n513"):            # 64 entries: dense exactly when 8 * 64 >= n
        rows, nd = [_row(n, rng.choice(n, size=64, replace=False), rng)] + sparse, int(n == 512)
    elif name == "nnz63_n64":                           # fewer than 64 entries: sparse, however small n is
        rows, nd = [_row(n, rng.choice(n, size=63, replace=False), rng)] + sparse, 0
    elif name in ("nd64", "nd65"):                      # panel width 64 (ldg 64) against 65 (ldg 128)
        nd = int(name[2:])
        rows = [_row(n, rng.choice(n, size=n // 2, replace=False), rng) for _ in range(nd)] + sparse
    elif name in ("all_dense_m_lt_n", "all_dense_m_gt_n"):
        m = n - 50 if name == "all_dense_m_lt_n" else 2 * n
        rows, nd = list(rng.standard_normal((m, n))), m
    elif name == "shared_column":                       # column 5 reached by dense and by sparse rows
        rows = [_row(n, np.union1d([5], rng.choice(n, size=100, replace=False)), rng) for _ in range(3)]
        rows += [_row(n, np.union1d([5], rng.choice(n, size=2, replace=False)), rng) for _ in range(20)] + sparse
        nd = 3
    elif name == "p0_empty_columns":                    # P = 0, columns >= 100 of A empty: those pivots are sigma
        P = _spd_p(n, rng, zero=True)
        rows = [_row(n, rng.choice(100, size=8, replace=False), rng) for _ in range(200)]
        rows.append(_row(n, np.arange(100), rng))
        nd = 1
    else:
        raise ValueError(name)
    A = sp.csc_matrix(np.array(rows))
    return P, A, nd


SPLIT = [("nnz64_n512", 512), ("nnz64_n513", 513), ("nnz63_n64", 64), ("nd64", 256), ("nd65", 256),
         ("all_dense_m_lt_n", 200), ("all_dense_m_gt_n", 150), ("shared_column", 300), ("p0_empty_columns", 130)]


@pytest.mark.parametrize("name,n", SPLIT, ids=[s[0] for s in SPLIT])
def test_assembly_split_edges(name, n, monkeypatch, capfd):
    P, A, nd = _split_case(name, n, seed=len(name) + n)
    if name == "p0_empty_columns":
        assert A[:, 100:].nnz == 0 and P.nnz == 0
    m = A.shape[0]
    rng = np.random.default_rng(n)
    mz = m // 3
    sets = [cosmo_b200.ZeroSet(mz), cosmo_b200.Nonnegatives(m - mz)]
    monkeypatch.setenv("COSMO_B200_SETUP_DEBUG", "1")
    eng = _engine(P, rng.standard_normal(n), A, rng.standard_normal(m), sets, scaling=0)
    log = capfd.readouterr().err
    got = re.search(r"\[direct\] n (\d+) NT \d+ dense rows (\d+)", log)
    assert got and int(got.group(1)) == n and int(got.group(2)) == nd, log
    _check(P, A, eng, _rhss(n, m, 500 + n), "split %s" % name)
    eng.close()


# ---- pivots -----------------------------------------------------------------------------------------------------------
PIVOT = 3 * NB + 10                                      # in tile column 3


def _pivot_problem(covered):
    n = 5 * NB + 7
    rng = np.random.default_rng(9)
    d = np.ones(n)
    d[PIVOT] = -1.0
    P = sp.diags(d).tocsc()
    rows = [_row(n, [c], rng) for c in range(n) if c != PIVOT]
    if covered:
        rows.insert(0, np.eye(n)[PIVOT])                # an equality row on the -1: rho_eq = 100 makes M definite
    A = sp.csc_matrix(np.array(rows))
    m = A.shape[0]
    sets = [cosmo_b200.ZeroSet(1), cosmo_b200.Nonnegatives(m - 1)]
    return P, rng.standard_normal(n), A, rng.standard_normal(m), sets


def test_pivot_failure_in_a_later_tile_column(monkeypatch, capfd):
    P, q, A, b, sets = _pivot_problem(covered=False)
    monkeypatch.setenv("COSMO_B200_SETUP_DEBUG", "1")
    with pytest.raises(E.EngineError) as ei:
        _engine(P, q, A, b, sets, scaling=0)
    assert ei.value.code == E.ERR_INVALID and "Objective function is not convex." in str(ei.value)
    assert "pivot failure in tile column 3" in capfd.readouterr().err


def test_indefinite_p_made_definite_by_the_constraints_and_a_failing_refactor():
    # P is indefinite, but K = [P + sigma I, A'; A, -R^-1] has inertia (n, m, 0): the reference's inertia check accepts
    # it, and so does the pivot check (Sylvester)
    P, q, A, b, sets = _pivot_problem(covered=True)
    n, m = A.shape[1], A.shape[0]
    eng = _engine(P, q, A, b, sets, scaling=0)
    rho = eng.rho_vec()
    assert np.isclose(rho[0], 100.0)
    rhss = _rhss(n, m, 13)
    want = _check(P, A, eng, rhss, "indefinite P, covered")
    # a rho that makes M indefinite: the refactor before the next solve fails with the create-time message.  The
    # reference's update_rho! refactors without checking the inertia again; the engine checks every factorisation on
    # purpose, because its sweeps would otherwise solve with a factor holding NaN
    bad = rho.copy()
    bad[0] = 0.5
    eng.update_rho(bad, 1.0)
    with pytest.raises(E.EngineError) as ei:
        eng.kkt_solve(rhss[0])
    assert ei.value.code == E.ERR_INVALID and "Objective function is not convex." in str(ei.value)
    eng.update_rho(rho, 1.0)
    for sol, w in zip(_check(P, A, eng, rhss, "indefinite P, after the failed refactor"), want):
        assert np.array_equal(sol, w)                   # the same factor as at create, bit for bit
    st = eng.kkt_factor_stats()
    assert st["factorizations"] == 2 and st["factor_update_time"] > 0.0, st
    eng.close()


# ---- duplicates -------------------------------------------------------------------------------------------------------
def _with_duplicate(X, i, j):
    """X (CSC) with its entry (i, j) split into two stored entries 0.25 x and 0.75 x, left unsummed."""
    X = sp.csc_matrix(X)
    X.sort_indices()
    k = X.indptr[j] + int(np.nonzero(X.indices[X.indptr[j]:X.indptr[j + 1]] == i)[0][0])
    data = np.insert(X.data, k + 1, 0.75 * X.data[k])
    data[k] *= 0.25
    indices = np.insert(X.indices, k + 1, i)
    indptr = X.indptr.copy()
    indptr[j + 1:] += 1
    D = sp.csc_matrix((data, indices, indptr), shape=X.shape)
    assert D.nnz == X.nnz + 1 and abs(D - X).sum() < 1e-12
    return D


@pytest.mark.parametrize("which", ["A", "P"])
def test_duplicate_entries_are_refused_and_solve_once_summed(which):
    n = 150
    P, q, A, b, sets = _ragged_problem(n, seed=21)
    Ac = sp.csc_matrix(A)
    if which == "A":
        j = int(np.argmax(np.diff(Ac.indptr)))
        A2, P2 = _with_duplicate(Ac, int(Ac.indices[Ac.indptr[j]]), j), P
    else:
        A2, P2 = A, _with_duplicate(P, 7, 7)
    with pytest.raises(E.EngineError) as ei:
        _engine(P2, q, A2, b, sets, scaling=0)
    assert ei.value.code == E.ERR_INVALID and "duplicate" in str(ei.value), str(ei.value)
    A2, P2 = sp.csc_matrix(A2), sp.csc_matrix(P2)
    A2.sum_duplicates()
    P2.sum_duplicates()
    eng = _engine(P2, q, A2, b, sets, scaling=0)
    _check(P2, A2, eng, _rhss(n, A.shape[0], 22), "summed duplicates in %s" % which)
    eng.close()


# ---- switching solvers ------------------------------------------------------------------------------------------------
def test_switch_to_cg_and_back_refactors_at_the_current_rho():
    n = 300
    P, q, A, b, sets = _ragged_problem(n, seed=31)
    m = A.shape[0]
    eng = _engine(P, q, A, b, sets, scaling=0)
    rhss = _rhss(n, m, 32)
    _check(P, A, eng, rhss[:1], "switch: direct at create")
    assert eng.kkt_factor_stats()["factorizations"] == 1
    eng.update_settings(cosmo_b200.Settings(kkt_solver="CGIndirectKKTSolver", scaling=0).to_struct())
    rv = np.random.default_rng(33).uniform(0.01, 10.0, m)
    eng.update_rho(rv, 1.0)
    _, inner = eng.kkt_solve(rhss[0])
    assert inner > 0                                     # CG ran, not the stale factor
    eng.update_settings(cosmo_b200.Settings(kkt_solver=DIRECT, scaling=0).to_struct())
    assert np.array_equal(eng.rho_vec(), rv)
    _check(P, A, eng, rhss, "switch: direct again after update_rho under CG", O.DirectKKT(P, A, SIGMA, rv))
    assert eng.kkt_factor_stats()["factorizations"] == 2
    eng.close()
