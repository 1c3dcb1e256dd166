"""The direct KKT solver (COSMO_B200_KKT_DIRECT, csrc/direct.cuh) through the C ABI, against the oracle's direct
path (O.DirectKKT, a sparse LU of the full quasi-definite KKT matrix: the stand-in for QdldlKKTSolver)."""
import numpy as np
import pytest
import scipy.sparse as sp

import cosmo_b200
from cosmo_b200 import engine as E
from oracle import cosmo_oracle as O
from oracle.bridge import to_oracle_cones
from tests import golden_problems as G

pytestmark = pytest.mark.gpu

DIRECT = "DirectReducedKKTSolver"
NB = 64


def _engine(P, q, A, b, sets, dtype=np.float64, **kw):
    st = cosmo_b200.Settings(kkt_solver=DIRECT, **kw).to_struct()
    return E.Engine(P, q, A, b, [cosmo_b200.model.set_tuple(S) for S in sets], st, dtype=dtype)


def _ragged_problem(n, seed):
    """Rows of A: empty ones, short ones and dense ones (both assembly paths); Zero, Nonnegatives and Box sets so that
    the three rho classes appear (x1e3 equality rows, RHO_MIN rows with b > COSMO_INFTY or an unbounded Box)."""
    rng = np.random.default_rng(seed)
    rows = []
    for i in range(max(12, n + 9)):
        k = [0, 1, 2, 5, n, 3, n // 2 + 1, 0][i % 8]
        k = min(k, n)
        c = np.sort(rng.choice(n, size=k, replace=False))
        row = np.zeros(n)
        row[c] = rng.standard_normal(k)
        rows.append(row)
    A = sp.csc_matrix(np.array(rows))
    m = A.shape[0]
    B = sp.random(n, n, density=min(1.0, 4.0 / n), random_state=rng, data_rvs=rng.standard_normal)
    S = (B + B.T) * 0.1
    P = (S + sp.diags(np.asarray(abs(S).sum(axis=1)).ravel() + rng.uniform(0.5, 1.5, n))).tocsc()
    q = rng.standard_normal(n)
    mz, mn = m // 4, m // 4
    mb = m - mz - mn
    b = rng.standard_normal(m)
    b[mz + mn - 2:mz + mn] = 1e21                      # Nonnegatives rows with b > COSMO_INFTY: RHO_MIN
    l = -rng.uniform(0.5, 1.0, mb)
    u = rng.uniform(0.5, 1.0, mb)
    l[:2], u[:2] = -np.inf, np.inf                     # unbounded Box rows: RHO_MIN
    sets = [cosmo_b200.ZeroSet(mz), cosmo_b200.Nonnegatives(mn), cosmo_b200.Box(l, u)]
    return P, q, A, b, sets


def _kkt(P, A, sigma, rho):
    n = P.shape[0]
    return sp.bmat([[P + sigma * sp.identity(n), A.T], [A, -sp.diags(1.0 / rho)]], format="csr")


@pytest.mark.parametrize("n", [1, 2, NB - 1, NB, NB + 1, 3 * NB + 5, 1500])
def test_kkt_solve_matches_the_oracle_direct_solve(n):
    P, q, A, b, sets = _ragged_problem(n, seed=n)
    m = A.shape[0]
    eng = _engine(P, q, A, b, sets, scaling=0)
    rho = eng.rho_vec()
    assert {0.1, 100.0, 1e-6} <= set(np.round(rho, 12).tolist())
    ref = O.DirectKKT(P, A, 1e-6, rho)
    K = _kkt(P, A, 1e-6, rho)
    normK = abs(K).sum(axis=1).max()
    rng = np.random.default_rng(100 + n)
    worst_fwd = worst_bwd = 0.0
    for _ in range(3):
        rhs = rng.standard_normal(n + m)
        sol, inner = eng.kkt_solve(rhs)
        want = ref.solve(rhs)
        assert inner == 0
        fwd = np.linalg.norm(sol - want) / (1 + np.linalg.norm(want))
        bwd = np.abs(K @ sol - rhs).max() / (normK * np.abs(sol).max() + np.abs(rhs).max())
        worst_fwd, worst_bwd = max(worst_fwd, fwd), max(worst_bwd, bwd)
    # measured on a B200 with the first build of the sweeps (division by the pivots instead of reciprocal pivots):
    # forward 9e-17 (n = 1) .. 6.6e-13 (n = 1500), backward 2e-23 .. 5.5e-19
    print("n=%d forward %.2e backward %.2e" % (n, worst_fwd, worst_bwd))
    assert worst_fwd <= 1e-10 and worst_bwd <= 1e-13, (worst_fwd, worst_bwd)
    st = eng.kkt_factor_stats()
    assert st["factorizations"] == 1 and st["init_factor_time"] > 0.0 and st["factor_update_time"] == 0.0


def test_refactor_after_rho_sigma_and_b_updates():
    P, q, A, b, sets = _ragged_problem(150, seed=5)
    m, n = A.shape
    eng = _engine(P, q, A, b, sets, scaling=0)
    rng = np.random.default_rng(3)
    rhs = rng.standard_normal(n + m)

    def check(sigma, count):
        rho = eng.rho_vec()
        sol, _ = eng.kkt_solve(rhs)
        want = O.DirectKKT(P, A, sigma, rho).solve(rhs)
        assert np.linalg.norm(sol - want) <= 1e-10 * (1 + np.linalg.norm(want))
        assert eng.kkt_factor_stats()["factorizations"] == count

    check(1e-6, 1)
    rv = rng.uniform(0.01, 10.0, m)
    eng.update_rho(rv, 1.0)                                   # update_rho!(kkt_solver, rho_vec)
    assert np.array_equal(eng.rho_vec(), rv)
    check(1e-6, 2)
    st = cosmo_b200.Settings(kkt_solver=DIRECT, scaling=0, sigma=1e-3).to_struct()
    eng.update_settings(st)
    check(1e-3, 3)
    b2 = b.copy()
    b2[m // 4:m // 2] = 1e21                                  # every Nonnegatives row becomes loose: rho changes
    eng.update_qb(None, b2)
    check(1e-3, 4)
    stats = eng.kkt_factor_stats()
    assert stats["factor_update_time"] > 0.0


def _solve_mine(builder, dtype=np.float64, **kw):
    P, q, cons = builder()
    model = cosmo_b200.Model(dtype=dtype)
    cosmo_b200.assemble(model, P, q, _to_mine(cons), cosmo_b200.Settings(kkt_solver=DIRECT, **kw))
    return cosmo_b200.optimize(model), model


def _solve_oracle(builder, **kw):
    P, q, cons = builder()
    Pm, qm, A, b, cones = O.assemble(P, q, cons)
    return O.solve(Pm, qm, A, b, cones, O.Settings(**kw))


def _to_mine(cons):
    out = []
    for c in cons:
        S = c.convex_set
        if isinstance(S, O.Box):
            S2 = cosmo_b200.Box(S.l, S.u)
        elif isinstance(S, (O.PowerCone, O.DualPowerCone)):
            S2 = getattr(cosmo_b200, type(S).__name__)(S.alpha)
        else:
            S2 = getattr(cosmo_b200, type(S).__name__)(S.dim)
        out.append(cosmo_b200.Constraint(c.A, c.b, S2))
    return out


def _same(res, ref, tol=1e-8):
    assert res.status == ref.status and res.iter == ref.iter, (res.status, res.iter, ref.status, ref.iter)
    if ref.status != "Solved":     # the iterates of an infeasible problem diverge; the certificate is the status
        return
    if np.isfinite(ref.obj_val):
        assert abs(res.obj_val - ref.obj_val) <= tol * max(1.0, abs(ref.obj_val))
    for a, r in ((res.x, ref.x), (res.s, ref.s), (res.y, ref.y)):
        assert np.max(np.abs(a - r), initial=0.0) <= tol * max(1.0, np.max(np.abs(r), initial=0.0))


@pytest.mark.parametrize("builder", [G.g1_qp_nonneg, G.g1_qp_box])
@pytest.mark.parametrize("scaling", [0, 10])
def test_g1_matches_the_oracle_direct_path(builder, scaling):
    res, model = _solve_mine(builder, scaling=scaling)
    ref = _solve_oracle(builder, scaling=scaling)
    _same(res, ref)
    assert np.max(np.abs(res.x - G.G1_X)) < 1e-3 and abs(res.obj_val - G.G1_OBJ) < 1e-3
    assert res.kkt_inner_iterations == 0
    assert {"init_factor_time", "factor_update_time"} <= set(res.times)


def test_g1_fixed_rho_reaches_the_survey_iteration_count():
    # SURVEY 8c: G1 with scaling = 0 and fixed rho takes 375 iterations with an exact KKT solve
    res, _ = _solve_mine(G.g1_qp_nonneg, scaling=0, adaptive_rho=False)
    assert res.status == "Solved" and res.iter == 375


@pytest.mark.parametrize("scaling", [0, 10])
def test_g2_statuses(scaling):
    for bld, status, kw in ((G.g2_box_feasible, "Solved", {}),
                            (G.g2_box_primal_infeasible_1, "Primal_infeasible", {}),
                            (G.g2_box_primal_infeasible_2, "Primal_infeasible", {}),
                            (G.g2_box_dual_infeasible, "Dual_infeasible", dict(check_infeasibility=20 if scaling == 0 else 40))):
        res, _ = _solve_mine(bld, scaling=scaling, **kw)
        ref = _solve_oracle(bld, scaling=scaling, **kw)
        assert res.status == status == ref.status and res.iter == ref.iter, (bld.__name__, res.status, res.iter, ref.iter)


@pytest.mark.parametrize("builder,kw", [(G.g3_hs21, {}), (G.g12_lp, dict(eps_abs=1e-4, eps_rel=1e-5)),
                                        (G.g4_small_sdp, dict(check_termination=1)), (G.g5_sigma_max_lmi, {})],
                         ids=["g3", "g12", "g4", "g5"])
def test_literal_problems_match_the_oracle_direct_path(builder, kw):
    res, _ = _solve_mine(builder, **kw)
    ref = _solve_oracle(builder, **kw)
    _same(res, ref)


@pytest.mark.parametrize("name,builder,status,obj,atol,kw", G.G15_G16, ids=[g[0] for g in G.G15_G16])
def test_g15_g16_exp_pow_cones(name, builder, status, obj, atol, kw):
    res, _ = _solve_mine(builder, **kw)
    ref = _solve_oracle(builder, **kw)
    assert res.status == status == ref.status
    _same(res, ref, tol=1e-6)
    if obj is not None:
        assert abs(res.obj_val - obj) < atol


def test_g14_model_updates_and_warm_start():
    P, q, cons = G.g1_qp_nonneg()
    model = cosmo_b200.Model()
    cosmo_b200.assemble(model, P, q, _to_mine(cons), cosmo_b200.Settings(kkt_solver=DIRECT, check_termination=1))
    r1 = model.optimize()
    r2 = model.optimize()
    assert abs(r1.obj_val - r2.obj_val) <= 1e-3 and r2.iter <= r1.iter       # model_modifications.jl:29-31
    model = cosmo_b200.Model()
    cosmo_b200.assemble(model, P, q, _to_mine(cons), cosmo_b200.Settings(kkt_solver=DIRECT))
    model.optimize()
    model.update(q=np.array([2.0, 3.0]))
    r = model.optimize()
    assert abs(r.obj_val - 3.5) < 1e-3 and np.linalg.norm(r.x - [0.5, 0.5]) < 1e-3   # :41-43
    model = cosmo_b200.Model()
    cosmo_b200.assemble(model, np.zeros((2, 2)), np.array([1.0, 1.0]),
                        cosmo_b200.Constraint(np.eye(2), np.array([-2.0, -3.0]), cosmo_b200.Nonnegatives),
                        cosmo_b200.Settings(kkt_solver=DIRECT, check_termination=20))
    r = model.optimize()
    assert np.linalg.norm(r.x - [2.0, 3.0]) < 1e-3
    before = model.engine.kkt_factor_stats()["factorizations"]
    model.update(b=np.array([0.0, 1.0]))
    assert model.engine.kkt_factor_stats()["factorizations"] == before      # refactored lazily, at the next solve
    assert np.linalg.norm(model.optimize().x - [0.0, -1.0]) < 1e-4               # :57-59
    assert model.engine.kkt_factor_stats()["factorizations"] > before


def _g6_decomposed(merge):
    from cosmo_b200 import chordal
    P, q, cons = G.g6_chordal_sdp()
    Pm, qm, A0, b0, _ = O.assemble(P, q, cons)
    return chordal.decompose(Pm, qm, A0, b0, [cosmo_b200.PsdConeTriangle(45)], merge=merge)


def test_g6_tight_tolerance_is_solved_where_cg_stalls():
    # DESIGN 6: at eps = 1e-7 the CG plugin stalls at Max_iter_reached; the exact solve reaches Solved
    P2, q2, A2, b2, sets2, _ = _g6_decomposed("none")
    tight = dict(eps_abs=1e-7, eps_rel=1e-7)
    model = cosmo_b200.Model()
    model.set(P2, q2, A2, b2, sets2, cosmo_b200.Settings(kkt_solver=DIRECT, **tight))
    res = model.optimize()
    ref = O.solve(P2, q2, A2, b2, to_oracle_cones(sets2), O.Settings(**tight))
    assert res.status == ref.status == "Solved" and res.iter == ref.iter, (res.status, res.iter, ref.iter)
    assert abs(res.obj_val - ref.obj_val) <= 1e-8 * max(1.0, abs(ref.obj_val))


def test_g6_decompose_with_the_direct_solver():
    # the reference's default pairing: chordal decomposition (CliqueGraphMerge) and a direct KKT solver
    P, q, cons = G.g6_chordal_sdp()
    model = cosmo_b200.Model()
    cosmo_b200.assemble(model, P, q, _to_mine(cons), cosmo_b200.Settings(kkt_solver=DIRECT, decompose=True))
    res = model.optimize()
    P2, q2, A2, b2, sets2, _ = _g6_decomposed("clique_graph")
    ref = O.solve(P2, q2, A2, b2, to_oracle_cones(sets2), O.Settings())
    assert res.status == ref.status == "Solved" and res.iter == ref.iter
    assert abs(res.obj_val - ref.obj_val) <= 1e-8 * max(1.0, abs(ref.obj_val))
    full = _solve_oracle(G.g6_chordal_sdp, eps_abs=1e-7, eps_rel=1e-7)
    assert abs(res.obj_val - full.obj_val) < 1e-3


@pytest.mark.parametrize("accelerator", ["EmptyAccelerator", "AndersonAccelerator"])
def test_iterates_match_the_oracle_direct_path(accelerator):
    # 90 iterations cross two rho adaptations (interval 40) and two infeasibility checks
    P, q, A, b, sets = cosmo_b200.problems.random_sparse_qp(40, 70, 0.15, seed=7)
    cones = to_oracle_cones(sets)
    acc = {"EmptyAccelerator": "empty", "AndersonAccelerator": "anderson"}[accelerator]
    for iters in (1, 41, 90):
        ref = O.solve(P, q, A, b, cones, O.Settings(max_iter=iters, eps_abs=1e-14, eps_rel=1e-14, accelerator=acc))
        model = cosmo_b200.Model()
        model.set(P, q, A, b, sets, cosmo_b200.Settings(kkt_solver=DIRECT, max_iter=iters, eps_abs=1e-14, eps_rel=1e-14,
                                                        accelerator=accelerator))
        res = model.optimize()
        w = model.engine.w()
        assert res.iter == ref.iter and list(np.round(res.info.rho_updates, 9)) == list(np.round(ref.info.rho_updates, 9))
        assert np.linalg.norm(w - ref.w) / np.linalg.norm(ref.w) <= 1e-10, (iters, np.linalg.norm(w - ref.w) / np.linalg.norm(ref.w))
        # one factorisation at create and one per rho adaptation (rho_updates starts with the initial rho)
        assert model.engine.kkt_factor_stats()["factorizations"] == len(res.info.rho_updates)


def test_refactor_count_follows_the_rho_adaptations():
    # AccelerationTests/max_rho_adaption.jl:21-36: a start at rho = 1e-6 is adapted several times
    res, model = _solve_mine(G.g1_qp_nonneg, adaptive_rho_interval=25, rho=1e-6, eps_abs=1e-6, eps_rel=1e-4)
    assert res.status == "Solved" and len(res.info.rho_updates) >= 3
    assert model.engine.kkt_factor_stats()["factorizations"] == len(res.info.rho_updates)
    assert res.times["factor_update_time"] > 0.0 and res.times["init_factor_time"] > 0.0


def test_float32_model_solves_g1():
    # Model{Float32}: the factor stays fp64; tolerance of the reference's simple.jl: 1e-3
    res, _ = _solve_mine(G.g1_qp_box, dtype=np.float32, eps_abs=1e-4, eps_rel=1e-4)
    assert res.status == "Solved" and np.max(np.abs(res.x - G.G1_X)) < 1e-3 and abs(res.obj_val - G.G1_OBJ) < 1e-3


def test_indefinite_objective_is_refused_at_create():
    P = sp.csc_matrix(np.diag([1.0, -1.0]))
    A = sp.csc_matrix(np.array([[1.0, 0.0]]))
    with pytest.raises(E.EngineError) as ei:
        _engine(P, np.zeros(2), A, np.zeros(1), [cosmo_b200.Nonnegatives(1)], scaling=0)
    assert ei.value.code == E.ERR_INVALID and "Objective function is not convex." in str(ei.value)


def test_memory_gate_refuses_a_factor_larger_than_half_the_device():
    n = 250_000                                       # packed lower factor: ~250 GB
    I = sp.identity(n, format="csc")
    with pytest.raises(E.EngineError) as ei:
        _engine(I, np.zeros(n), I, np.zeros(n), [cosmo_b200.Nonnegatives(n)], scaling=0)
    assert ei.value.code == E.ERR_UNSUPPORTED and "bytes" in str(ei.value), str(ei.value)


def test_bitwise_reproducible():
    P, q, A, b, sets = cosmo_b200.problems.portfolio_socp(n=700, k=70, seed=4)   # dense rows: both assembly paths
    out = []
    for _ in range(2):
        model = cosmo_b200.Model()
        model.set(P, q, A, b, sets, cosmo_b200.Settings(kkt_solver=DIRECT, max_iter=300))
        res = model.optimize()
        out.append((res.x.copy(), res.s.copy(), res.y.copy(), res.iter))
    assert out[0][3] == out[1][3]
    for a, c in zip(out[0][:3], out[1][:3]):
        assert np.array_equal(a, c)
