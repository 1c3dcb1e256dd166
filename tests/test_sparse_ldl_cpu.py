"""CPU checks of the symbolic analysis of the full KKT matrix K = [P + sigma I, A'; A, -R^-1] (csrc/ldl_symbolic.h,
`cosmo_b200_kkt_symbolic`): the returned order is a permutation, an independent symbolic elimination of the permuted K
in NumPy gives the reported nnz(L), a NumPy restatement of the supernode partition (fundamental supernodes, relaxed
amalgamation) reproduces the reported supernode counts and sizes and keeps every column's exact structure inside its
supernode with the explicit zeros inside the amalgamation bound, an LDL' factorisation held only in the supernodal blocks
solves K x = b as SuperLU does, the ordering's fill is within 1.5x SuperLU's minimum degree on C3, C4 and C5, dense nodes
are ordered last, and the analysis is deterministic."""
import math
import os
import re

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as sla

import cosmo_b200
from cosmo_b200 import chordal, problems
from cosmo_b200 import engine as E
from tests import golden_problems as GP

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAN_IN_CHUNK = 256


def relax_fraction(width):
    return 0.5 if width <= 16 else (0.2 if width <= 64 else 0.05)


def kkt_matrix(P, A):
    """K with P's pattern made diagonally dominant, so that K = [P', A'; A, -I] is quasi-definite (only the pattern
    matters to the analysis)."""
    m = A.shape[0]
    Pabs = abs(sp.csc_matrix(P))
    Psym = (Pabs + Pabs.T) * 0.5
    Psym = Psym + sp.diags(np.asarray(Psym.sum(axis=1)).ravel() + 1.0)
    return sp.bmat([[Psym, sp.csc_matrix(A).T], [sp.csc_matrix(A), -sp.identity(m)]], format="csc")


def exact_structure(K, perm):
    """Rows i > j of every column j of L for the permuted K, by elimination over the elimination tree."""
    N = K.shape[0]
    Kp = sp.tril(K[perm][:, perm], k=-1, format="csc")
    Kp.sort_indices()
    structs = [None] * N
    parent = np.full(N, -1)
    kids = [[] for _ in range(N)]
    for j in range(N):
        parts = [Kp.indices[Kp.indptr[j]:Kp.indptr[j + 1]]]
        for c in kids[j]:
            s = structs[c]
            parts.append(s[s > j])
        s = np.unique(np.concatenate(parts)) if len(parts) > 1 else parts[0].copy()
        structs[j] = s
        if len(s):
            parent[j] = s[0]
            kids[s[0]].append(j)
    return parent, structs


def supernodes(parent, colcount):
    """Restatement of ldl_symbolic.h's partition: fundamental supernodes, then merging with the contiguous last child
    while the explicit zeros stay within relax_fraction(width) of the stored trapezoid."""
    N = len(parent)
    nchild = np.bincount(parent[parent >= 0], minlength=N)
    fund_last = np.empty(N, dtype=np.int64)
    f = 0
    for j in range(N):
        if j + 1 < N and parent[j] == j + 1 and nchild[j + 1] == 1 and colcount[j] == colcount[j + 1] + 1:
            continue
        fund_last[f:j + 1] = j
        f = j + 1
    stack = []   # [first, last, exact, parent_last]
    f = 0
    while f < N:
        l = fund_last[f]
        cur = [f, l, int(colcount[f:l + 1].sum()), -1 if parent[l] == -1 else fund_last[parent[l]]]
        below = colcount[l] - 1
        while stack and stack[-1][1] == cur[0] - 1 and cur[0] <= stack[-1][3] <= l:
            c = stack[-1]
            k = l - c[0] + 1
            stored = k * (k + 1) // 2 + k * below
            if stored - (cur[2] + c[2]) > relax_fraction(k) * stored:
                break
            cur[0] = c[0]
            cur[2] += c[2]
            stack.pop()
        stack.append(cur)
        f = l + 1
    return [(s[0], s[1]) for s in stack]


def check_analysis(P, A):
    m, n = A.shape
    N = n + m
    perm, info = E.kkt_symbolic(P, A)
    assert np.array_equal(np.sort(perm), np.arange(N))
    K = kkt_matrix(P, A)
    parent, structs = exact_structure(K, perm)
    colcount = np.array([len(s) + 1 for s in structs], dtype=np.int64)
    assert info["nnz_L"] == int(colcount.sum())
    # the returned order is postordered: every parent comes after its children, every subtree is contiguous
    assert np.all((parent == -1) | (parent > np.arange(N)))
    sns = supernodes(parent, colcount)
    assert info["supernodes"] == len(sns)
    sn_of = np.empty(N, dtype=np.int64)
    widest = front = fbytes = 0
    for s, (f, l) in enumerate(sns):
        sn_of[f:l + 1] = s
        k = l - f + 1
        below = set(structs[l].tolist())
        assert len(below) == colcount[l] - 1
        for j in range(f, l + 1):      # the exact structure lies inside the supernode's rows
            assert set(structs[j].tolist()) <= set(range(j + 1, l + 1)) | below
        stored = k * (k + 1) // 2 + k * len(below)
        zeros = stored - int(colcount[f:l + 1].sum())
        assert 0 <= zeros <= relax_fraction(k) * stored
        widest = max(widest, k)
        front = max(front, k + len(below))
        fbytes += 8 * (k + len(below)) * k
    depth = np.ones(len(sns), dtype=np.int64)
    for s in range(len(sns) - 1, -1, -1):
        p = parent[sns[s][1]]
        if p != -1:
            depth[s] = depth[sn_of[p]] + 1
    assert (info["widest"], info["largest_front"], info["factor_bytes"], info["height"]) == (widest, front, fbytes,
                                                                                            int(depth.max()))
    Pc = sp.csc_matrix(P)
    p_upper = int(sp.triu(Pc).nnz)
    assert info["workspace_bytes"] == 8 * front * FAN_IN_CHUNK + 16 * N + 8 * (p_upper + sp.csc_matrix(A).nnz + N)
    return perm, sns, structs


def supernodal_ldl_solve(K, perm, sns, structs, rhs):
    """LDL' of the permuted K held only in the supernodal blocks the analysis sizes: block s is (w + r) x w over the rows
    [f..l] + the structure of column l.  Values are scattered into the blocks, each supernode is factored without
    pivoting, and its update D-scaled is subtracted from the blocks of its ancestors; an entry with no slot in a block
    fails the test.  Returns the solution of K x = rhs and the number of positive pivots."""
    N = K.shape[0]
    sn_of = np.empty(N, dtype=np.int64)
    rows, pos, blocks = [], [], []
    for s, (f, l) in enumerate(sns):
        sn_of[f:l + 1] = s
        R = np.concatenate([np.arange(f, l + 1), structs[l]])
        rows.append(R)
        pos.append({int(i): k for k, i in enumerate(R)})
        blocks.append(np.zeros((len(R), l - f + 1)))
    Kp = sp.tril(K[perm][:, perm], format="coo")
    for i, j, v in zip(Kp.row, Kp.col, Kp.data):
        s = sn_of[j]
        blocks[s][pos[s][int(i)], j - sns[s][0]] += v
    d = np.empty(N)
    for s, (f, l) in enumerate(sns):
        B, w = blocks[s], l - f + 1
        for c in range(w):
            d[f + c] = B[c, c]
            B[c + 1:, c + 1:w] -= np.outer(B[c + 1:, c], B[c + 1:w, c]) / B[c, c]
            B[c + 1:, c] /= B[c, c]
            B[c, c] = 1.0
        Lb = B[w:, :]
        if not len(Lb):
            continue
        U = (Lb * d[f:l + 1]) @ Lb.T
        below = rows[s][w:]
        for jj, j in enumerate(below):
            t = sn_of[j]
            tgt = [pos[t][int(i)] for i in below[jj:]]
            blocks[t][tgt, j - sns[t][0]] -= U[jj:, jj]
    y = np.asarray(rhs, dtype=np.float64)[perm].copy()
    for s, (f, l) in enumerate(sns):                 # L y = b
        B, w = blocks[s], l - f + 1
        for c in range(w):
            y[rows[s][c + 1:]] -= B[c + 1:, c] * y[f + c]
    y /= d
    for s in range(len(sns) - 1, -1, -1):            # L' x = D^-1 y
        f, l = sns[s]
        B, w = blocks[s], l - f + 1
        for c in range(w - 1, -1, -1):
            y[f + c] -= B[c + 1:, c] @ y[rows[s][c + 1:]]
    x = np.empty(N)
    x[perm] = y
    return x, int((d > 0).sum())


def _ragged(n, seed, p_dense=True):
    """Rows of A: empty, short and dense; P random symmetric (or zero)."""
    rng = np.random.default_rng(seed)
    rows = []
    for i in range(max(12, n + 9)):
        k = min([0, 1, 2, 5, n, 3, n // 2 + 1, 0][i % 8], n)
        row = np.zeros(n)
        c = rng.choice(n, size=k, replace=False)
        row[c] = rng.standard_normal(k)
        rows.append(row)
    A = sp.csc_matrix(np.array(rows))
    if not p_dense:
        return sp.csc_matrix((n, n)), A
    B = sp.random(n, n, density=min(1.0, 4.0 / n), random_state=rng)
    return (B + B.T + sp.identity(n)).tocsc(), A


def _g_problems():
    out = []
    for name in ("g1_qp_nonneg", "g1_qp_box", "g2_box_feasible", "g3_hs21", "g12_lp", "g4_small_sdp",
                 "g5_sigma_max_lmi", "g6_chordal_sdp", "g13_lovasz_petersen"):
        P, _, cons = getattr(GP, name)()
        A = sp.vstack([sp.csr_matrix(c.A if sp.issparse(c.A) else np.atleast_2d(c.A)) for c in cons], format="csc")
        out.append((name, sp.csc_matrix(P), A))
    return out


@pytest.mark.parametrize("name,P,A", _g_problems(), ids=lambda v: v if isinstance(v, str) else "")
def test_golden_problems(name, P, A):
    check_analysis(P, A)


@pytest.mark.parametrize("n", [1, 2, 7, 64, 65, 200, 700])
def test_ragged_shapes(n):
    check_analysis(*_ragged(n, n))
    check_analysis(*_ragged(n, n + 1, p_dense=False))   # P = 0


def test_block_tridiagonal_chain_and_extreme_aspect():
    nb, bs = 60, 5
    blocks = sp.random(bs, bs, density=1.0, random_state=0) + sp.identity(bs)
    P = sp.kron(sp.diags([1.0, 1.0, 1.0], [-1, 0, 1], shape=(nb, nb)), blocks, format="csc")
    check_analysis(P + P.T, sp.csc_matrix((0, nb * bs)))                # deep chain, m = 0
    check_analysis(P + P.T, sp.random(3, nb * bs, density=0.02, random_state=1, format="csc"))      # m << n
    check_analysis(sp.csc_matrix((4, 4)), sp.random(400, 4, density=0.5, random_state=2, format="csc"))   # m >> n
    check_analysis(sp.csc_matrix(np.ones((30, 30))), sp.csc_matrix(np.ones((20, 30))))   # one dense front


def _c5(nv):
    rows, cols, w = problems.banded_random_graph(nv, 3.0, 20, seed=1)
    P, q, A, b, sets = problems.maxcut_dual_sdp(nv, rows, cols, w)
    P2, q2, A2, b2, sets2, _ = chordal.decompose(P, q, A, b, sets, merge="parent_child")
    return P2, A2


def _numeric_cases():
    out = [("ragged%d" % n, *_ragged(n, n)) for n in (1, 7, 65, 150)]
    out.append(("ragged_P0", *_ragged(90, 3, p_dense=False)))
    P, _, A, _, _ = problems.portfolio_socp(300, 30, seed=3)
    out.append(("c3", P, A))
    P, _, A, _, _ = problems.closest_correlation_sdp(12)
    out.append(("c4", P, A))
    out.append(("c5", *_c5(120)))
    out.extend(("golden_" + name, P, A) for name, P, A in _g_problems())
    return out


@pytest.mark.parametrize("name,P,A", _numeric_cases(), ids=lambda v: v if isinstance(v, str) else "")
def test_supernodal_layout_holds_the_factor(name, P, A):
    """The LDL' factor of K fits the supernodal blocks the analysis sizes, its solve matches SuperLU to 1e-12, and it
    has n positive pivots (K is quasi-definite)."""
    perm, sns, structs = check_analysis(P, A)
    K = kkt_matrix(P, A)
    if sp.csc_matrix(A).nnz:                       # the values of A matter for the solve, not for the analysis
        A = sp.csc_matrix(A, dtype=np.float64, copy=True)
        A.data = np.random.default_rng(0).standard_normal(A.nnz)
        K = kkt_matrix(P, A)
    rhs = np.random.default_rng(1).standard_normal(K.shape[0])
    x, npos = supernodal_ldl_solve(K, perm, sns, structs, rhs)
    ref = sla.splu(K, permc_spec="MMD_AT_PLUS_A", diag_pivot_thresh=0.0, options={"SymmetricMode": True}).solve(rhs)
    err = np.linalg.norm(x - ref) / max(np.linalg.norm(ref), 1e-300)
    print("%s: N = %d, supernodes = %d, |x - splu| / |splu| = %.1e" % (name, K.shape[0], len(sns), err))
    assert err <= 1e-12 and npos == P.shape[0]


def test_small_workloads_c3_c4_c5():
    P, _, A, _, _ = problems.portfolio_socp(300, 30, seed=3)
    check_analysis(P, A)
    P, _, A, _, _ = problems.closest_correlation_sdp(30)
    check_analysis(P, A)
    check_analysis(*_c5(300))


@pytest.mark.parametrize("which", ["C3", "C4", "C5"])
def test_ordering_quality_against_superlu_mmd(which):
    if which == "C3":
        P, _, A, _, _ = problems.portfolio_socp(4000, 400, seed=1)
    elif which == "C4":
        P, _, A, _, _ = problems.closest_correlation_sdp(200)
    else:
        P, A = _c5(2000)
    perm, info = E.kkt_symbolic(P, A)
    lu = sla.splu(kkt_matrix(P, A), permc_spec="MMD_AT_PLUS_A", diag_pivot_thresh=0.0,
                  options={"SymmetricMode": True})
    print("%s: n = %d, m = %d, nnz(L) = %d, SuperLU MMD %d, %s" % (which, A.shape[1], A.shape[0], info["nnz_L"],
                                                                  lu.L.nnz, info))
    assert info["nnz_L"] <= 1.5 * lu.L.nnz


def test_dense_nodes_are_postponed_and_counted():
    P, _, A, _, _ = problems.portfolio_socp(2000, 40, seed=2)
    m, n = A.shape
    N = n + m
    perm, info = E.kkt_symbolic(P, A)
    K = kkt_matrix(P, A)
    deg = np.diff(K.indptr) - 1
    thr = max(16, int(10.0 * math.sqrt(N)))
    dense = np.flatnonzero(deg > thr)
    assert info["dense"] == len(dense) > 0          # the 1'x = 1 row and the F' rows
    assert set(perm[N - len(dense):].tolist()) == set(dense.tolist())


def test_deterministic():
    P, _, A, _, _ = problems.portfolio_socp(500, 50, seed=4)
    p1, i1 = E.kkt_symbolic(P, A)
    p2, i2 = E.kkt_symbolic(P, A)
    assert np.array_equal(p1, p2) and i1 == i2


def test_invalid_input_is_refused():
    A = sp.csc_matrix((np.ones(2), np.array([0, 0]), np.array([0, 2, 2])), shape=(3, 2))   # duplicate (0, 0)
    with pytest.raises(E.EngineError) as ei:
        E.kkt_symbolic(sp.identity(2, format="csc"), A)
    assert ei.value.code == E.ERR_INVALID and "duplicate" in str(ei.value)
    with pytest.raises(E.EngineError):
        E.kkt_symbolic(sp.identity(3, format="csc"), sp.csc_matrix((2, 2)))


def test_exported_and_declared():
    assert "cosmo_b200_kkt_symbolic" in E.EXPORTS
    src = open(os.path.join(ROOT, "include", "cosmo_b200.h")).read()
    assert re.search(r"int cosmo_b200_kkt_symbolic\(const cosmo_b200_problem\* prob, int64_t\* perm, int64_t info\[8\]\)",
                     src)
