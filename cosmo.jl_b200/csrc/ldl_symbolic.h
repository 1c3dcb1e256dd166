// ldl_symbolic.h -- host symbolic analysis of the full quasi-definite KKT matrix (DESIGN §3d).
//
//   K = [P + sigma I, A'; A, -R^-1]   (n + m square; node j < n is x_j, node n + i is row i of A)
//
// The pattern of K does not depend on rho or sigma, so this runs once per problem.  It computes:
//   1. a fill-reducing ordering: approximate minimum degree on the quotient graph (Amestoy, Davis, Duff, SIAM J. Matrix
//      Anal. Appl. 17(4), 1996) with element absorption, aggressive absorption, supervariables and mass elimination.
//      Nodes of degree > max(16, 10 sqrt(n + m)) are removed before the ordering and placed last, in index order.
//      Every choice is made on integers in a fixed order (ties of the minimum degree go to the node with fewer dense
//      neighbours, then to the smallest node), so the ordering is deterministic;
//   2. the elimination tree of the permuted K, renumbered in postorder (the ordering returned is AMD's composed with it);
//   3. exact column counts of L (Gilbert, Ng, Peyton, SIAM J. Matrix Anal. Appl. 15(4), 1994: row-subtree leaves with
//      a disjoint-set forest, O(nnz(K) alpha)), so nnz(L) is known without forming the structure;
//   4. fundamental supernodes, then relaxed amalgamation of a supernode with its contiguous last child while the
//      explicit zeros of the merged trapezoid stay within relax_fraction(width) of it;
//   5. the row structure below each supernode, and the sizes the device factor would need.
// No CUDA in here: the analysis runs on a machine without a GPU.
#pragma once

#include <math.h>
#include <stdint.h>

#include <algorithm>
#include <set>
#include <string>
#include <tuple>
#include <utility>
#include <vector>

namespace cosmo {
namespace ldl {

// The fan-in factorisation gathers the updates of a target supernode's descendants into a panel of the target's front
// height and this many columns at a time (DESIGN §3d); the panel is the only workspace that scales with a front.
constexpr int64_t kFanInChunk = 256;

// Amalgamation bound: a merged supernode of `width` columns may hold at most this fraction of explicit zeros in its
// stored trapezoid width (width + 1) / 2 + width * below.
inline double relax_fraction(int64_t width) { return width <= 16 ? 0.5 : (width <= 64 ? 0.2 : 0.05); }

// dense-node rule of the ordering
inline int64_t dense_degree(int64_t N) { return std::max<int64_t>(16, (int64_t)(10.0 * sqrt((double)N))); }

struct Symbolic {
  int64_t N = 0;
  std::vector<int64_t> perm;          // perm[k] = node eliminated k-th (postordered)
  std::vector<int64_t> parent;        // elimination tree in the permuted numbering (-1 at a root)
  std::vector<int64_t> colcount;      // nnz of column k of L, diagonal included
  std::vector<int64_t> sn_first;      // supernode s holds columns sn_first[s] .. sn_first[s + 1] - 1
  std::vector<int64_t> sn_parent;     // supernodal tree (-1 at a root)
  std::vector<int64_t> sn_rowptr;     // rows below supernode s: sn_rows[sn_rowptr[s] .. sn_rowptr[s + 1]), ascending
  std::vector<int64_t> sn_rows;
  int64_t nnz_L = 0, height = 0, widest = 0, largest_front = 0, dense = 0;
  int64_t factor_bytes = 0, workspace_bytes = 0;
};

// ---- approximate minimum degree ---------------------------------------------------------------------------------------
// adj: symmetric pattern without the diagonal, sorted rows.  Returns the elimination order of all N nodes.
inline std::vector<int64_t> amd_order(int64_t N, const std::vector<std::vector<int64_t>>& adj, int64_t* n_dense) {
  enum : char { VAR = 0, MERGED = 1, ELEMENT = 2, DEAD = 3, DENSE = 4 };
  std::vector<char> st(N, VAR);
  const int64_t dthr = dense_degree(N);
  int64_t nd = 0;
  for (int64_t i = 0; i < N; ++i)
    if ((int64_t)adj[i].size() > dthr) { st[i] = DENSE; ++nd; }
  *n_dense = nd;
  std::vector<std::vector<int64_t>> A(N), E(N), Le(N), members(N);
  std::vector<int64_t> nv(N, 1), deg(N, 0), esize(N, 0), w(N, 0), wmark(N, -1), mark(N, -1);
  // (approximate degree, dense neighbours, node).  The dense nodes are out of the graph, but every one next to a node
  // ends up in its column of L: among equal degrees, the node with fewer of them goes first.  (C3: of the chain
  // D_i - x_i, D_i goes first, and x_i's ~k/2 dense F' rows are not copied into D_i's column.)
  std::vector<int64_t> ndense(N, 0);
  typedef std::tuple<int64_t, int64_t, int64_t> Key;
  std::set<Key> pq;
  int64_t nleft = 0;
  for (int64_t i = 0; i < N; ++i) {
    if (st[i] == DENSE) continue;
    for (int64_t j : adj[i])
      if (st[j] != DENSE) A[i].push_back(j);
      else ++ndense[i];
    deg[i] = (int64_t)A[i].size();
    members[i].push_back(i);
    pq.insert(Key(deg[i], ndense[i], i));
    ++nleft;
  }
  std::vector<int64_t> order;
  order.reserve(N);
  int64_t stamp = 0;
  std::vector<int64_t> Lp;
  while (!pq.empty()) {
    const int64_t p = std::get<2>(*pq.begin());
    pq.erase(pq.begin());
    ++stamp;
    // Lp = (A_p U  union of L_e over e in E_p) \ {p}; the elements of E_p are absorbed into p
    Lp.clear();
    mark[p] = stamp;
    for (int64_t i : A[p])
      if (st[i] == VAR && mark[i] != stamp) { mark[i] = stamp; Lp.push_back(i); }
    for (int64_t e : E[p]) {
      if (st[e] != ELEMENT) continue;
      for (int64_t i : Le[e])
        if (st[i] == VAR && mark[i] != stamp) { mark[i] = stamp; Lp.push_back(i); }
      st[e] = DEAD;
      std::vector<int64_t>().swap(Le[e]);
    }
    std::sort(Lp.begin(), Lp.end());
    st[p] = ELEMENT;
    std::vector<int64_t>().swap(A[p]);
    std::vector<int64_t>().swap(E[p]);
    for (int64_t v : members[p]) order.push_back(v);
    nleft -= nv[p];
    int64_t degLp = 0;
    for (int64_t i : Lp) degLp += nv[i];
    // prune: E_i <- live elements + p, A_i <- A_i \ Lp \ {p} (those are reached through p now)
    for (int64_t i : Lp) {
      pq.erase(Key(deg[i], ndense[i], i));
      auto& Ei = E[i];
      size_t k = 0;
      for (int64_t e : Ei)
        if (st[e] == ELEMENT) Ei[k++] = e;
      Ei.resize(k);
      Ei.push_back(p);
      auto& Ai = A[i];
      k = 0;
      for (int64_t j : Ai)
        if (st[j] == VAR && mark[j] != stamp) Ai[k++] = j;
      Ai.resize(k);
    }
    // w(e) = |L_e \ Lp| for the elements next to Lp
    for (int64_t i : Lp)
      for (int64_t e : E[i]) {
        if (e == p) continue;
        if (wmark[e] != stamp) { wmark[e] = stamp; w[e] = esize[e]; }
        w[e] -= nv[i];
      }
    // approximate external degrees; an element inside Lp (w = 0) is absorbed into p (aggressive absorption)
    for (int64_t i : Lp) {
      int64_t d = degLp - nv[i];
      auto& Ei = E[i];
      size_t k = 0;
      for (int64_t e : Ei) {
        if (e != p) {
          if (st[e] != ELEMENT) continue;
          if (w[e] == 0) { st[e] = DEAD; std::vector<int64_t>().swap(Le[e]); continue; }
          d += w[e];
        }
        Ei[k++] = e;
      }
      Ei.resize(k);
      for (int64_t j : A[i]) d += nv[j];
      deg[i] = std::min(d, std::min(deg[i] + degLp - nv[i], nleft - nv[i]));
    }
    // mass elimination: a variable whose only neighbour is element p adds no fill; it is eliminated right after p
    {
      size_t k = 0;
      for (int64_t i : Lp) {
        if (A[i].empty() && E[i].size() == 1) {
          st[i] = DEAD;
          for (int64_t v : members[i]) order.push_back(v);
          nleft -= nv[i];
          degLp -= nv[i];
          std::vector<int64_t>().swap(E[i]);
          continue;
        }
        Lp[k++] = i;
      }
      Lp.resize(k);
    }
    // supervariables: equal (E_i, A_i) -> one variable; candidates share a hash, compared in (hash, node) order
    {
      std::vector<std::pair<uint64_t, int64_t>> h;
      h.reserve(Lp.size());
      for (int64_t i : Lp) {
        uint64_t s = 0;
        for (int64_t e : E[i]) s += (uint64_t)e;
        for (int64_t j : A[i]) s += (uint64_t)j;
        h.push_back({s + (uint64_t)E[i].size() * 0x9E3779B97F4A7C15ull + (uint64_t)A[i].size(), i});
      }
      std::sort(h.begin(), h.end());
      for (size_t a = 0; a < h.size(); ++a) {
        const int64_t i = h[a].second;
        if (st[i] != VAR) continue;
        std::vector<int64_t> Ei(E[i]), Ai(A[i]);
        std::sort(Ei.begin(), Ei.end());
        std::sort(Ai.begin(), Ai.end());
        for (size_t b = a + 1; b < h.size() && h[b].first == h[a].first; ++b) {
          const int64_t j = h[b].second;
          if (st[j] != VAR || E[j].size() != Ei.size() || A[j].size() != Ai.size()) continue;
          std::vector<int64_t> Ej(E[j]), Aj(A[j]);
          std::sort(Ej.begin(), Ej.end());
          std::sort(Aj.begin(), Aj.end());
          if (Ej != Ei || Aj != Ai) continue;
          nv[i] += nv[j];
          deg[i] -= nv[j];
          nv[j] = 0;
          st[j] = MERGED;
          members[i].insert(members[i].end(), members[j].begin(), members[j].end());
          std::vector<int64_t>().swap(members[j]);
          std::vector<int64_t>().swap(A[j]);
          std::vector<int64_t>().swap(E[j]);
        }
      }
    }
    // p becomes an element over the surviving principal variables of Lp
    auto& L = Le[p];
    int64_t sz = 0;
    for (int64_t i : Lp)
      if (st[i] == VAR) { L.push_back(i); sz += nv[i]; }
    esize[p] = sz;
    for (int64_t i : L) {
      deg[i] = std::max<int64_t>(0, std::min(deg[i], nleft - nv[i]));
      pq.insert(Key(deg[i], ndense[i], i));
    }
  }
  for (int64_t i = 0; i < N; ++i)
    if (st[i] == DENSE) order.push_back(i);
  return order;
}

// ---- the whole analysis -------------------------------------------------------------------------------------------------
// Upper-triangle entries of K come from P (either triangle; (i, j) and (j, i) are one edge) and A; the diagonal is always
// present.  Indices are 0-based and validated by the caller.
inline Symbolic analyse(int64_t n, int64_t m, const std::vector<int64_t>& P_colptr, const std::vector<int64_t>& P_row,
                        const std::vector<int64_t>& A_colptr, const std::vector<int64_t>& A_row) {
  Symbolic S;
  const int64_t N = n + m;
  S.N = N;
  std::vector<std::vector<int64_t>> adj(N);
  for (int64_t j = 0; j < n; ++j) {
    for (int64_t k = P_colptr[j]; k < P_colptr[j + 1]; ++k) {
      const int64_t i = P_row[k];
      if (i != j) { adj[i].push_back(j); adj[j].push_back(i); }
    }
    for (int64_t k = A_colptr[j]; k < A_colptr[j + 1]; ++k) {
      const int64_t i = n + A_row[k];
      adj[i].push_back(j);
      adj[j].push_back(i);
    }
  }
  for (auto& a : adj) {
    std::sort(a.begin(), a.end());
    a.erase(std::unique(a.begin(), a.end()), a.end());
  }
  std::vector<int64_t> order = amd_order(N, adj, &S.dense);

  // elimination tree of the permuted matrix (Liu: ancestors with path compression)
  std::vector<int64_t> pinv(N), parent(N, -1), anc(N, -1);
  for (int64_t k = 0; k < N; ++k) pinv[order[k]] = k;
  for (int64_t k = 0; k < N; ++k)
    for (int64_t v : adj[order[k]]) {
      int64_t i = pinv[v];
      while (i != -1 && i < k) {
        const int64_t next = anc[i];
        anc[i] = k;
        if (next == -1) parent[i] = k;
        i = next;
      }
    }
  // postorder: children in ascending order, roots in ascending order
  std::vector<int64_t> head(N, -1), next(N, -1), post;
  post.reserve(N);
  for (int64_t j = N - 1; j >= 0; --j)
    if (parent[j] != -1) { next[j] = head[parent[j]]; head[parent[j]] = j; }
  {
    std::vector<int64_t> stack;
    for (int64_t r = 0; r < N; ++r) {
      if (parent[r] != -1) continue;
      stack.push_back(r);
      while (!stack.empty()) {
        const int64_t j = stack.back();
        if (head[j] != -1) { const int64_t c = head[j]; head[j] = next[c]; stack.push_back(c); }
        else { stack.pop_back(); post.push_back(j); }
      }
    }
  }
  S.perm.resize(N);
  std::vector<int64_t> postinv(N);
  for (int64_t k = 0; k < N; ++k) { S.perm[k] = order[post[k]]; postinv[post[k]] = k; }
  for (int64_t k = 0; k < N; ++k) pinv[S.perm[k]] = k;
  S.parent.assign(N, -1);
  for (int64_t k = 0; k < N; ++k) {
    const int64_t p = parent[post[k]];
    S.parent[k] = p == -1 ? -1 : postinv[p];
  }
  const auto& par = S.parent;
  // lower pattern of column j of the permuted K: rows i > j
  std::vector<int64_t> lp(N + 1, 0), li;
  for (int64_t j = 0; j < N; ++j) {
    for (int64_t v : adj[S.perm[j]])
      if (pinv[v] > j) li.push_back(pinv[v]);
    std::sort(li.begin() + lp[j], li.end());
    lp[j + 1] = (int64_t)li.size();
  }
  std::vector<std::vector<int64_t>>().swap(adj);

  // column counts (postordered: first descendants are plain column indices)
  std::vector<int64_t> first(N, -1), maxfirst(N, -1), prevleaf(N, -1), ancestor(N), delta(N, 0);
  for (int64_t k = 0; k < N; ++k) {
    delta[k] = first[k] == -1 ? 1 : 0;
    for (int64_t j = k; j != -1 && first[j] == -1; j = par[j]) first[j] = k;
  }
  for (int64_t i = 0; i < N; ++i) ancestor[i] = i;
  for (int64_t j = 0; j < N; ++j) {
    if (par[j] != -1) --delta[par[j]];
    for (int64_t t = lp[j]; t < lp[j + 1]; ++t) {
      const int64_t i = li[t];   // j is in the row subtree of i; is it a new leaf of it?
      if (first[j] <= maxfirst[i]) continue;
      maxfirst[i] = first[j];
      const int64_t jprev = prevleaf[i];
      prevleaf[i] = j;
      ++delta[j];
      if (jprev == -1) continue;
      int64_t q = jprev;
      while (q != ancestor[q]) q = ancestor[q];
      for (int64_t s = jprev; s != q;) { const int64_t sp = ancestor[s]; ancestor[s] = q; s = sp; }
      --delta[q];
    }
    if (par[j] != -1) ancestor[j] = par[j];
  }
  for (int64_t j = 0; j < N; ++j)
    if (par[j] != -1) delta[par[j]] += delta[j];
  S.colcount = delta;
  for (int64_t j = 0; j < N; ++j) S.nnz_L += S.colcount[j];

  // fundamental supernodes, then relaxed amalgamation with the contiguous last child
  std::vector<int64_t> nchild(N, 0);
  for (int64_t j = 0; j < N; ++j)
    if (par[j] != -1) ++nchild[par[j]];
  struct Node { int64_t first, last, exact, parent_last; };   // parent_last: last column of the parent's fundamental node
  std::vector<Node> stack;
  std::vector<int64_t> fund_last(N);   // column -> last column of its fundamental supernode
  {
    int64_t f = 0;
    for (int64_t j = 0; j < N; ++j) {
      const bool join = j + 1 < N && par[j] == j + 1 && nchild[j + 1] == 1 && S.colcount[j] == S.colcount[j + 1] + 1;
      if (join) continue;
      for (int64_t c = f; c <= j; ++c) fund_last[c] = j;
      f = j + 1;
    }
  }
  for (int64_t f = 0; f < N;) {
    const int64_t l = fund_last[f];
    Node cur{f, l, 0, par[l] == -1 ? -1 : fund_last[par[l]]};
    for (int64_t c = f; c <= l; ++c) cur.exact += S.colcount[c];
    const int64_t below = S.colcount[l] - 1;
    // a candidate is the node just below cur whose parent lies inside cur (a child of s, or of a child merged already)
    while (!stack.empty() && stack.back().last == cur.first - 1 && stack.back().parent_last >= cur.first &&
           stack.back().parent_last <= l) {
      const Node& c = stack.back();
      const int64_t k = l - c.first + 1;
      const int64_t stored = k * (k + 1) / 2 + k * below;
      const int64_t zeros = stored - (cur.exact + c.exact);
      if ((double)zeros > relax_fraction(k) * (double)stored) break;
      cur.first = c.first;
      cur.exact += c.exact;
      stack.pop_back();
    }
    stack.push_back(cur);
    f = l + 1;
  }
  const int64_t ns = (int64_t)stack.size();
  S.sn_first.resize(ns + 1);
  std::vector<int64_t> sn_of(N);
  for (int64_t s = 0; s < ns; ++s) {
    S.sn_first[s] = stack[s].first;
    for (int64_t c = stack[s].first; c <= stack[s].last; ++c) sn_of[c] = s;
  }
  S.sn_first[ns] = N;
  S.sn_parent.assign(ns, -1);
  for (int64_t s = 0; s < ns; ++s) {
    const int64_t p = par[S.sn_first[s + 1] - 1];
    S.sn_parent[s] = p == -1 ? -1 : sn_of[p];
  }
  // row structure below each supernode: K's rows below it plus its children's rows below it (children come first)
  std::vector<std::vector<int64_t>> rows(ns);
  std::vector<int64_t> rmark(N, -1);
  std::vector<std::vector<int64_t>> kids(ns);
  for (int64_t s = 0; s < ns; ++s)
    if (S.sn_parent[s] != -1) kids[S.sn_parent[s]].push_back(s);
  S.sn_rowptr.assign(ns + 1, 0);
  std::vector<int64_t> depth(ns, 1);
  for (int64_t s = 0; s < ns; ++s) {
    const int64_t f = S.sn_first[s], l = S.sn_first[s + 1] - 1;
    auto& R = rows[s];
    for (int64_t j = f; j <= l; ++j)
      for (int64_t t = lp[j]; t < lp[j + 1]; ++t)
        if (li[t] > l && rmark[li[t]] != s) { rmark[li[t]] = s; R.push_back(li[t]); }
    for (int64_t c : kids[s]) {
      for (int64_t i : rows[c])
        if (i > l && rmark[i] != s) { rmark[i] = s; R.push_back(i); }
      std::vector<int64_t>().swap(rows[c]);
    }
    std::sort(R.begin(), R.end());
    const int64_t k = l - f + 1, r = (int64_t)R.size();
    S.sn_rowptr[s + 1] = S.sn_rowptr[s] + r;
    S.sn_rows.insert(S.sn_rows.end(), R.begin(), R.end());
    S.widest = std::max(S.widest, k);
    S.largest_front = std::max(S.largest_front, k + r);
    S.factor_bytes += 8 * (k + r) * k;
  }
  for (int64_t s = ns - 1; s >= 0; --s)
    if (S.sn_parent[s] != -1) depth[s] = depth[S.sn_parent[s]] + 1;
  for (int64_t s = 0; s < ns; ++s) S.height = std::max(S.height, depth[s]);
  // workspace: the fan-in panel (largest front x kFanInChunk), the solve's two vectors, and one int64 factor position per
  // stored entry of P's upper triangle, A and the two diagonals (the scatter map of a refactorisation)
  int64_t p_upper = 0;
  for (int64_t j = 0; j < n; ++j)
    for (int64_t k = P_colptr[j]; k < P_colptr[j + 1]; ++k)
      if (P_row[k] <= j) ++p_upper;
  S.workspace_bytes = 8 * S.largest_front * kFanInChunk + 16 * N + 8 * (p_upper + A_colptr[n] + N);
  return S;
}

}  // namespace ldl
}  // namespace cosmo
