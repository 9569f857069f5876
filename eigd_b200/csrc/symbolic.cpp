// Symbolic analysis: supervariable compression, nested dissection (geometric when node
// coordinates are supplied, BFS level-set otherwise), elimination tree, postorder, column
// counts, supernode partition (collapsed leaf subtrees + fundamental chains + relaxed
// amalgamation + width cap), front row structures, child->parent relative indices, levels.
//
// The reference has no counterpart (SuperLU/COLAMD inside scipy splu,
// eigd/eigenvector_derivatives.py:13); results are pinned against oracle/multifrontal_oracle.py (tests/test_symbolic_cpu.py).
#include "symbolic.hpp"
#include "../../include/eigd_b200.h"

#include <algorithm>
#include <cstdlib>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <set>
#include <numeric>
#include <string>

static thread_local std::string g_err;
void eigd_set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
}
extern "C" const char* eigd_last_error(void) { return g_err.c_str(); }
extern "C" int eigd_version(void) { return 100; }

namespace {

struct Graph {
  int nv = 0;
  std::vector<int64_t> ptr;
  std::vector<int> adj;
  std::vector<int> wgt;  // vertex weights (#dofs merged)
};

// ---- adjacency of the symmetrised pattern without the diagonal ------------------------
Graph build_graph(int n, const int* indptr, const int* indices) {
  Graph g;
  g.nv = n;
  std::vector<int64_t> cnt(n + 1, 0);
  for (int r = 0; r < n; ++r)
    for (int p = indptr[r]; p < indptr[r + 1]; ++p) {
      int c = indices[p];
      if (c == r) continue;
      cnt[r + 1]++;
      cnt[c + 1]++;
    }
  for (int i = 0; i < n; ++i) cnt[i + 1] += cnt[i];
  std::vector<int> tmp(cnt[n]);
  std::vector<int64_t> pos(cnt.begin(), cnt.end() - 1);
  for (int r = 0; r < n; ++r)
    for (int p = indptr[r]; p < indptr[r + 1]; ++p) {
      int c = indices[p];
      if (c == r) continue;
      tmp[pos[r]++] = c;
      tmp[pos[c]++] = r;
    }
  // sort + unique each list
  g.ptr.assign(n + 1, 0);
  g.adj.reserve(cnt[n] / 2 + n);
  for (int r = 0; r < n; ++r) {
    auto b = tmp.begin() + cnt[r], e = tmp.begin() + cnt[r + 1];
    std::sort(b, e);
    e = std::unique(b, e);
    g.adj.insert(g.adj.end(), b, e);
    g.ptr[r + 1] = (int64_t)g.adj.size();
  }
  g.wgt.assign(n, 1);
  return g;
}

// ---- supervariables: vertices with identical closed neighbourhoods ---------------------
// returns map vertex -> supervertex and the compressed graph
Graph compress_graph(const Graph& g, std::vector<int>& v2s, std::vector<std::vector<int>>& members) {
  int n = g.nv;
  std::vector<uint64_t> h(n);
  auto hv = [](int u) { uint64_t x = (uint64_t)(u + 1) * 0x9E3779B97F4A7C15ull; x ^= x >> 29; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 32; return x; };
  for (int v = 0; v < n; ++v) {
    uint64_t x = hv(v);  // commutative hash of the closed neighbourhood
    for (int64_t p = g.ptr[v]; p < g.ptr[v + 1]; ++p) x += hv(g.adj[p]);
    h[v] = x;
  }
  auto same = [&](int a, int b) {
    // a, b adjacent: closed neighbourhoods are equal iff N(a)\{b} == N(b)\{a}
    if (g.ptr[a + 1] - g.ptr[a] != g.ptr[b + 1] - g.ptr[b]) return false;
    int64_t pa = g.ptr[a], pb = g.ptr[b], ea = g.ptr[a + 1], eb = g.ptr[b + 1];
    while (true) {
      if (pa < ea && g.adj[pa] == b) ++pa;
      if (pb < eb && g.adj[pb] == a) ++pb;
      if (pa >= ea || pb >= eb) return pa >= ea && pb >= eb;
      if (g.adj[pa] != g.adj[pb]) return false;
      ++pa; ++pb;
    }
  };
  v2s.assign(n, -1);
  members.clear();
  // only neighbours can share a closed neighbourhood
  for (int v = 0; v < n; ++v) {
    if (v2s[v] >= 0) continue;
    int s = (int)members.size();
    members.emplace_back();
    members[s].push_back(v);
    v2s[v] = s;
    for (int64_t p = g.ptr[v]; p < g.ptr[v + 1]; ++p) {
      int u = g.adj[p];
      if (u > v && v2s[u] < 0 && h[u] == h[v] && same(v, u)) {
        v2s[u] = s;
        members[s].push_back(u);
      }
    }
  }
  Graph c;
  c.nv = (int)members.size();
  c.ptr.assign(c.nv + 1, 0);
  c.wgt.resize(c.nv);
  std::vector<int> mark(c.nv, -1);
  for (int s = 0; s < c.nv; ++s) {
    c.wgt[s] = (int)members[s].size();
    int v = members[s][0];  // all members share the neighbourhood
    mark[s] = s;
    size_t start = c.adj.size();
    for (int64_t p = g.ptr[v]; p < g.ptr[v + 1]; ++p) {
      int t = v2s[g.adj[p]];
      if (mark[t] != s) { mark[t] = s; c.adj.push_back(t); }
    }
    std::sort(c.adj.begin() + start, c.adj.end());
    c.ptr[s + 1] = (int64_t)c.adj.size();
  }
  return c;
}

// ---- nested dissection ------------------------------------------------------------------
struct NDContext {
  const Graph& g;
  const double* xy;  // per supervertex coordinates (dim values) or null
  int dim;
  int nd_leaf;
  std::vector<int> stamp;  // membership stamps
  std::vector<int> dist;
  std::vector<int> order;  // output: elimination order of supervertices
  int cur_stamp = 0;
  NDContext(const Graph& g_, const double* xy_, int dim_, int leaf) : g(g_), xy(xy_), dim(dim_), nd_leaf(leaf) {
    stamp.assign(g.nv, 0);
    dist.assign(g.nv, -1);
  }
};

// BFS inside the subset marked with stamp == tag; returns visit order, fills dist
static void bfs(NDContext& c, int root, int tag, std::vector<int>& out) {
  out.clear();
  out.push_back(root);
  c.dist[root] = 0;
  for (size_t h = 0; h < out.size(); ++h) {
    int v = out[h];
    for (int64_t p = c.g.ptr[v]; p < c.g.ptr[v + 1]; ++p) {
      int u = c.g.adj[p];
      if (c.stamp[u] == tag && c.dist[u] < 0) {
        c.dist[u] = c.dist[v] + 1;
        out.push_back(u);
      }
    }
  }
}

// Split S (connected, stamped with tag) into A, B, Sep. Returns false if no useful split.
static bool bisect_graph(NDContext& c, const std::vector<int>& S, int tag, std::vector<int>& A,
                         std::vector<int>& B, std::vector<int>& Sep) {
  std::vector<int> q;
  int root = S[0];
  int lastdepth = -1;
  for (int it = 0; it < 4; ++it) {
    for (int v : S) c.dist[v] = -1;
    bfs(c, root, tag, q);
    int far = q.back();
    int depth = c.dist[far];
    if (depth <= lastdepth) break;
    lastdepth = depth;
    // among the deepest level choose the vertex of smallest degree
    int best = far;
    int64_t bestdeg = c.g.ptr[far + 1] - c.g.ptr[far];
    for (size_t i = q.size(); i-- > 0;) {
      int v = q[i];
      if (c.dist[v] != depth) break;
      int64_t d = c.g.ptr[v + 1] - c.g.ptr[v];
      if (d < bestdeg) { bestdeg = d; best = v; }
    }
    if (it == 3) break;
    root = best;
  }
  for (int v : S) c.dist[v] = -1;
  bfs(c, root, tag, q);
  int nl = c.dist[q.back()] + 1;
  if (nl < 3) return false;
  std::vector<int64_t> lw(nl, 0);
  int64_t tot = 0;
  for (int v : q) { lw[c.dist[v]] += c.g.wgt[v]; tot += c.g.wgt[v]; }
  int64_t acc = 0;
  int best = -1;
  double bestscore = 1e300;
  for (int l = 0; l < nl; ++l) {
    int64_t left = acc, right = tot - acc - lw[l];
    acc += lw[l];
    if (l == 0 || l == nl - 1) continue;
    double bal = (double)std::min(left, right) / (double)std::max<int64_t>(1, std::max(left, right));
    if (bal < 0.4) continue;
    double score = (double)lw[l] * (1.0 + 0.3 * (1.0 - bal));
    if (score < bestscore) { bestscore = score; best = l; }
  }
  if (best < 0) {  // no balanced level: take the weighted median level
    acc = 0;
    for (int l = 0; l < nl; ++l) {
      acc += lw[l];
      if (2 * acc >= tot) { best = std::min(std::max(l, 1), nl - 2); break; }
    }
  }
  A.clear(); B.clear(); Sep.clear();
  for (int v : q) {
    int d = c.dist[v];
    if (d < best) A.push_back(v);
    else if (d > best) B.push_back(v);
    else {
      // thin the separator: a level vertex with no neighbour in the next level joins A
      bool touchesB = false;
      for (int64_t p = c.g.ptr[v]; p < c.g.ptr[v + 1]; ++p) {
        int u = c.g.adj[p];
        if (c.stamp[u] == tag && c.dist[u] == best + 1) { touchesB = true; break; }
      }
      if (touchesB) Sep.push_back(v); else A.push_back(v);
    }
  }
  return !A.empty() && !B.empty();
}

static bool bisect_geometric(NDContext& c, const std::vector<int>& S, int tag, std::vector<int>& A,
                             std::vector<int>& B, std::vector<int>& Sep) {
  int dim = c.dim;
  double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
  for (int v : S)
    for (int d = 0; d < dim; ++d) {
      double x = c.xy[(int64_t)v * dim + d];
      lo[d] = std::min(lo[d], x);
      hi[d] = std::max(hi[d], x);
    }
  int axes[3] = {0, 1, 2};
  std::sort(axes, axes + dim, [&](int a, int b) { return (hi[a] - lo[a]) > (hi[b] - lo[b]); });
  std::vector<double> vals(S.size());
  for (int ai = 0; ai < dim; ++ai) {
    int ax = axes[ai];
    if (!(hi[ax] > lo[ax])) continue;
    for (size_t i = 0; i < S.size(); ++i) vals[i] = c.xy[(int64_t)S[i] * dim + ax];
    std::vector<double> tmp(vals);
    std::nth_element(tmp.begin(), tmp.begin() + tmp.size() / 2, tmp.end());
    double thr = tmp[tmp.size() / 2];
    // left: x < thr, right: x >= thr; make sure left is non-empty
    size_t nleft = 0;
    for (double x : vals) nleft += (x < thr);
    if (nleft == 0) {
      // threshold equals the minimum: split above it instead
      double nxt = 1e300;
      for (double x : vals) if (x > thr) nxt = std::min(nxt, x);
      if (nxt == 1e300) continue;
      thr = nxt;
      nleft = 0;
      for (double x : vals) nleft += (x < thr);
    }
    if (nleft == 0 || nleft == S.size()) continue;
    // side flag in dist: 0 = left, 1 = right
    for (size_t i = 0; i < S.size(); ++i) c.dist[S[i]] = (vals[i] < thr) ? 0 : 1;
    // candidate separators: right vertices touching left, or left vertices touching right
    int64_t wR = 0, wL = 0;
    std::vector<char> bR(S.size(), 0), bL(S.size(), 0);
    for (size_t i = 0; i < S.size(); ++i) {
      int v = S[i];
      int side = c.dist[v];
      for (int64_t p = c.g.ptr[v]; p < c.g.ptr[v + 1]; ++p) {
        int u = c.g.adj[p];
        if (c.stamp[u] == tag && c.dist[u] == 1 - side) {
          if (side) { bR[i] = 1; wR += c.g.wgt[v]; } else { bL[i] = 1; wL += c.g.wgt[v]; }
          break;
        }
      }
    }
    bool useR = (wR <= wL);
    A.clear(); B.clear(); Sep.clear();
    for (size_t i = 0; i < S.size(); ++i) {
      int v = S[i];
      int side = c.dist[v];
      bool insep = useR ? (bR[i] != 0) : (bL[i] != 0);
      if (insep) Sep.push_back(v);
      else if (side == 0) A.push_back(v);
      else B.push_back(v);
    }
    if (!A.empty() && !B.empty()) return true;
  }
  return false;
}

static void nested_dissection(NDContext& c) {
  int nv = c.g.nv;
  c.order.clear();
  c.order.reserve(nv);
  // work stack of (subset, emit-after list); separators are emitted after both halves, so we
  // build the order back to front: process a subset by placing its separator at the END of
  // its output range.
  std::vector<int> out(nv, -1);
  struct Job { std::vector<int> S; int64_t begin; };  // S occupies out[begin, begin+|S|)
  std::vector<Job> stack;
  {
    Job j;
    j.S.resize(nv);
    std::iota(j.S.begin(), j.S.end(), 0);
    j.begin = 0;
    stack.push_back(std::move(j));
  }
  std::vector<int> q, A, B, Sep;
  while (!stack.empty()) {
    Job job = std::move(stack.back());
    stack.pop_back();
    std::vector<int>& S = job.S;
    if (S.empty()) continue;
    int tag = ++c.cur_stamp;
    for (int v : S) { c.stamp[v] = tag; c.dist[v] = -1; }
    // connected components
    bfs(c, S[0], tag, q);
    if (q.size() < S.size()) {
      // split into components, each becomes an independent job laid out consecutively
      int64_t pos = job.begin;
      std::vector<int> comp(q);
      while (true) {
        Job cj;
        cj.S = comp;
        cj.begin = pos;
        pos += (int64_t)comp.size();
        stack.push_back(std::move(cj));
        int next = -1;
        for (int v : S) if (c.dist[v] < 0) { next = v; break; }
        if (next < 0) break;
        bfs(c, next, tag, comp);
      }
      continue;
    }
    bool leaf = (int)S.size() <= c.nd_leaf;
    bool ok = false;
    if (!leaf) {
      ok = c.xy ? bisect_geometric(c, S, tag, A, B, Sep) : bisect_graph(c, S, tag, A, B, Sep);
      if (!ok && c.xy) ok = bisect_graph(c, S, tag, A, B, Sep);
    }
    if (!ok) {
      // leaf: BFS order from the first vertex (q holds it if still valid)
      for (int v : S) c.dist[v] = -1;
      bfs(c, S[0], tag, q);
      for (size_t i = 0; i < q.size(); ++i) out[job.begin + (int64_t)i] = q[i];
      continue;
    }
    int64_t pa = job.begin, pb = pa + (int64_t)A.size(), ps = pb + (int64_t)B.size();
    for (size_t i = 0; i < Sep.size(); ++i) out[ps + (int64_t)i] = Sep[i];
    Job ja, jb;
    ja.S = A; ja.begin = pa;
    jb.S = B; jb.begin = pb;
    stack.push_back(std::move(ja));
    stack.push_back(std::move(jb));
  }
  c.order = out;
}

// ---- lower-triangular pattern of the permuted matrix, by column (rows > col) -------------
struct LowerPattern {
  std::vector<int64_t> ptr;
  std::vector<int> rows;
};
static LowerPattern build_lower(int n, const int* indptr, const int* indices, const std::vector<int>& iperm) {
  LowerPattern L;
  L.ptr.assign(n + 1, 0);
  for (int r = 0; r < n; ++r)
    for (int p = indptr[r]; p < indptr[r + 1]; ++p) {
      int pr = iperm[r], pc = iperm[indices[p]];
      if (pr == pc) continue;
      int lo = std::min(pr, pc);
      L.ptr[lo + 1]++;
    }
  for (int i = 0; i < n; ++i) L.ptr[i + 1] += L.ptr[i];
  std::vector<int> tmp(L.ptr[n]);
  std::vector<int64_t> pos(L.ptr.begin(), L.ptr.end() - 1);
  for (int r = 0; r < n; ++r)
    for (int p = indptr[r]; p < indptr[r + 1]; ++p) {
      int pr = iperm[r], pc = iperm[indices[p]];
      if (pr == pc) continue;
      int lo = std::min(pr, pc), hi = std::max(pr, pc);
      tmp[pos[lo]++] = hi;
    }
  // unique per column (both (r,c) and (c,r) are usually stored)
  std::vector<int64_t> nptr(n + 1, 0);
  L.rows.reserve(tmp.size() / 2 + 1);
  for (int j = 0; j < n; ++j) {
    auto b = tmp.begin() + L.ptr[j], e = tmp.begin() + L.ptr[j + 1];
    std::sort(b, e);
    e = std::unique(b, e);
    L.rows.insert(L.rows.end(), b, e);
    nptr[j + 1] = (int64_t)L.rows.size();
  }
  L.ptr.swap(nptr);
  return L;
}

// Liu's elimination tree from the by-column lower pattern (column j lists rows i > j):
// equivalent to processing, for each row i, its columns j < i.  We need the by-row view, so
// transpose once.
static void etree_and_counts(int n, const LowerPattern& L, std::vector<int>& parent, std::vector<int>& count) {
  // by-row view: for each i the columns j < i
  std::vector<int64_t> rptr(n + 1, 0);
  for (int j = 0; j < n; ++j)
    for (int64_t p = L.ptr[j]; p < L.ptr[j + 1]; ++p) rptr[L.rows[p] + 1]++;
  for (int i = 0; i < n; ++i) rptr[i + 1] += rptr[i];
  std::vector<int> rcol(rptr[n]);
  {
    std::vector<int64_t> pos(rptr.begin(), rptr.end() - 1);
    for (int j = 0; j < n; ++j)
      for (int64_t p = L.ptr[j]; p < L.ptr[j + 1]; ++p) rcol[pos[L.rows[p]]++] = j;
  }
  parent.assign(n, -1);
  std::vector<int> anc(n, -1);
  for (int i = 0; i < n; ++i)
    for (int64_t p = rptr[i]; p < rptr[i + 1]; ++p) {
      int j = rcol[p];
      while (j != -1 && j < i) {
        int nx = anc[j];
        anc[j] = i;
        if (nx == -1) parent[j] = i;
        j = nx;
      }
    }
  count.assign(n, 0);
  std::vector<int> mark(n, -1);
  for (int i = 0; i < n; ++i) {
    mark[i] = i;
    for (int64_t p = rptr[i]; p < rptr[i + 1]; ++p) {
      int k = rcol[p];
      while (k != -1 && mark[k] != i) {
        count[k]++;
        mark[k] = i;
        k = parent[k];
      }
    }
  }
}

static std::vector<int> postorder(int n, const std::vector<int>& parent) {
  std::vector<int> head(n, -1), next(n, -1);
  for (int j = n - 1; j >= 0; --j)
    if (parent[j] >= 0) { next[j] = head[parent[j]]; head[parent[j]] = j; }
  std::vector<int> post;
  post.reserve(n);
  std::vector<int> stack;
  for (int r = 0; r < n; ++r) {
    if (parent[r] >= 0) continue;
    stack.push_back(r);
    while (!stack.empty()) {
      int v = stack.back();
      int c = head[v];
      if (c >= 0) { head[v] = next[c]; stack.push_back(c); }
      else { post.push_back(v); stack.pop_back(); }
    }
  }
  return post;
}

}  // namespace

// Offsets of the fronts in the pooled front workspace.  Front k is live from its own level (assembly, factorisation,
// inverse and solve panels) through its parent's level (extend-add of its contribution block); a root only at its own
// level.  Fronts are placed level by level, best fit (smallest free block that holds the front, lowest offset among
// equals) after the fronts whose last level has passed are released, so no two fronts live at the same level share
// memory; in particular a child and its parent never do.  Sizes are rounded up to 256 bytes.
static void pool_layout(eigd_symbolic* S) {
  const int ns = S->nsuper;
  S->pool_off.assign(ns, 0);
  std::vector<std::vector<int>> dies(S->nlevels + 1);   // fronts released before level l + 1
  for (int k = 0; k < ns; ++k) {
    int p = S->sn_parent[k];
    dies[p >= 0 ? S->sn_level[p] : S->sn_level[k]].push_back(k);
  }
  std::map<int64_t, int64_t> free_at;                    // offset -> size of every free block below the top
  std::set<std::pair<int64_t, int64_t>> by_size;         // (size, offset) of the same blocks
  int64_t top = 0, peak = 0;
  auto size_of = [&](int k) { int64_t f = sn_fsize(S, k); return (f * f + 31) / 32 * 32; };
  auto release = [&](int64_t off, int64_t sz) {
    auto nx = free_at.lower_bound(off);
    if (nx != free_at.end() && nx->first == off + sz) { sz += nx->second; by_size.erase({nx->second, nx->first}); nx = free_at.erase(nx); }
    if (nx != free_at.begin()) {
      auto pv = std::prev(nx);
      if (pv->first + pv->second == off) { off = pv->first; sz += pv->second; by_size.erase({pv->second, pv->first}); free_at.erase(pv); }
    }
    if (off + sz == top) { top = off; return; }          // the block reaches the top: the used region shrinks
    free_at[off] = sz;
    by_size.insert({sz, off});
  };
  for (int l = 0; l < S->nlevels; ++l) {
    if (l > 0)
      for (int k : dies[l - 1]) release(S->pool_off[k], size_of(k));
    for (int q = S->level_ptr[l]; q < S->level_ptr[l + 1]; ++q) {
      const int k = S->level_sn[q];
      const int64_t sz = size_of(k);
      auto it = by_size.lower_bound({sz, INT64_MIN});
      if (it == by_size.end()) {
        S->pool_off[k] = top;
        top += sz;
        peak = std::max(peak, top);
        continue;
      }
      const int64_t off = it->second, bsz = it->first;
      by_size.erase(it);
      free_at.erase(off);
      S->pool_off[k] = off;
      if (bsz > sz) { free_at[off + sz] = bsz - sz; by_size.insert({bsz - sz, off + sz}); }
    }
  }
  S->pool_doubles = peak;
}

extern "C" int eigd_symbolic_create(int n, const int* indptr, const int* indices, const double* coords,
                                    int dim, int dof_per_node, const int* opts, eigd_symbolic** out) {
  if (n <= 0 || !indptr || !indices || !out) { eigd_set_error("symbolic_create: bad arguments"); return 1; }
  if (coords && (dim < 1 || dim > 3 || dof_per_node < 1 || n % dof_per_node)) {
    eigd_set_error("symbolic_create: bad coords spec (dim=%d dof_per_node=%d n=%d)", dim, dof_per_node, n);
    return 1;
  }
  auto* S = new eigd_symbolic();
  S->n = n;
  if (opts) {
    if (opts[0] > 0) S->leaf_cols = opts[0];
    if (opts[1] > 0) S->max_super_cols = opts[1];
    if (opts[2] > 0) S->nd_leaf = opts[2];
    if (opts[3] >= 0) S->relax = opts[3];
  }
  if (const char* e = getenv("EIGD_MAX_SUPER_COLS")) S->max_super_cols = atoi(e);   // developer override (tuning runs)
  if (S->max_super_cols > 512) S->max_super_cols = 512;  // widest pivot block the factor kernels handle (factor.cu)
  if (S->leaf_cols > S->max_super_cols) S->leaf_cols = S->max_super_cols;

  // ---- ordering ---------------------------------------------------------------------
  {
    Graph g = build_graph(n, indptr, indices);
    std::vector<int> v2s;
    std::vector<std::vector<int>> members;
    Graph cg = compress_graph(g, v2s, members);
    std::vector<double> sxy;
    if (coords) {
      sxy.resize((size_t)cg.nv * dim);
      for (int s = 0; s < cg.nv; ++s) {
        int node = members[s][0] / dof_per_node;
        for (int d = 0; d < dim; ++d) sxy[(size_t)s * dim + d] = coords[(size_t)node * dim + d];
      }
    }
    NDContext ctx(cg, coords ? sxy.data() : nullptr, dim, S->nd_leaf);
    nested_dissection(ctx);
    S->perm.clear();
    S->perm.reserve(n);
    for (int s : ctx.order)
      for (int v : members[s]) S->perm.push_back(v);
    if ((int)S->perm.size() != n) { eigd_set_error("symbolic: ordering lost vertices"); delete S; return 2; }
  }
  S->iperm.assign(n, -1);
  for (int k = 0; k < n; ++k) S->iperm[S->perm[k]] = k;
  for (int k = 0; k < n; ++k) if (S->iperm[k] < 0) { eigd_set_error("symbolic: perm is not a permutation"); delete S; return 2; }

  // ---- etree, postorder, counts ---------------------------------------------------------
  LowerPattern L = build_lower(n, indptr, indices, S->iperm);
  {
    std::vector<int> par, cnt;
    etree_and_counts(n, L, par, cnt);
    std::vector<int> post = postorder(n, par);
    std::vector<int> np(n);
    for (int k = 0; k < n; ++k) np[k] = S->perm[post[k]];
    S->perm.swap(np);
    for (int k = 0; k < n; ++k) S->iperm[S->perm[k]] = k;
    L = build_lower(n, indptr, indices, S->iperm);
    etree_and_counts(n, L, S->parent, S->colcount);
  }
  const std::vector<int>& parent = S->parent;
  const std::vector<int>& count = S->colcount;
  for (int j = 0; j < n; ++j)
    if (parent[j] != -1 && parent[j] <= j) { eigd_set_error("symbolic: etree not postordered"); delete S; return 2; }
  S->exact_nnzL = 0;
  for (int j = 0; j < n; ++j) S->exact_nnzL += count[j];

  // ---- supernode partition ---------------------------------------------------------------
  std::vector<int> sz(n, 1), nchild(n, 0);
  for (int j = 0; j < n; ++j)
    if (parent[j] >= 0) { sz[parent[j]] += sz[j]; nchild[parent[j]]++; }
  // start[j] = 1 if a supernode starts at column j
  std::vector<char> start(n, 1);
  std::vector<char> collapsed(n, 0);
  for (int j = 0; j < n; ++j) {
    bool root_of_collapse = sz[j] <= S->leaf_cols && sz[j] > 1 && (parent[j] == -1 || sz[parent[j]] > S->leaf_cols);
    if (root_of_collapse)
      for (int c = j - sz[j] + 1; c <= j; ++c) { collapsed[c] = 1; start[c] = (c == j - sz[j] + 1); }
  }
  for (int j = 1; j < n; ++j) {
    if (collapsed[j]) continue;
    if (collapsed[j - 1]) continue;  // a chain never extends a collapsed subtree here (relaxation may)
    if (parent[j - 1] == j && count[j - 1] == count[j] + 1 && nchild[j] == 1) start[j] = 0;
  }
  struct SN { int first, last; int64_t zeros; };
  std::vector<SN> sns;
  for (int j = 0; j < n; ++j) {
    if (start[j]) sns.push_back({j, j, 0});
    else sns.back().last = j;
  }
  // explicit zeros of collapsed subtrees
  for (auto& s : sns) {
    if (!collapsed[s.first]) continue;
    int64_t nc = s.last - s.first + 1, nb = count[s.last];
    int64_t dense = nc * (nc - 1) / 2 + nc * nb, exact = 0;
    for (int c = s.first; c <= s.last; ++c) exact += count[c];
    s.zeros = dense - exact;
  }
  if (S->relax) {
    std::vector<SN> merged;
    for (size_t k = 0; k < sns.size(); ++k) {
      SN cur = sns[k];
      // try to absorb the previous (already merged) supernode if cur is its parent
      while (!merged.empty()) {
        SN& prev = merged.back();
        if (prev.last + 1 != cur.first || parent[prev.last] < cur.first || parent[prev.last] > cur.last) break;
        int64_t n1 = prev.last - prev.first + 1, n2 = cur.last - cur.first + 1;
        int64_t c1 = count[prev.last], c2 = count[cur.last];
        int64_t nn = n1 + n2;
        if (nn > S->max_super_cols) break;
        int64_t newz = prev.zeros + cur.zeros + n1 * (n2 + c2 - c1);
        int64_t total = nn * (nn + 1) / 2 + nn * c2;
        double z = (double)newz / (double)std::max<int64_t>(1, total);
        bool ok = (nn <= 4) || (nn <= 16 && z < 0.8) || (nn <= 48 && z < 0.1) || (z < 0.05);
        if (!ok) break;
        cur.first = prev.first;
        cur.zeros = newz;
        merged.pop_back();
      }
      merged.push_back(cur);
    }
    sns.swap(merged);
  }
  // width cap
  {
    std::vector<SN> capped;
    for (auto& s : sns) {
      int nc = s.last - s.first + 1;
      if (nc <= S->max_super_cols) { capped.push_back(s); continue; }
      int parts = (nc + S->max_super_cols - 1) / S->max_super_cols;
      int base = nc / parts, extra = nc % parts, f = s.first;
      for (int p = 0; p < parts; ++p) {
        int w = base + (p < extra ? 1 : 0);
        capped.push_back({f, f + w - 1, 0});
        f += w;
      }
    }
    sns.swap(capped);
  }
  int ns = (int)sns.size();
  S->nsuper = ns;
  S->sn_first.resize(ns + 1);
  S->col2sn.resize(n);
  for (int k = 0; k < ns; ++k) {
    S->sn_first[k] = sns[k].first;
    for (int c = sns[k].first; c <= sns[k].last; ++c) S->col2sn[c] = k;
  }
  S->sn_first[ns] = n;
  S->sn_parent.assign(ns, -1);
  for (int k = 0; k < ns; ++k) {
    int p = parent[sns[k].last];
    S->sn_parent[k] = (p < 0) ? -1 : S->col2sn[p];
    if (S->sn_parent[k] >= 0 && S->sn_parent[k] <= k) { eigd_set_error("symbolic: supernodal tree not ordered"); delete S; return 2; }
  }
  // children lists
  S->child_ptr.assign(ns + 1, 0);
  for (int k = 0; k < ns; ++k) if (S->sn_parent[k] >= 0) S->child_ptr[S->sn_parent[k] + 1]++;
  for (int k = 0; k < ns; ++k) S->child_ptr[k + 1] += S->child_ptr[k];
  S->child_idx.resize(S->child_ptr[ns]);
  {
    std::vector<int> pos(S->child_ptr.begin(), S->child_ptr.end() - 1);
    for (int k = 0; k < ns; ++k) if (S->sn_parent[k] >= 0) S->child_idx[pos[S->sn_parent[k]]++] = k;
  }
  // ---- row structures ----------------------------------------------------------------------
  S->sn_rowptr.assign(ns + 1, 0);
  S->sn_rows.clear();
  {
    std::vector<int> stamp(n, -1), rows;
    for (int k = 0; k < ns; ++k) {
      rows.clear();
      int last = sns[k].last;
      for (int c = sns[k].first; c <= last; ++c)
        for (int64_t p = L.ptr[c]; p < L.ptr[c + 1]; ++p) {
          int r = L.rows[p];
          if (r > last && stamp[r] != k) { stamp[r] = k; rows.push_back(r); }
        }
      for (int q = S->child_ptr[k]; q < S->child_ptr[k + 1]; ++q) {
        int c = S->child_idx[q];
        for (int64_t p = S->sn_rowptr[c]; p < S->sn_rowptr[c + 1]; ++p) {
          int r = S->sn_rows[p];
          if (r > last && stamp[r] != k) { stamp[r] = k; rows.push_back(r); }
        }
      }
      std::sort(rows.begin(), rows.end());
      S->sn_rows.insert(S->sn_rows.end(), rows.begin(), rows.end());
      S->sn_rowptr[k + 1] = (int64_t)S->sn_rows.size();
    }
  }
  // ---- relative indices, offsets, levels ---------------------------------------------------
  S->rel.assign(S->sn_rows.size(), -1);
  for (int k = 0; k < ns; ++k) {
    int p = S->sn_parent[k];
    if (p < 0) {
      if (S->sn_rowptr[k + 1] != S->sn_rowptr[k]) { eigd_set_error("symbolic: root front has below rows"); delete S; return 2; }
      continue;
    }
    int pf = S->sn_first[p], pl = S->sn_first[p + 1] - 1, pnc = pl - pf + 1;
    const int* prow = S->sn_rows.data() + S->sn_rowptr[p];
    int pn = (int)(S->sn_rowptr[p + 1] - S->sn_rowptr[p]);
    int cursor = 0;
    for (int64_t q = S->sn_rowptr[k]; q < S->sn_rowptr[k + 1]; ++q) {
      int r = S->sn_rows[q];
      if (r < pf) { eigd_set_error("symbolic: child row before parent front"); delete S; return 2; }
      if (r <= pl) { S->rel[q] = r - pf; continue; }
      while (cursor < pn && prow[cursor] < r) ++cursor;
      if (cursor >= pn || prow[cursor] != r) { eigd_set_error("symbolic: child row missing from parent front"); delete S; return 2; }
      S->rel[q] = pnc + cursor;
    }
  }
  S->front_off.assign(ns + 1, 0);
  S->w_off.assign(ns + 1, 0);
  S->nnzL = 0; S->flops = 0; S->maxfront = 0; S->maxcols = 0;
  for (int k = 0; k < ns; ++k) {
    int64_t nc = sn_ncols(S, k), nb = sn_nbelow(S, k), f = nc + nb;
    S->front_off[k + 1] = S->front_off[k] + f * f;
    S->w_off[k + 1] = S->w_off[k] + f;
    S->nnzL += nc * (nc - 1) / 2 + nc * nb;
    S->flops += nc * nb * nb + nc * nc * nb + nc * nc * nc / 3;
    S->maxfront = std::max<int>(S->maxfront, (int)f);
    S->maxcols = std::max<int>(S->maxcols, (int)nc);
  }
  S->sn_level.assign(ns, 0);
  int nl = 0;
  for (int k = 0; k < ns; ++k) {
    int p = S->sn_parent[k];
    if (p >= 0) S->sn_level[p] = std::max(S->sn_level[p], S->sn_level[k] + 1);
    nl = std::max(nl, S->sn_level[k] + 1);
  }
  S->nlevels = nl;
  S->level_ptr.assign(nl + 1, 0);
  for (int k = 0; k < ns; ++k) S->level_ptr[S->sn_level[k] + 1]++;
  for (int l = 0; l < nl; ++l) S->level_ptr[l + 1] += S->level_ptr[l];
  S->level_sn.resize(ns);
  {
    std::vector<int> pos(S->level_ptr.begin(), S->level_ptr.end() - 1);
    for (int k = 0; k < ns; ++k) S->level_sn[pos[S->sn_level[k]]++] = k;
  }
  pool_layout(S);
  *out = S;
  return 0;
}

extern "C" void eigd_symbolic_destroy(eigd_symbolic* s) {
  if (!s) return;
  if (s->dev && s->dev_free) s->dev_free(s->dev);
  delete s;
}

extern "C" int64_t eigd_symbolic_query(const eigd_symbolic* s, int what) {
  switch (what) {
    case 0: return s->n;
    case 1: return s->nsuper;
    case 2: return s->nlevels;
    case 3: return s->nnzL;
    case 4: return s->front_off[s->nsuper];
    case 5: return s->w_off[s->nsuper];
    case 6: return s->maxfront;
    case 7: return s->maxcols;
    case 8: return s->flops;
    case 9: return s->exact_nnzL;
    case 10: return s->pool_doubles;
    default: return -1;
  }
}

template <class T>
static int64_t copy_out(const std::vector<T>& v, int64_t* out, int64_t cap) {
  int64_t m = std::min<int64_t>((int64_t)v.size(), cap);
  if (out) for (int64_t i = 0; i < m; ++i) out[i] = (int64_t)v[i];
  return (int64_t)v.size();
}

extern "C" int64_t eigd_symbolic_get(const eigd_symbolic* s, int which, int64_t* out, int64_t cap) {
  switch (which) {
    case 0: return copy_out(s->perm, out, cap);
    case 1: return copy_out(s->parent, out, cap);
    case 2: return copy_out(s->sn_first, out, cap);
    case 3: return copy_out(s->sn_rowptr, out, cap);
    case 4: return copy_out(s->sn_rows, out, cap);
    case 5: return copy_out(s->sn_parent, out, cap);
    case 6: return copy_out(s->sn_level, out, cap);
    case 7: return copy_out(s->front_off, out, cap);
    case 8: return copy_out(s->rel, out, cap);
    case 9: return copy_out(s->colcount, out, cap);
    case 10: return copy_out(s->level_ptr, out, cap);
    case 11: return copy_out(s->level_sn, out, cap);
    case 12: return copy_out(s->pool_off, out, cap);
    default: return -1;
  }
}

extern "C" int eigd_symbolic_assembly_map_host(const eigd_symbolic* s, int n, const int* indptr,
                                               const int* indices, int64_t* out_map) {
  if (n != s->n) { eigd_set_error("assembly_map: n mismatch"); return 1; }
  for (int r = 0; r < n; ++r)
    for (int p = indptr[r]; p < indptr[r + 1]; ++p) {
      int pr = s->iperm[r], pc = s->iperm[indices[p]];
      if (pr < pc) { out_map[p] = -1; continue; }
      int k = s->col2sn[pc];
      int first = s->sn_first[k], nc = s->sn_first[k + 1] - first;
      int64_t f = nc + (s->sn_rowptr[k + 1] - s->sn_rowptr[k]);
      int64_t lr;
      if (pr < first + nc) lr = pr - first;
      else {
        const int* b = s->sn_rows.data() + s->sn_rowptr[k];
        const int* e = s->sn_rows.data() + s->sn_rowptr[k + 1];
        const int* it = std::lower_bound(b, e, pr);
        if (it == e || *it != pr) { eigd_set_error("assembly_map: entry (%d,%d) outside the symbolic pattern", r, indices[p]); return 2; }
        lr = nc + (it - b);
      }
      out_map[p] = s->front_off[k] + lr + (int64_t)(pc - first) * f;
    }
  return 0;
}
