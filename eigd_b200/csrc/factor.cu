// Supernodal multifrontal LDL^T of the shifted matrix and its multi-RHS triangular solves.
// Replaces scipy.sparse.linalg.splu (SuperLU gstrf) and SuperLU.solve behind SpLuOperator
// (reference eigd/eigenvector_derivatives.py:11-23): x <- (A - sigma B)^{-1} x, or
// (B + sigma A)^{-1} x in buckling mode (:786-790).
//
// Data layout in HBM
//   fronts : one dense column-major f x f block per supernode (lower triangle used);
//            columns [0, ncols) hold L (unit diagonal implied, D on the diagonal), the
//            trailing (f-ncols)^2 block is the contribution passed to the parent.  Resident (front_off, in the
//            factor's workspace for its life) or pooled (pool_off, in a pool the caller lends to one numeric call;
//            a front is live from its own level through its parent's, see pool_layout in symbolic.cpp).
//   linv   : explicit inverses of the 32x32 unit-lower diagonal blocks of every L11 (used by the
//            panel solves of the factorisation); with restricted Bunch-Kaufman pivoting the inverses of
//            the dense diagonal blocks M (diag_factor_bk_kernel).
//   xinv   : the full inverse X = L11^{-1} of every pivot block (recursive doubling from the
//            32x32 inverses: X21 = -B^{-1} C A^{-1}).
//   sfwd / sbwd : the solve panels S = [X ; -L21 X] (f x nc, column-major) and S^T (nc x f):
//            with them both triangular sweeps of a front are plain dense products with no
//            dependency inside the front (solve.cu), one grid barrier per tree level.
// Execution: supernodes are grouped by height in the assembly tree; every level is a handful
// of batched launches driven by host-built task lists (front, tile).
#include "factor_internal.cuh"
#include "../../include/eigd_b200.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

namespace {

template <class T>
int upload(SymDevHolder* h, const std::vector<T>& v, T** out) {
  void* p = nullptr;
  size_t bytes = std::max<size_t>(v.size(), 1) * sizeof(T);
  EIGD_CUDA(cudaMalloc(&p, bytes));
  h->allocs.push_back(p);
  if (!v.empty()) EIGD_CUDA(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  *out = (T*)p;
  return 0;
}

}  // namespace

static void free_symdev(void* p) {
  auto* h = (SymDevHolder*)p;
  free_solve_plan_dev(h);
  for (void* a : h->allocs) cudaFree(a);
  if (h->tasks) cudaFree(h->tasks);
  if (h->pool_tasks) cudaFree(h->pool_tasks);
  delete h;
}

inline int tri_tiles(int m, int tile) {
  int t = (m + tile - 1) / tile;
  return t * (t + 1) / 2;
}

static void push_launch(std::vector<int2>& tasks, std::vector<Launch>& plan, int kind, int kb, int64_t off) {
  int count = (int)((int64_t)tasks.size() - off);
  if (count > 0) plan.push_back({kind, kb, off, count});
}

// extend-add into the fronts of level l (one launch per sibling rank), then the pivot-block chain of its fronts
static void push_level_tasks(const eigd_symbolic* S, int l, std::vector<int2>& tasks, std::vector<Launch>& plan) {
  const int* sn = S->level_sn.data() + S->level_ptr[l];
  int cnt = S->level_ptr[l + 1] - S->level_ptr[l];
  // extend-add: one launch per sibling rank so that no two tasks touch the same parent
  int maxrank = 0;
  for (int i = 0; i < cnt; ++i) maxrank = std::max(maxrank, S->child_ptr[sn[i] + 1] - S->child_ptr[sn[i]]);
  for (int r = 0; r < maxrank; ++r) {
    int64_t off = (int64_t)tasks.size();
    for (int i = 0; i < cnt; ++i) {
      int p = sn[i];
      if (S->child_ptr[p] + r >= S->child_ptr[p + 1]) continue;
      int c = S->child_idx[S->child_ptr[p] + r];
      int nt = tri_tiles(sn_nbelow(S, c), EA_TILE);
      for (int t = 0; t < nt; ++t) tasks.push_back(make_int2(c, t));
    }
    push_launch(tasks, plan, 0, r, off);
  }
  int maxsteps = 0;
  for (int i = 0; i < cnt; ++i) maxsteps = std::max(maxsteps, (sn_ncols(S, sn[i]) + NB - 1) / NB);
  for (int kb = 0; kb < maxsteps; ++kb) {
    int64_t off = (int64_t)tasks.size();
    for (int i = 0; i < cnt; ++i)
      if (sn_ncols(S, sn[i]) > kb * NB) tasks.push_back(make_int2(sn[i], 0));
    push_launch(tasks, plan, 1, kb, off);
    off = (int64_t)tasks.size();
    for (int i = 0; i < cnt; ++i) {
      int k = sn[i], nc = sn_ncols(S, k), f = sn_fsize(S, k);
      if (nc <= kb * NB) continue;
      int r0 = std::min(nc, (kb + 1) * NB);
      int nt = (f - r0 + TRSM_ROWS - 1) / TRSM_ROWS;
      for (int t = 0; t < nt; ++t) tasks.push_back(make_int2(k, t));
    }
    push_launch(tasks, plan, 2, kb, off);
    off = (int64_t)tasks.size();
    for (int i = 0; i < cnt; ++i) {
      int k = sn[i], nc = sn_ncols(S, k), f = sn_fsize(S, k);
      if (nc <= kb * NB) continue;
      int r0 = std::min(nc, (kb + 1) * NB);
      int nt = tri_tiles(f - r0, UPD_TILE);
      for (int t = 0; t < nt; ++t) tasks.push_back(make_int2(k, t));
    }
    push_launch(tasks, plan, 3, kb, off);
  }
}

// full inverses of the pivot blocks (recursive doubling) and the solve panels of the fronts sn[0 .. cnt)
static void push_panel_tasks(const eigd_symbolic* S, const int* sn, int cnt, std::vector<int2>& tasks,
                             std::vector<Launch>& plan) {
  int64_t off = (int64_t)tasks.size();
  int maxcols = 0;
  for (int i = 0; i < cnt; ++i) {
    tasks.push_back(make_int2(sn[i], 0));
    maxcols = std::max(maxcols, sn_ncols(S, sn[i]));
  }
  push_launch(tasks, plan, 4, 0, off);
  for (int stage = 0, hb = NB; hb < maxcols; ++stage, hb *= 2) {
    off = (int64_t)tasks.size();
    for (int i = 0; i < cnt; ++i) {
      int k = sn[i], nc = sn_ncols(S, k);
      for (int q = 0; (2 * q + 1) * hb < nc; ++q) {
        int hh = std::min(hb, nc - (2 * q + 1) * hb);
        for (int ti = 0; ti * NB < hh; ++ti)
          for (int tj = 0; tj * NB < hb; ++tj) tasks.push_back(make_int2(k, q * 64 + ti * 8 + tj));
      }
    }
    int64_t end = (int64_t)tasks.size();
    push_launch(tasks, plan, 5, stage, off);       // T = C A^-1
    if (end > off) plan.push_back({6, stage, off, (int)(end - off)});   // X21 = -B^-1 T (same tasks)
  }
  off = (int64_t)tasks.size();
  for (int i = 0; i < cnt; ++i)
    for (int t = 0; t * NB < sn_fsize(S, sn[i]); ++t) tasks.push_back(make_int2(sn[i], t));
  push_launch(tasks, plan, 7, 0, off);
}

int build_symdev(eigd_symbolic* S) {
  if (S->dev) return 0;
  auto* h = new SymDevHolder();
  S->dev = h;
  S->dev_free = free_symdev;
  int ns = S->nsuper;
  h->d.n = S->n;
  h->d.nsuper = ns;
  std::vector<int64_t> linv_off(ns + 1, 0);
  for (int k = 0; k < ns; ++k) linv_off[k + 1] = linv_off[k] + (int64_t)((sn_ncols(S, k) + NB - 1) / NB) * NB * NB;
  h->linv_total = linv_off[ns];
  std::vector<int64_t> soff(ns + 1, 0), xoff(ns + 1, 0);
  for (int k = 0; k < ns; ++k) {
    soff[k + 1] = soff[k] + solve_panel_doubles(sn_fsize(S, k), sn_ncols(S, k));
    xoff[k + 1] = xoff[k] + (int64_t)sn_ncols(S, k) * sn_ncols(S, k);
  }
  h->panel_total = soff[ns];
  h->xinv_total = xoff[ns];
  if (S->maxcols > 512) { eigd_set_error("build_symdev: supernodes wider than 512 columns are not supported"); return 4; }
  int rc = 0;
  rc |= upload(h, S->perm, &h->d.perm);
  rc |= upload(h, S->iperm, &h->d.iperm);
  rc |= upload(h, S->col2sn, &h->d.col2sn);
  rc |= upload(h, S->sn_first, &h->d.sn_first);
  rc |= upload(h, S->sn_rowptr, &h->d.sn_rowptr);
  rc |= upload(h, S->sn_rows, &h->d.sn_rows);
  rc |= upload(h, S->rel, &h->d.rel);
  rc |= upload(h, S->front_off, &h->d.front_off);
  rc |= upload(h, S->w_off, &h->d.w_off);
  rc |= upload(h, linv_off, &h->d.linv_off);
  rc |= upload(h, soff, &h->d.soff);
  rc |= upload(h, xoff, &h->d.xoff);
  rc |= upload(h, S->sn_parent, &h->d.sn_parent);
  rc |= upload(h, S->child_ptr, &h->d.child_ptr);
  rc |= upload(h, S->child_idx, &h->d.child_idx);
  if (rc) return rc;

  // ---- task lists ---------------------------------------------------------------------
  std::vector<int2> tasks;
  std::vector<int> all(ns);
  for (int k = 0; k < ns; ++k) all[k] = k;
  for (int l = 0; l < S->nlevels; ++l) push_level_tasks(S, l, tasks, h->factor_plan);
  // after the last level: full inverses of the pivot blocks and the solve panels (all fronts at once)
  push_panel_tasks(S, all.data(), ns, tasks, h->factor_plan);
  EIGD_CUDA(cudaMalloc((void**)&h->tasks, std::max<size_t>(tasks.size(), 1) * sizeof(int2)));
  EIGD_CUDA(cudaMemcpy(h->tasks, tasks.data(), tasks.size() * sizeof(int2), cudaMemcpyHostToDevice));
  return build_solve_plan_dev(S, h);
}

// The plan of the pooled front mode, built on first use: per level, the fronts of the level are zeroed in the pool and
// receive their matrix entries (kind 8), take their children's contributions, are factorised, and leave their pivot-
// block inverses and solve panels before any front of a later level can reuse their memory.  Same kernels and the
// same per-front arithmetic as factor_plan; the fronts are addressed through pool_off instead of front_off.
int build_pool_plan(eigd_symbolic* S) {
  int rc = build_symdev(S);
  if (rc) return rc;
  auto* h = (SymDevHolder*)S->dev;
  if (h->pool_tasks) return 0;
  if (S->maxfront > 46340) { eigd_set_error("pooled fronts: a front of %d rows is wider than the 32-bit slot index allows", S->maxfront); return 4; }
  rc = upload(h, S->pool_off, &h->pool_off);
  if (rc) return rc;
  std::vector<int2> tasks;
  for (int l = 0; l < S->nlevels; ++l) {
    const int* sn = S->level_sn.data() + S->level_ptr[l];
    int cnt = S->level_ptr[l + 1] - S->level_ptr[l];
    int64_t off = (int64_t)tasks.size();
    for (int i = 0; i < cnt; ++i) {
      int64_t f = sn_fsize(S, sn[i]);
      for (int64_t t = 0; t * POOL_CHUNK < f * f; ++t) tasks.push_back(make_int2(sn[i], (int)t));
    }
    push_launch(tasks, h->pool_plan, 8, 0, off);
    push_level_tasks(S, l, tasks, h->pool_plan);
    push_panel_tasks(S, sn, cnt, tasks, h->pool_plan);
  }
  EIGD_CUDA(cudaMalloc((void**)&h->pool_tasks, std::max<size_t>(tasks.size(), 1) * sizeof(int2)));
  EIGD_CUDA(cudaMemcpy(h->pool_tasks, tasks.data(), tasks.size() * sizeof(int2), cudaMemcpyHostToDevice));
  return 0;
}

namespace {

// ---------------------------------------------------------------------------------------
// integer kernel: CSR non-zero -> slot in front storage (bit-exact twin of the host routine)
// ---------------------------------------------------------------------------------------
__global__ void assembly_map_kernel(SymDev d, const int* __restrict__ indptr, const int* __restrict__ indices,
                                    int64_t* __restrict__ map, int* __restrict__ err) {
  int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= d.n) return;
  int pr = d.iperm[r];
  for (int p = indptr[r]; p < indptr[r + 1]; ++p) {
    int pc = d.iperm[indices[p]];
    if (pr < pc) { map[p] = -1; continue; }
    int k = d.col2sn[pc];
    int first = d.sn_first[k], nc = d.sn_first[k + 1] - first;
    int64_t rb = d.sn_rowptr[k], re = d.sn_rowptr[k + 1];
    int64_t f = nc + (re - rb);
    int64_t lr;
    if (pr < first + nc) lr = pr - first;
    else {
      int64_t lo = rb, hi = re;
      while (lo < hi) {
        int64_t mid = (lo + hi) >> 1;
        if (d.sn_rows[mid] < pr) lo = mid + 1; else hi = mid;
      }
      if (lo >= re || d.sn_rows[lo] != pr) { atomicExch(err, 1); map[p] = -1; continue; }
      lr = nc + (lo - rb);
    }
    map[p] = d.front_off[k] + lr + (int64_t)(pc - first) * f;
  }
}

// ---------------------------------------------------------------------------------------
// numeric factorisation kernels
// ---------------------------------------------------------------------------------------
__global__ void absmax_kernel(int64_t nnz, const double* __restrict__ v, unsigned long long* __restrict__ out) {
  double m = 0.0;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (int64_t)gridDim.x * blockDim.x) {
    double a = fabs(v[e]);
    if (a == a) m = fmax(m, a);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, (unsigned long long)__double_as_longlong(m));
}

__global__ void scatter_values_kernel(int64_t nnz, const double* __restrict__ vals, const int64_t* __restrict__ map,
                                      double* __restrict__ fronts) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t m = map[e];
    if (m >= 0) fronts[m] = vals[e];
  }
}

// Pooled fronts: chunk tk.y (POOL_CHUNK doubles) of front tk.x is zeroed, then receives the matrix entries whose slots
// fall in it: ent[seg[s] .. seg[s + 1]) are (CSR index, slot in the front) pairs sorted by slot.  One CTA owns the
// chunk, so the zero stores and the entry stores need no atomics, only one block barrier between them.  Front offsets
// are multiples of 32 doubles and chunks start at multiples of POOL_CHUNK: the 16-byte zero stores are aligned.
__global__ void __launch_bounds__(256)
front_assemble_kernel(SymDev d, const int2* __restrict__ tasks, const double* __restrict__ vals,
                      const int64_t* __restrict__ seg, const int2* __restrict__ ent, double* __restrict__ pool) {
  __shared__ int64_t range[2];
  const int2 tk = tasks[blockIdx.x];
  const int s = tk.x;
  const int64_t f = (d.sn_first[s + 1] - d.sn_first[s]) + (d.sn_rowptr[s + 1] - d.sn_rowptr[s]);
  const int64_t lo = (int64_t)tk.y * POOL_CHUNK, hi = min(f * f, lo + POOL_CHUNK);
  double* F = pool + d.front_off[s];
  double2* Z = reinterpret_cast<double2*>(F + lo);
  const int nz2 = (int)((hi - lo) >> 1);
  for (int i = threadIdx.x; i < nz2; i += blockDim.x) Z[i] = make_double2(0.0, 0.0);
  if (((hi - lo) & 1) && threadIdx.x == 0) F[hi - 1] = 0.0;
  if (threadIdx.x < 2) {                    // first entry with slot >= lo (thread 0) / >= hi (thread 1)
    const int64_t key = threadIdx.x ? hi : lo;
    int64_t a = seg[s], b = seg[s + 1];
    while (a < b) {
      const int64_t m = (a + b) >> 1;
      if (ent[m].y < key) a = m + 1; else b = m;
    }
    range[threadIdx.x] = a;
  }
  __syncthreads();
  for (int64_t e = range[0] + threadIdx.x; e < range[1]; e += blockDim.x) {
    const int2 v = ent[e];
    F[v.y] = vals[v.x];
  }
}

__device__ __forceinline__ void tri_decode(int t, int& ti, int& tj) {
  int i = (int)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
  while ((i + 1) * (i + 2) / 2 <= t) ++i;
  while (i * (i + 1) / 2 > t) --i;
  ti = i;
  tj = t - i * (i + 1) / 2;
}

// parent(rel[i], rel[j]) += child contribution (i, j), lower triangle, 32x32 tiles
__global__ void __launch_bounds__(256)
extend_add_kernel(SymDev d, const int2* __restrict__ tasks, double* __restrict__ fronts) {
  int2 tk = tasks[blockIdx.x];
  int c = tk.x;
  int ti, tj;
  tri_decode(tk.y, ti, tj);
  int p = d.sn_parent[c];
  int ncc = d.sn_first[c + 1] - d.sn_first[c];
  int nb = (int)(d.sn_rowptr[c + 1] - d.sn_rowptr[c]);
  int64_t fc = ncc + nb;
  int64_t fp = (d.sn_first[p + 1] - d.sn_first[p]) + (d.sn_rowptr[p + 1] - d.sn_rowptr[p]);
  const double* C = fronts + d.front_off[c] + ncc + (int64_t)ncc * fc;
  double* P = fronts + d.front_off[p];
  const int* rel = d.rel + d.sn_rowptr[c];
  int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  int i = ti * EA_TILE + tx;
  if (i >= nb) return;
  int ri = rel[i];
  // loads first, stores afterwards (parent and child live in the same array: see trailing_update_kernel)
  double pv[EA_TILE / 8], cv[EA_TILE / 8];
  int64_t pa[EA_TILE / 8];
#pragma unroll
  for (int q = 0; q < EA_TILE / 8; ++q) {
    int j = tj * EA_TILE + ty + 8 * q;
    bool ok = j < nb && j <= i;
    pa[q] = ok ? ri + (int64_t)rel[j] * fp : -1;
    cv[q] = ok ? C[i + (int64_t)j * fc] : 0.0;
    pv[q] = ok ? P[pa[q]] : 0.0;
  }
#pragma unroll
  for (int q = 0; q < EA_TILE / 8; ++q)
    if (pa[q] >= 0) P[pa[q]] = pv[q] + cv[q];
}

// LDL^T of one 32-wide pivot block + inverse of its unit-lower factor; one CTA per front.
// Threads are (tx = row, ty = column class mod 8).  Right-looking elimination with ONE barrier per
// column: every thread derives the (possibly perturbed) pivot from the same shared entry, the column is
// kept unscaled during the elimination and divided by its pivot afterwards.  The inverse of the unit
// lower triangle is computed column by column by groups of 8 consecutive lanes (shuffle reductions,
// no block barrier).
__global__ void __launch_bounds__(256)
diag_factor_kernel(SymDev d, const int2* __restrict__ tasks, int kb, double* __restrict__ fronts,
                   double* __restrict__ linv, double* __restrict__ dval, double* __restrict__ dinv,
                   const unsigned long long* __restrict__ amax_bits, double piv_tol,
                   unsigned long long* __restrict__ info) {
  __shared__ double T[NB][NB + 1];
  __shared__ double Li[NB][NB + 1];
  __shared__ double ds[NB];
  int s = tasks[blockIdx.x].x;
  int first = d.sn_first[s];
  int nc = d.sn_first[s + 1] - first;
  int64_t f = nc + (d.sn_rowptr[s + 1] - d.sn_rowptr[s]);
  int j0 = kb * NB;
  int bs = min(NB, nc - j0);
  double* F = fronts + d.front_off[s];
  const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
  for (int c = ty; c < NB; c += 8) {
    T[tx][c] = (tx < bs && c < bs && tx >= c) ? F[(j0 + tx) + (int64_t)(j0 + c) * f] : 0.0;
    Li[tx][c] = (tx == c) ? 1.0 : 0.0;
  }
  const double thr = piv_tol * __longlong_as_double((long long)(*amax_bits));
  int nneg = 0, npert = 0, nbad = 0;
  __syncthreads();
  for (int j = 0; j < bs; ++j) {
    double dj = T[j][j];
    if (!(dj == dj) || fabs(dj) > 1e300) { nbad++; dj = thr > 0.0 ? thr : 1.0; }
    if (fabs(dj) < thr) { dj = (dj >= 0.0) ? thr : -thr; npert++; }
    if (dj < 0.0) nneg++;
    if (tid == 0) ds[j] = dj;
    const double rd = 1.0 / dj;
    if (tx > j) {
      const double lij = T[tx][j] * rd;
      for (int c = j + 1 + ((ty - (j + 1)) & 7); c <= tx; c += 8) T[tx][c] = fma(-lij, T[c][j], T[tx][c]);
    }
    __syncthreads();
  }
  // scale the columns: L(i, j) = T(i, j) / d_j
  for (int c = ty; c < bs; c += 8)
    if (tx > c && tx < bs) T[tx][c] *= 1.0 / ds[c];
  __syncthreads();
  // inverse of the unit lower triangle: column c by lanes 8c .. 8c+7 of the block (32 columns x 8 lanes)
  {
    const int c = tid >> 3, q = tid & 7;
    const unsigned gmask = 0xffu << (8 * (c & 3));        // the four column groups of a warp run different trip counts
    for (int i = c + 1; i < bs; ++i) {
      double sum = 0.0;
      for (int k = c + q; k < i; k += 8) sum = fma(T[i][k], Li[k][c], sum);
      sum += __shfl_xor_sync(gmask, sum, 1);
      sum += __shfl_xor_sync(gmask, sum, 2);
      sum += __shfl_xor_sync(gmask, sum, 4);
      if (q == 0) Li[i][c] = -sum;
      __syncwarp(gmask);
    }
  }
  __syncthreads();
  for (int c = ty; c < bs; c += 8)
    if (tx < bs && tx > c) F[(j0 + tx) + (int64_t)(j0 + c) * f] = T[tx][c];
  if (tid < bs) F[(j0 + tid) + (int64_t)(j0 + tid) * f] = ds[tid];
  double* Lo = linv + d.linv_off[s] + (int64_t)kb * NB * NB;
  for (int c = ty; c < NB; c += 8) Lo[tx + c * NB] = Li[tx][c];   // column-major: Lo[i + j*NB]
  if (tid < bs) {
    dval[first + j0 + tid] = ds[tid];
    dinv[first + j0 + tid] = 1.0 / ds[tid];
  }
  if (tid == 0) {
    if (nneg) atomicAdd(&info[0], (unsigned long long)nneg);
    if (npert) atomicAdd(&info[1], (unsigned long long)npert);
    if (nbad) atomicAdd(&info[2], (unsigned long long)nbad);
  }
}

// Restricted Bunch-Kaufman variant of diag_factor_kernel (pivoting mode 1).  Bunch-Kaufman with alpha = (1 + sqrt 17) / 8,
// the pivot search restricted to the rows and columns of this 32-column block, ties to the lowest index: 1x1 pivots,
// 1x1 pivots with an interchange, or 2x2 pivots, which are rotated to diagonal form (Jacobi rotation) and eliminated
// as two 1x1 pivots.  With R the product of the interchanges and rotations (orthogonal) and L unit lower,
// R T R^T = L Lam L^T, i.e. T = M Lam M^T with M = R^T L, Lam diagonal.  Outputs as diag_factor_kernel: Li = M^-1 =
// L^-1 R (dense), Lam in dval / dinv; the kernels after this one only use Li and Lam (see trsm_kernel,
// inverse_init_kernel and the solve's tile bounds).  info[3] += 2x2 pivots, info[4] += interchanges.
// Every warp takes the pivot decision redundantly from shared memory (warp reductions over the column / row,
// lane 0's result broadcast: the decision is uniform), so a step costs a block barrier only where it writes.
constexpr double BK_ALPHA = 0.6403882032022076;        // (1 + sqrt(17)) / 8

__device__ __forceinline__ void warp_absmax(double& v, int& i) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double v2 = __shfl_xor_sync(0xffffffffu, v, o);
    const int i2 = __shfl_xor_sync(0xffffffffu, i, o);
    if (v2 > v || (v2 == v && i2 < i)) { v = v2; i = i2; }
  }
  v = __shfl_sync(0xffffffffu, v, 0);
  i = __shfl_sync(0xffffffffu, i, 0);
}

__global__ void __launch_bounds__(256)
diag_factor_bk_kernel(SymDev d, const int2* __restrict__ tasks, int kb, double* __restrict__ fronts,
                      double* __restrict__ linv, double* __restrict__ dval, double* __restrict__ dinv,
                      const unsigned long long* __restrict__ amax_bits, double piv_tol,
                      unsigned long long* __restrict__ info) {
  __shared__ double T[NB][NB + 1];        // lower triangle; column j < current step holds d_j * L(:, j)
  __shared__ double Li[NB][NB + 1];       // R during the elimination, L^-1 R afterwards
  __shared__ double ds[NB];
  int s = tasks[blockIdx.x].x;
  int first = d.sn_first[s];
  int nc = d.sn_first[s + 1] - first;
  int64_t f = nc + (d.sn_rowptr[s + 1] - d.sn_rowptr[s]);
  int j0 = kb * NB;
  int bs = min(NB, nc - j0);
  double* F = fronts + d.front_off[s];
  const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
  for (int c = ty; c < NB; c += 8) {
    T[tx][c] = (tx < bs && c < bs && tx >= c) ? F[(j0 + tx) + (int64_t)(j0 + c) * f] : 0.0;
    Li[tx][c] = (tx == c) ? 1.0 : 0.0;
  }
  const double thr = piv_tol * __longlong_as_double((long long)(*amax_bits));
  int nneg = 0, npert = 0, nbad = 0, n2 = 0, nswap = 0;
  auto at = [&](int i, int j) { return i >= j ? T[i][j] : T[j][i]; };
  // symmetric interchange of positions p < q (both >= the current step): thread m < 32 swaps the pair of lower-triangle
  // entries of index m, threads 32 .. 63 swap rows p, q of R
  auto swap = [&](int p, int q) {
    if (tid < 32) {
      const int m = tid;
      double *x = nullptr, *y = nullptr;
      if (m < p) { x = &T[p][m]; y = &T[q][m]; }
      else if (m == p) { x = &T[p][p]; y = &T[q][q]; }
      else if (m < q) { x = &T[m][p]; y = &T[q][m]; }
      else if (m > q) { x = &T[m][p]; y = &T[m][q]; }
      if (x) { const double t = *x; *x = *y; *y = t; }
    } else if (tid < 64) {
      const int m = tid - 32;
      const double t = Li[p][m]; Li[p][m] = Li[q][m]; Li[q][m] = t;
    }
  };
  __syncthreads();
  bool second = false;                    // step j is the second column of a rotated 2x2 pivot
  for (int j = 0; j < bs; ++j) {
    if (!second) {
      const double akk = fabs(T[j][j]);
      double cmax = (tx > j && tx < bs) ? fabs(T[tx][j]) : 0.0;
      int imax = (tx > j && tx < bs) ? tx : NB;
      warp_absmax(cmax, imax);
      int piv = j;
      if (imax < bs && !(akk >= BK_ALPHA * cmax)) {
        double rmax = (tx >= j && tx < bs && tx != imax) ? fabs(at(imax, tx)) : 0.0;
        int dummy = 0;
        warp_absmax(rmax, dummy);
        const double a = T[j][j], b = T[imax][j], c = T[imax][imax];
        __syncthreads();                  // every warp has read the row of imax: the step may now write
        if (akk >= BK_ALPHA * cmax * (cmax / rmax)) {
        } else if (fabs(c) >= BK_ALPHA * rmax) {
          piv = imax;
        } else {
          n2++;
          if (imax != j + 1) { swap(j + 1, imax); nswap++; __syncthreads(); }
          // Jacobi rotation J = [cs sn; -sn cs] with J^T [a b; b c] J = diag(a - t b, c + t b); rows / columns j, j + 1
          // of the block and rows j, j + 1 of R and of L(:, < j) become J^T (x_j, x_j+1)
          const double tau = (c - a) / (2.0 * b);
          const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
          const double cs = 1.0 / sqrt(1.0 + t * t), sn = t * cs;
          if (tid < 32) {
            const int m = tid;
            if (m < j) {
              const double x = T[j][m], y = T[j + 1][m];
              T[j][m] = cs * x - sn * y;
              T[j + 1][m] = sn * x + cs * y;
            } else if (m == j) {
              T[j][j] = a - t * b;
              T[j + 1][j + 1] = c + t * b;
              T[j + 1][j] = 0.0;
            } else if (m > j + 1) {
              const double x = T[m][j], y = T[m][j + 1];
              T[m][j] = cs * x - sn * y;
              T[m][j + 1] = sn * x + cs * y;
            }
          } else if (tid < 64) {
            const int m = tid - 32;
            const double x = Li[j][m], y = Li[j + 1][m];
            Li[j][m] = cs * x - sn * y;
            Li[j + 1][m] = sn * x + cs * y;
          }
          __syncthreads();
          second = true;
        }
      }
      if (piv != j) { swap(j, piv); nswap++; __syncthreads(); }
    } else {
      second = false;
    }
    double dj = T[j][j];
    if (!(dj == dj) || fabs(dj) > 1e300) { nbad++; dj = thr > 0.0 ? thr : 1.0; }
    if (fabs(dj) < thr) { dj = (dj >= 0.0) ? thr : -thr; npert++; }
    if (dj < 0.0) nneg++;
    if (tid == 0) ds[j] = dj;
    const double rd = 1.0 / dj;
    if (tx > j) {
      const double lij = T[tx][j] * rd;
      for (int c = j + 1 + ((ty - (j + 1)) & 7); c <= tx; c += 8) T[tx][c] = fma(-lij, T[c][j], T[tx][c]);
    }
    __syncthreads();
  }
  for (int c = ty; c < bs; c += 8)
    if (tx > c && tx < bs) T[tx][c] *= 1.0 / ds[c];
  __syncthreads();
  // Li <- L^-1 R: forward substitution on every column of R, column c by lanes 8c .. 8c+7 (as diag_factor_kernel)
  {
    const int c = tid >> 3, q = tid & 7;
    const unsigned gmask = 0xffu << (8 * (c & 3));
    for (int i = 1; i < bs; ++i) {
      double sum = 0.0;
      for (int k = q; k < i; k += 8) sum = fma(T[i][k], Li[k][c], sum);
      sum += __shfl_xor_sync(gmask, sum, 1);
      sum += __shfl_xor_sync(gmask, sum, 2);
      sum += __shfl_xor_sync(gmask, sum, 4);
      if (q == 0) Li[i][c] -= sum;
      __syncwarp(gmask);
    }
  }
  __syncthreads();
  for (int c = ty; c < bs; c += 8)
    if (tx < bs && tx > c) F[(j0 + tx) + (int64_t)(j0 + c) * f] = T[tx][c];
  if (tid < bs) F[(j0 + tid) + (int64_t)(j0 + tid) * f] = ds[tid];
  double* Lo = linv + d.linv_off[s] + (int64_t)kb * NB * NB;
  for (int c = ty; c < NB; c += 8) Lo[tx + c * NB] = Li[tx][c];
  if (tid < bs) {
    dval[first + j0 + tid] = ds[tid];
    dinv[first + j0 + tid] = 1.0 / ds[tid];
  }
  if (tid == 0) {
    if (nneg) atomicAdd(&info[0], (unsigned long long)nneg);
    if (npert) atomicAdd(&info[1], (unsigned long long)npert);
    if (nbad) atomicAdd(&info[2], (unsigned long long)nbad);
    if (n2) atomicAdd(&info[3], (unsigned long long)n2);
    if (nswap) atomicAdd(&info[4], (unsigned long long)nswap);
  }
}

// rows below the pivot block: L_row = (F_row * Linv^T) * D^-1 ; one thread per row.  DENSE (pivoted factor): Li is a
// dense 32x32 block, otherwise unit lower triangular
template <bool DENSE>
__global__ void __launch_bounds__(TRSM_ROWS)
trsm_kernel(SymDev d, const int2* __restrict__ tasks, int kb, double* __restrict__ fronts,
            const double* __restrict__ linv, const double* __restrict__ dinv) {
  __shared__ double Li[NB][NB + 1];
  __shared__ double di[NB];
  int2 tk = tasks[blockIdx.x];
  int s = tk.x;
  int first = d.sn_first[s];
  int nc = d.sn_first[s + 1] - first;
  int64_t f = nc + (d.sn_rowptr[s + 1] - d.sn_rowptr[s]);
  int j0 = kb * NB;
  int bs = min(NB, nc - j0);
  const double* Lg = linv + d.linv_off[s] + (int64_t)kb * NB * NB;
  for (int e = threadIdx.x; e < NB * NB; e += blockDim.x) Li[e % NB][e / NB] = Lg[e];
  if (threadIdx.x < NB) di[threadIdx.x] = (threadIdx.x < bs) ? dinv[first + j0 + threadIdx.x] : 0.0;
  __syncthreads();
  int64_t i = (int64_t)j0 + bs + (int64_t)tk.y * TRSM_ROWS + threadIdx.x;
  if (i >= f) return;
  double* F = fronts + d.front_off[s] + i + (int64_t)j0 * f;
  double x[NB];
#pragma unroll
  for (int k = 0; k < NB; ++k) x[k] = (k < bs) ? F[(int64_t)k * f] : 0.0;
#pragma unroll
  for (int c = 0; c < NB; ++c) {
    double sum = 0.0;
#pragma unroll
    for (int k = 0; k < (DENSE ? NB : c + 1); ++k) sum = fma(x[k], Li[c][k], sum);
    if (c < bs) F[(int64_t)c * f] = sum * di[c];
  }
}

// trailing update C(i,c) -= sum_k L(i,k) d_k L(c,k) over one pivot block; 64x64 lower tiles on the FP64
// tensor pipe (mma.sync.m8n8k4.f64 -> DMMA): 8 warps as 4 row groups x 2 column groups, each warp owns a
// 16 x 32 block = 2 x 4 MMA tiles, K = 32 in eight k-steps.  Operands are staged in shared memory with a
// row stride of NB + 4 doubles: the fragment loads (row = lane / 4, k = lane % 4) are then conflict-free.
constexpr int UPD_LD = NB + 4;

__device__ __forceinline__ void dmma_m8n8k4(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(256)
trailing_update_kernel(SymDev d, const int2* __restrict__ tasks, int kb, double* __restrict__ fronts,
                       const double* __restrict__ dval) {
  __shared__ double As[UPD_TILE][UPD_LD];
  __shared__ double Bs[UPD_TILE][UPD_LD];
  int2 tk = tasks[blockIdx.x];
  int s = tk.x;
  int ti, tj;
  tri_decode(tk.y, ti, tj);
  int first = d.sn_first[s];
  int nc = d.sn_first[s + 1] - first;
  int64_t f = nc + (d.sn_rowptr[s + 1] - d.sn_rowptr[s]);
  int j0 = kb * NB;
  int bs = min(NB, nc - j0);
  int64_t r0 = j0 + bs;
  double* F = fronts + d.front_off[s];
  int64_t ib = r0 + (int64_t)ti * UPD_TILE, cb = r0 + (int64_t)tj * UPD_TILE;
  for (int e = threadIdx.x; e < UPD_TILE * NB; e += blockDim.x) {
    int r = e % UPD_TILE, k = e / UPD_TILE;
    double a = 0.0, b = 0.0;
    if (k < bs) {
      if (ib + r < f) a = F[(ib + r) + (int64_t)(j0 + k) * f];
      if (cb + r < f) b = F[(cb + r) + (int64_t)(j0 + k) * f] * dval[first + j0 + k];
    }
    As[r][k] = a;
    Bs[r][k] = b;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int wr = (warp & 3) * 16, wc = (warp >> 2) * 32;
  const int fr = lane >> 2, fk = lane & 3;
  double acc[2][4][2];
#pragma unroll
  for (int mi = 0; mi < 2; ++mi)
#pragma unroll
    for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
#pragma unroll
  for (int k0 = 0; k0 < NB; k0 += 4) {
    double a[2], b[4];
#pragma unroll
    for (int mi = 0; mi < 2; ++mi) a[mi] = As[wr + mi * 8 + fr][k0 + fk];
#pragma unroll
    for (int ni = 0; ni < 4; ++ni) b[ni] = Bs[wc + ni * 8 + fr][k0 + fk];
#pragma unroll
    for (int mi = 0; mi < 2; ++mi)
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) dmma_m8n8k4(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
  }
  // accumulator layout: row = lane / 4, columns 2 * (lane % 4) + {0, 1}.  All old values are loaded before
  // the first store: loads and stores go through the same pointer, so a load placed after a store would
  // have to wait for it (16 serialised DRAM round trips instead of one).
  double old[2][4][2];
#pragma unroll
  for (int ni = 0; ni < 4; ++ni)
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int64_t c = cb + wc + ni * 8 + 2 * fk + q;
#pragma unroll
      for (int mi = 0; mi < 2; ++mi) {
        const int64_t i = ib + wr + mi * 8 + fr;
        old[mi][ni][q] = (c < f && i < f && i >= c) ? F[i + c * f] : 0.0;
      }
    }
#pragma unroll
  for (int ni = 0; ni < 4; ++ni)
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int64_t c = cb + wc + ni * 8 + 2 * fk + q;
#pragma unroll
      for (int mi = 0; mi < 2; ++mi) {
        const int64_t i = ib + wr + mi * 8 + fr;
        if (c < f && i < f && i >= c) F[i + c * f] = old[mi][ni][q] - acc[mi][ni][q];
      }
    }
}

// ---------------------------------------------------------------------------------------
// solve panels: X = L11^{-1} by recursive doubling, S = [X ; -L21 X] and S^T
// ---------------------------------------------------------------------------------------
// 32 x 32 output tile of a product with 256 threads: thread (tx, ty) accumulates the four outputs
// (tx, ty + 8q).  fa(i, kk) / fb(kk, j) return the operand entries (0 outside their valid range).
template <class FA, class FB>
__device__ __forceinline__ void tile_gemm32(int K, FA fa, FB fb, double acc[4], double (*As)[NB + 1], double (*Bs)[NB + 1]) {
  const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
#pragma unroll
  for (int q = 0; q < 4; ++q) acc[q] = 0.0;
  for (int k0 = 0; k0 < K; k0 += NB) {
    for (int e = tid; e < NB * NB; e += 256) {
      int i = e & 31, kk = e >> 5;
      As[i][kk] = (k0 + kk < K) ? fa(i, k0 + kk) : 0.0;
      Bs[i][kk] = (k0 + i < K) ? fb(k0 + i, kk) : 0.0;      // Bs[kk][j] with (kk, j) = (i, kk) of this loop
    }
    __syncthreads();
#pragma unroll 8
    for (int kk = 0; kk < NB; ++kk) {
      double a = As[tx][kk];
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[q] = fma(a, Bs[kk][ty + 8 * q], acc[q]);
    }
    __syncthreads();
  }
}

// X <- diag(linv blocks) (X was zeroed by a memset); one CTA per front.  DENSE (pivoted factor): the whole 32x32 block
// M^-1 of every pivot block, otherwise its lower triangle.  X = M11^-1 is then block lower triangular at 32-column
// granularity; the doubling stages below (inverse_ca_kernel, inverse_bt_kernel) assume triangularity only at that
// granularity -- their reduction bounds start / end at 32-column tile edges -- and so compute M11^-1 as written.
template <bool DENSE>
__global__ void __launch_bounds__(256)
inverse_init_kernel(SymDev d, const int2* __restrict__ tasks, const double* __restrict__ linv, double* __restrict__ xinv) {
  int s = tasks[blockIdx.x].x;
  int nc = d.sn_first[s + 1] - d.sn_first[s];
  double* X = xinv + d.xoff[s];
  const double* Lo = linv + d.linv_off[s];
  int nblk = (nc + NB - 1) / NB;
  for (int e = threadIdx.x; e < nblk * NB * NB; e += blockDim.x) {
    int kb = e / (NB * NB), r = e - kb * NB * NB;
    int i = r & 31, j = r >> 5;
    int gi = kb * NB + i, gj = kb * NB + j;
    if (gi < nc && gj < nc && (DENSE || i >= j)) X[gi + (int64_t)gj * nc] = Lo[e];
  }
}

// doubling stage, first product: T = C A^{-1} for the pair (lo block, hi block) of width hb
__global__ void __launch_bounds__(256)
inverse_ca_kernel(SymDev d, const int2* __restrict__ tasks, int hb, const double* __restrict__ fronts,
                  const double* __restrict__ xinv, double* __restrict__ xtmp) {
  __shared__ double As[NB][NB + 1];
  __shared__ double Bs[NB][NB + 1];
  int2 tk = tasks[blockIdx.x];
  int s = tk.x, q = tk.y >> 6, ti = (tk.y >> 3) & 7, tj = tk.y & 7;
  int nc = d.sn_first[s + 1] - d.sn_first[s];
  int64_t f = nc + (d.sn_rowptr[s + 1] - d.sn_rowptr[s]);
  int lo0 = 2 * q * hb, hi0 = lo0 + hb, hh = min(hb, nc - hi0);
  const double* F = fronts + d.front_off[s];
  const double* X = xinv + d.xoff[s];
  double* T = xtmp + d.xoff[s];
  int c0 = lo0 + tj * NB;                 // A^{-1} is lower triangular: terms c >= first column of the tile
  int K = hb - tj * NB;
  double acc[4];
  tile_gemm32(K,
              [&](int i, int kk) { return (ti * NB + i < hh) ? F[(hi0 + ti * NB + i) + (int64_t)(c0 + kk) * f] : 0.0; },
              [&](int kk, int j) { return X[(c0 + kk) + (int64_t)(c0 + j) * nc]; }, acc, As, Bs);
  int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  if (ti * NB + tx < hh)
#pragma unroll
    for (int qq = 0; qq < 4; ++qq) T[(hi0 + ti * NB + tx) + (int64_t)(c0 + ty + 8 * qq) * nc] = acc[qq];
}

// doubling stage, second product: X21 = -B^{-1} T
__global__ void __launch_bounds__(256)
inverse_bt_kernel(SymDev d, const int2* __restrict__ tasks, int hb, double* __restrict__ xinv,
                  const double* __restrict__ xtmp) {
  __shared__ double As[NB][NB + 1];
  __shared__ double Bs[NB][NB + 1];
  int2 tk = tasks[blockIdx.x];
  int s = tk.x, q = tk.y >> 6, ti = (tk.y >> 3) & 7, tj = tk.y & 7;
  int nc = d.sn_first[s + 1] - d.sn_first[s];
  int lo0 = 2 * q * hb, hi0 = lo0 + hb, hh = min(hb, nc - hi0);
  double* X = xinv + d.xoff[s];
  const double* T = xtmp + d.xoff[s];
  int c0 = lo0 + tj * NB;
  int K = min(hh, (ti + 1) * NB);         // B^{-1} is lower triangular: terms c <= last row of the tile
  double acc[4];
  tile_gemm32(K,
              [&](int i, int kk) { return (ti * NB + i < hh) ? X[(hi0 + ti * NB + i) + (int64_t)(hi0 + kk) * nc] : 0.0; },
              [&](int kk, int j) { return T[(hi0 + kk) + (int64_t)(c0 + j) * nc]; }, acc, As, Bs);
  int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  if (ti * NB + tx < hh)
#pragma unroll
    for (int qq = 0; qq < 4; ++qq) X[(hi0 + ti * NB + tx) + (int64_t)(c0 + ty + 8 * qq) * nc] = -acc[qq];
}

// one 32-row tile of the solve panel: S rows < nc are X, rows >= nc are -L21 X; also written transposed
__global__ void __launch_bounds__(256)
panel_build_kernel(SymDev d, const int2* __restrict__ tasks, const double* __restrict__ fronts,
                   const double* __restrict__ xinv, double* __restrict__ sfwd, double* __restrict__ sbwd) {
  __shared__ double As[NB][NB + 1];
  __shared__ double Bs[NB][NB + 1];
  __shared__ double Ts[NB][NB + 1];
  int2 tk = tasks[blockIdx.x];
  int s = tk.x;
  int nc = d.sn_first[s + 1] - d.sn_first[s];
  int64_t f = nc + (d.sn_rowptr[s + 1] - d.sn_rowptr[s]);
  int r0 = tk.y * NB;
  const double* F = fronts + d.front_off[s];
  const double* X = xinv + d.xoff[s];
  double* S = sfwd + d.soff[s];
  double* St = sbwd + d.soff[s];
  const int thf = d.th_f[s], thb = d.th_b[s];   // tile-major storage above the cut of the solve plan (0: column-major)
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const bool below = r0 + NB > nc;          // the tile holds rows of L21
  for (int jb = 0; jb * NB < nc; ++jb) {
    int c0 = jb * NB;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    if (below)
      tile_gemm32(nc - c0,
                  [&](int i, int kk) { int r = r0 + i; return (r >= nc && r < f) ? F[r + (int64_t)(c0 + kk) * f] : 0.0; },
                  [&](int kk, int j) { return (c0 + j < nc) ? X[(c0 + kk) + (int64_t)(c0 + j) * nc] : 0.0; }, acc, As, Bs);
    int r = r0 + tx;
#pragma unroll
    for (int qq = 0; qq < 4; ++qq) {
      int c = c0 + ty + 8 * qq;
      double v = 0.0;
      if (r < f && c < nc) {
        v = (r < nc) ? X[r + (int64_t)c * nc] : -acc[qq];
        if (thf) {
          const int t0 = r / thf * thf;                        // first row of the row tile; th rows in it
          S[(int64_t)t0 * nc + (int64_t)c * min(thf, (int)f - t0) + (r - t0)] = v;
        } else {
          S[r + (int64_t)c * f] = v;
        }
      }
      Ts[tx][ty + 8 * qq] = v;
    }
    __syncthreads();
#pragma unroll
    for (int qq = 0; qq < 4; ++qq) {
      int rr = r0 + ty + 8 * qq, c = c0 + tx;
      if (rr < f && c < nc) {
        if (thb) {
          const int t0 = c / thb * thb;                        // first pivot column of the column tile; tw columns in it
          St[(int64_t)t0 * f + (int64_t)rr * min(thb, nc - t0) + (c - t0)] = Ts[ty + 8 * qq][tx];
        } else {
          St[c + (int64_t)rr * nc] = Ts[ty + 8 * qq][tx];
        }
      }
    }
    __syncthreads();
  }
}

}  // namespace


extern "C" int eigd_symbolic_assembly_map_device(eigd_symbolic* s, int n, const int* d_indptr, const int* d_indices,
                                                 int64_t* d_map) {
  if (n != s->n) { eigd_set_error("assembly_map_device: n mismatch"); return 1; }
  int rc = build_symdev(s);
  if (rc) return rc;
  auto* h = (SymDevHolder*)s->dev;
  int* err = nullptr;
  EIGD_CUDA(cudaMalloc((void**)&err, sizeof(int)));
  EIGD_CUDA(cudaMemsetAsync(err, 0, sizeof(int), g_eigd_stream));
  EIGD_LAUNCH(assembly_map_kernel, (n + 127) / 128, 128, 0, h->d, d_indptr, d_indices, d_map, err);
  EIGD_CHECK_LAUNCH();
  int herr = 0;
  EIGD_CUDA(cudaMemcpyAsync(&herr, err, sizeof(int), cudaMemcpyDeviceToHost, g_eigd_stream));
  EIGD_CUDA(cudaStreamSynchronize(g_eigd_stream));
  cudaFree(err);
  if (herr) { eigd_set_error("assembly_map_device: matrix entry outside the symbolic pattern"); return 2; }
  return 0;
}

static inline int64_t align256(int64_t b) { return (b + 255) / 256 * 256; }

// sizes (bytes, 256-aligned) of the device arrays of a factor, in carving order
constexpr int NARR = 16;
static void factor_layout(const eigd_symbolic* s, const SymDevHolder* h, int max_rhs, bool pooled, int64_t sz[NARR]) {
  int64_t nfront = s->front_off[s->nsuper], sumf = s->w_off[s->nsuper];
  int kc = std::min(max_rhs, 16);                      // the solve processes at most 16 columns per sweep
  sz[0] = pooled ? 0 : align256(nfront * 8);           // fronts (pooled: borrowed per numeric call)
  sz[1] = align256(h->linv_total * 8);                 // linv
  sz[2] = align256(h->xinv_total * 8);                 // xinv
  sz[3] = align256(h->xinv_total * 8);                 // xtmp
  sz[4] = align256(h->panel_total * 8 + 16);           // sfwd (+ one 16-byte unit: bulk copies round a slice up to 16 bytes)
  sz[5] = align256(h->panel_total * 8 + 16);           // sbwd
  sz[6] = align256((int64_t)s->n * 8);                 // dval
  sz[7] = align256((int64_t)s->n * 8);                 // dinv
  sz[8] = align256(3 * sumf * kc * 8);                 // wbuf: three child slabs, one plane per right-hand side
  sz[9] = align256((int64_t)s->n * kc * 8);            // ybuf
  sz[10] = align256((int64_t)s->n * kc * 8);           // xperm
  sz[11] = 256;                                        // amax
  sz[12] = 256;                                        // info
  sz[13] = align256(256 + (int64_t)s->nsuper * 8);     // grid-barrier counter (first 256 bytes) + completion counters of the solve
  sz[14] = align256((int64_t)s->n * kc * 8);           // bperm
  sz[15] = 0;
}

static bool fronts_mode_ok(int fronts) {
  if (fronts == 0 || fronts == 1) return true;
  eigd_set_error("factor: fronts mode %d (0 resident, 1 pooled)", fronts);
  return false;
}

extern "C" int64_t eigd_factor_workspace_bytes_fronts(eigd_symbolic* s, int max_rhs, int fronts) {
  if (!fronts_mode_ok(fronts) || build_symdev(s)) return -1;
  int64_t sz[NARR], tot = 0;
  factor_layout(s, (SymDevHolder*)s->dev, std::max(1, max_rhs), fronts == 1, sz);
  for (int i = 0; i < NARR; ++i) tot += sz[i];
  return tot + 256;
}

extern "C" int64_t eigd_factor_workspace_bytes(eigd_symbolic* s, int max_rhs) {
  return eigd_factor_workspace_bytes_fronts(s, max_rhs, 0);
}

// d_workspace == NULL: the library allocates (cudaMalloc) and owns the arrays; otherwise they are carved
// out of the caller's buffer (a torch tensor: the caching allocator then recycles it between factors)
extern "C" int eigd_factor_create_in_fronts(eigd_symbolic* s, int max_rhs, int fronts, void* d_workspace,
                                            int64_t workspace_bytes, eigd_factor** out) {
  if (!fronts_mode_ok(fronts)) return 1;
  int rc = fronts == 1 ? build_pool_plan(s) : build_symdev(s);
  if (rc) return rc;
  auto* f = new eigd_factor();
  f->sym = s;
  f->h = (SymDevHolder*)s->dev;
  f->max_rhs = std::max(1, max_rhs);
  f->pooled = fronts == 1;
  int64_t sz[NARR], tot = 0;
  factor_layout(s, f->h, f->max_rhs, f->pooled, sz);
  for (int i = 0; i < NARR; ++i) tot += sz[i];
  char* base = nullptr;
  if (d_workspace) {
    base = (char*)(((uintptr_t)d_workspace + 255) / 256 * 256);
    if ((base - (char*)d_workspace) + tot > workspace_bytes) {
      eigd_set_error("factor_create_in: workspace too small (%lld < %lld)", (long long)workspace_bytes, (long long)(tot + 256));
      delete f;
      return 3;
    }
    f->owns = false;
  } else {
    cudaError_t e = cudaMalloc((void**)&base, (size_t)tot);
    if (e != cudaSuccess) { eigd_set_error("factor_create: cudaMalloc(%lld) -> %s", (long long)tot, cudaGetErrorString(e)); delete f; return 100 + (int)e; }
    f->owns = true;
  }
  f->base = base;
  f->bytes = tot;
  char* p = base;
  f->fronts = f->pooled ? nullptr : (double*)p; p += sz[0];
  f->linv = (double*)p; p += sz[1];
  f->xinv = (double*)p; p += sz[2];
  f->xtmp = (double*)p; p += sz[3];
  f->sfwd = (double*)p; p += sz[4];
  f->sbwd = (double*)p; p += sz[5];
  f->dval = (double*)p; p += sz[6];
  f->dinv = (double*)p; p += sz[7];
  f->wbuf = (double*)p; p += sz[8];
  f->ybuf = (double*)p; p += sz[9];
  f->xperm = (double*)p; p += sz[10];
  f->amax = (unsigned long long*)p; p += sz[11];
  f->info = (unsigned long long*)p; p += sz[12];
  f->barrier = (unsigned long long*)p;
  f->cnt = (unsigned*)(p + 256); p += sz[13];
  f->epoch = 0;
  f->bperm = (double*)p;
  f->bar_base = 0;
  // slab rows that no child writes must read as zero for ever; the written ones are rewritten by every solve
  cudaError_t eb = cudaMemsetAsync(f->wbuf, 0, (size_t)sz[8], g_eigd_stream);
  if (eb == cudaSuccess) eb = cudaMemsetAsync(f->barrier, 0, (size_t)sz[13], g_eigd_stream);
  if (eb != cudaSuccess) { eigd_set_error("factor_create: memset -> %s", cudaGetErrorString(eb)); eigd_factor_destroy(f); return 100 + (int)eb; }
  *out = f;
  return 0;
}

extern "C" int eigd_factor_create_in(eigd_symbolic* s, int max_rhs, void* d_workspace, int64_t workspace_bytes,
                                     eigd_factor** out) {
  return eigd_factor_create_in_fronts(s, max_rhs, 0, d_workspace, workspace_bytes, out);
}

extern "C" int eigd_factor_create(eigd_symbolic* s, int max_rhs, eigd_factor** out) {
  return eigd_factor_create_in(s, max_rhs, nullptr, 0, out);
}

extern "C" void eigd_factor_destroy(eigd_factor* f) {
  if (!f) return;
  if (f->owns && f->base) cudaFree(f->base);
  delete f;
}

extern "C" int64_t eigd_factor_bytes(const eigd_factor* f) { return f->bytes; }

// The launches of a factor plan.  d: the device symbolic data with front_off pointing at the fronts' layout
// (front_off for resident fronts, pool_off for pooled ones); vals / seg / ent: the inputs of kind 8 (pooled only).
static int run_factor_plan(eigd_factor* f, const std::vector<Launch>& plan, const int2* tasks, const SymDev& d,
                           double* fronts, const double* vals, const int64_t* seg, const int2* ent) {
  eigd_symbolic* s = f->sym;
  // developer profiling (EIGD_FACTOR_PROF=1): device time per launch kind, synchronising after every launch
  static int prof = -1;
  if (prof < 0) { const char* e = getenv("EIGD_FACTOR_PROF"); prof = e ? atoi(e) : 0; }
  double kind_ms[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  int kind_n[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  cudaEvent_t pe0 = nullptr, pe1 = nullptr;
  if (prof) { cudaEventCreate(&pe0); cudaEventCreate(&pe1); }
  for (const Launch& L : plan) {
    const int2* t = tasks + L.off;
    if (prof) cudaEventRecord(pe0, g_eigd_stream);
    switch (L.kind) {
      case 0: EIGD_LAUNCH(extend_add_kernel, L.count, 256, 0, d, t, fronts); break;
      case 1:
        if (f->pivoting) EIGD_LAUNCH(diag_factor_bk_kernel, L.count, 256, 0, d, t, L.kb, fronts, f->linv, f->dval, f->dinv, f->amax, f->piv_tol, f->info);
        else EIGD_LAUNCH(diag_factor_kernel, L.count, 256, 0, d, t, L.kb, fronts, f->linv, f->dval, f->dinv, f->amax, f->piv_tol, f->info);
        break;
      case 2:
        if (f->pivoting) EIGD_LAUNCH(trsm_kernel<true>, L.count, TRSM_ROWS, 0, d, t, L.kb, fronts, f->linv, f->dinv);
        else EIGD_LAUNCH(trsm_kernel<false>, L.count, TRSM_ROWS, 0, d, t, L.kb, fronts, f->linv, f->dinv);
        break;
      case 3: EIGD_LAUNCH(trailing_update_kernel, L.count, 256, 0, d, t, L.kb, fronts, f->dval); break;
      case 4:
        if (f->pivoting) EIGD_LAUNCH(inverse_init_kernel<true>, L.count, 256, 0, d, t, f->linv, f->xinv);
        else EIGD_LAUNCH(inverse_init_kernel<false>, L.count, 256, 0, d, t, f->linv, f->xinv);
        break;
      case 5: EIGD_LAUNCH(inverse_ca_kernel, L.count, 256, 0, d, t, NB << L.kb, fronts, f->xinv, f->xtmp); break;
      case 6: EIGD_LAUNCH(inverse_bt_kernel, L.count, 256, 0, d, t, NB << L.kb, f->xinv, f->xtmp); break;
      case 7: EIGD_LAUNCH(panel_build_kernel, L.count, 256, 0, d, t, fronts, f->xinv, f->sfwd, f->sbwd); break;
      case 8: EIGD_LAUNCH(front_assemble_kernel, L.count, 256, 0, d, t, vals, seg, ent, fronts); break;
      default: break;
    }
    EIGD_CHECK_LAUNCH();
    if (prof) {
      cudaEventRecord(pe1, g_eigd_stream);
      cudaEventSynchronize(pe1);
      float ms = 0.f;
      cudaEventElapsedTime(&ms, pe0, pe1);
      kind_ms[L.kind] += ms;
      kind_n[L.kind]++;
    }
  }
  if (prof) {
    static const char* names[9] = {"extend_add", "diag_factor", "trsm", "trailing_update", "inverse_init", "inverse_ca",
                                   "inverse_bt", "panel_build", "front_assemble"};
    fprintf(stderr, "[factor prof] n=%d levels=%d%s:", s->n, s->nlevels, f->pooled ? " pooled" : "");
    for (int k = 0; k < (f->pooled ? 9 : 8); ++k) fprintf(stderr, " %s %.3f ms / %d;", names[k], kind_ms[k], kind_n[k]);
    fprintf(stderr, "\n");
    cudaEventDestroy(pe0);
    cudaEventDestroy(pe1);
  }
  return 0;
}

// the per-call set-up both modes share: pivot statistics, |A|max for the pivot threshold, zeroed full inverses
static int numeric_begin(eigd_factor* f, int64_t nnz, const double* d_vals, int* grid) {
  EIGD_CUDA(cudaMemsetAsync(f->amax, 0, 8, g_eigd_stream));
  EIGD_CUDA(cudaMemsetAsync(f->info, 0, f->pivoting ? 40 : 32, g_eigd_stream));
  EIGD_CUDA(cudaMemsetAsync(f->xinv, 0, (size_t)std::max<int64_t>(f->h->xinv_total, 1) * 8, g_eigd_stream));
  int g = (int)std::min<int64_t>((nnz + 255) / 256, 148 * 16);
  if (g < 1) g = 1;
  EIGD_LAUNCH(absmax_kernel, g, 256, 0, nnz, d_vals, f->amax);
  EIGD_CHECK_LAUNCH();
  *grid = g;
  return 0;
}

extern "C" int eigd_factor_numeric(eigd_factor* f, int64_t nnz, const double* d_vals, const int64_t* d_map) {
  if (f->pooled) { eigd_set_error("factor_numeric: this factor has pooled fronts; use eigd_factor_numeric_pool"); return 1; }
  eigd_symbolic* s = f->sym;
  SymDevHolder* h = f->h;
  int64_t nfront = s->front_off[s->nsuper];
  EIGD_CUDA(cudaMemsetAsync(f->fronts, 0, (size_t)nfront * 8, g_eigd_stream));
  int g = 0, rc = numeric_begin(f, nnz, d_vals, &g);
  if (rc) return rc;
  EIGD_LAUNCH(scatter_values_kernel, g, 256, 0, nnz, d_vals, d_map, f->fronts);
  EIGD_CHECK_LAUNCH();
  return run_factor_plan(f, h->factor_plan, h->tasks, h->d, f->fronts, nullptr, nullptr, nullptr);
}

extern "C" int eigd_factor_numeric_pool(eigd_factor* f, int64_t nnz, const double* d_vals, const int64_t* d_seg,
                                        const int* d_ent, void* d_pool, int64_t pool_bytes) {
  if (!f->pooled) { eigd_set_error("factor_numeric_pool: this factor has resident fronts; use eigd_factor_numeric"); return 1; }
  eigd_symbolic* s = f->sym;
  SymDevHolder* h = f->h;
  const int64_t need = s->pool_doubles * 8;
  if (!d_pool || pool_bytes < need) {
    eigd_set_error("factor_numeric_pool: front pool of %lld bytes, the fronts need %lld (eigd_symbolic_query(s, 10) doubles)",
                   (long long)pool_bytes, (long long)need);
    return 3;
  }
  if ((uintptr_t)d_pool % 256) { eigd_set_error("factor_numeric_pool: the front pool must be 256-byte aligned"); return 3; }
  int g = 0, rc = numeric_begin(f, nnz, d_vals, &g);
  if (rc) return rc;
  SymDev d = h->d;
  d.front_off = h->pool_off;
  return run_factor_plan(f, h->pool_plan, h->pool_tasks, d, (double*)d_pool, d_vals, d_seg, (const int2*)d_ent);
}

// ---- FP64 tensor-pipe peak of this GPU, measured: every warp of every SM issues independent DMMA chains on register
// operands (8 accumulator pairs per warp, no memory traffic).  bench.py divides the factorisation's flop rate by it
// (roofline_fp64_tensor); profiles/ holds the ncu pipe utilisation of trailing_update_kernel next to it.
__global__ void __launch_bounds__(256) dmma_peak_kernel(int iters, double* __restrict__ sink) {
  double c[8][2];
#pragma unroll
  for (int i = 0; i < 8; ++i) { c[i][0] = 0.0; c[i][1] = 0.0; }
  double a = 1.0 + 1e-9 * threadIdx.x, b = 1.0 - 1e-9 * threadIdx.x;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 8; ++i) dmma_m8n8k4(c[i][0], c[i][1], a, b);
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += c[i][0] + c[i][1];
  if (s == 123.456) sink[0] = s;          // keep the chains alive
}

// -> TFLOP/s (2 * 8 * 8 * 4 flop per warp-level MMA), best of `reps` timed launches on the library's stream
extern "C" int eigd_dmma_peak(int iters, int reps, double* tflops_out) {
  int dev = 0, sms = 0;
  EIGD_CUDA(cudaGetDevice(&dev));
  EIGD_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  double* sink = nullptr;
  EIGD_CUDA(cudaMalloc((void**)&sink, 8));
  cudaEvent_t e0, e1;
  EIGD_CUDA(cudaEventCreate(&e0));
  EIGD_CUDA(cudaEventCreate(&e1));
  const int grid = sms * 8, block = 256;
  double best = 0.0;
  for (int r = 0; r < reps + 1; ++r) {
    EIGD_CUDA(cudaEventRecord(e0, g_eigd_stream));
    EIGD_LAUNCH(dmma_peak_kernel, grid, block, 0, iters, sink);
    EIGD_CHECK_LAUNCH();
    EIGD_CUDA(cudaEventRecord(e1, g_eigd_stream));
    EIGD_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    EIGD_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    const double flops = (double)grid * (block / 32) * (double)iters * 8.0 * 512.0;
    if (r > 0 && ms > 0.f) best = std::max(best, flops / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(sink);
  *tflops_out = best;
  return 0;
}

extern "C" int eigd_factor_set_pivoting(eigd_factor* f, int mode) {
  if (mode != 0 && mode != 1) { eigd_set_error("factor_set_pivoting: mode %d (0 static, 1 restricted Bunch-Kaufman)", mode); return 1; }
  f->pivoting = mode;
  return 0;
}

extern "C" int eigd_factor_pivot_counts(eigd_factor* f, int64_t* out2) {
  out2[0] = out2[1] = 0;
  if (!f->pivoting) return 0;
  unsigned long long h[2];
  EIGD_CUDA(cudaMemcpyAsync(h, f->info + 3, 16, cudaMemcpyDeviceToHost, g_eigd_stream));
  EIGD_CUDA(cudaStreamSynchronize(g_eigd_stream));
  out2[0] = (int64_t)h[0];
  out2[1] = (int64_t)h[1];
  return 0;
}

extern "C" int eigd_factor_info(eigd_factor* f, int64_t* info3) {
  unsigned long long hinfo[4];
  EIGD_CUDA(cudaMemcpyAsync(hinfo, f->info, 32, cudaMemcpyDeviceToHost, g_eigd_stream));
  EIGD_CUDA(cudaStreamSynchronize(g_eigd_stream));
  for (int i = 0; i < 3; ++i) info3[i] = (int64_t)hinfo[i];
  return 0;
}

