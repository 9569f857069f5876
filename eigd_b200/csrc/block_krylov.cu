// Device-resident BLOCK shift-and-invert Lanczos recurrence (block size P = 2 .. 4).
//
// Why a block method: on B200 a sparse triangular solve is bound by the dependency depth of the assembly tree,
// not by bandwidth, so P right-hand sides cost little more than one (DESIGN.md section 5) -- and the tall-skinny
// orthogonalisation products read the Krylov basis once for all P new vectors.  The block recurrence needs about
// the same number of operator applications as the single-vector one (measured on the bench problems), i.e. 1/P of
// the sequential solves.  Replaces, like krylov.cu, the reverse-communication loop of reference eigd/arpack.py:438-442
// (ARPACK dsaupd is a single-vector method; the (d, z, Tm, v) contract of eigd/arpack.py:58-101 -- v^T B v = I,
// Tm = v^T B OP v, z = v y -- holds for the block basis as well; Tm is block tridiagonal plus the restart arrow).
//
// One call runs the block steps of a restart cycle without returning to the host.  Per step (m = basis vectors so far,
// j = first vector of the block being expanded):
//     W   = factor^{-1} BV[j : j+P]                      (one P-column eigd_factor_apply)
//     H1  = BV[lo:m] W, W -= V[lo:m]^T H1                (local Gram-Schmidt pass in the B inner product: lo = j - P, the two
//                                                         blocks of the three-term recurrence; lo = 0 after a restart)
//     H2  = BV[0:m] W,  W -= V[0:m]^T H2                 (unconditional full pass: full reorthogonalisation)
//     BW  = B W,  G = W^T BW = R1^T R1,  W <- W R1^-1, BW <- BW R1^-1      (Cholesky QR ...
//     G2  = W^T BW = R2^T R2,  W <- W R2^-1, BW <- BW R2^-1                 ... twice: orthonormal to rounding)
//     V[m : m+P] = W, BV[m : m+P] = BW;  A_j = (H1 + H2)[j : j+P] (diagonal block), R_j = R2 R1 (sub-diagonal block)
// Everything after the solve is ONE cooperative launch per step (block_step_kernel: CTAs own 1024-element chunks of n,
// software grid barriers only where a dot product crosses CTAs, bitwise-reproducible fixed-order sums); the small
// P x P factorisations run in one thread of every CTA (no host round trip inside a cycle).
//
// Storage as in krylov.cu: V and BV are (ncv + P) x n row-major (one vector per row, leading dimension ld).
#include "common.cuh"
#include "../../include/eigd_b200.h"

#include <algorithm>

namespace {

constexpr int BK_THREADS = 256;
constexpr int BK_WARPS = BK_THREADS / 32;
constexpr int BK_EPT = 4;                        // elements per thread and chunk
constexpr int BK_CHUNK = BK_THREADS * BK_EPT;
constexpr int BK_JMAX = 128;                     // basis vectors per launch
constexpr int BK_PMAX = 4;
constexpr int BK_RMAX = BK_JMAX + BK_PMAX;       // basis rows a Gram-Schmidt pass can see

// Cholesky G = R^T R of the P x P Gram matrix (row-major G[a * P + c]); writes the inverse Rinv (upper triangular,
// row-major) for the scaling kernel and accumulates Racc <- R * Racc (Racc = identity on the first pass: pass 0).
// A non-positive pivot (rank-deficient block: breakdown) is flagged by NaNs, which the host checks once per cycle.
template <int P>
__device__ void block_chol(const double* __restrict__ G, double* __restrict__ Rinv, double* __restrict__ Racc, int pass) {
  double R[P][P], X[P][P];
#pragma unroll
  for (int a = 0; a < P; ++a)
#pragma unroll
    for (int c = 0; c < P; ++c) { R[a][c] = 0.0; X[a][c] = 0.0; }
  bool ok = true;
#pragma unroll
  for (int c = 0; c < P; ++c) {                  // column-by-column (upper factor): R[a][c], a <= c
#pragma unroll
    for (int a = 0; a <= c; ++a) {
      double s = 0.5 * (G[a * P + c] + G[c * P + a]);
#pragma unroll
      for (int t = 0; t < a; ++t) s -= R[t][a] * R[t][c];
      if (a < c) R[a][c] = s / R[a][a];
      else {
        if (!(s > 0.0)) ok = false;
        R[c][c] = sqrt(s);
      }
    }
  }
  // X = R^-1 (upper triangular) by back substitution
#pragma unroll
  for (int c = 0; c < P; ++c) {
    X[c][c] = 1.0 / R[c][c];
#pragma unroll
    for (int a = c - 1; a >= 0; --a) {
      double s = 0.0;
#pragma unroll
      for (int t = a + 1; t <= c; ++t) s += R[a][t] * X[t][c];
      X[a][c] = -s / R[a][a];
    }
  }
  const double bad = ok ? 0.0 : __longlong_as_double(0x7ff8000000000000LL);
#pragma unroll
  for (int a = 0; a < P; ++a)
#pragma unroll
    for (int c = 0; c < P; ++c) Rinv[a * P + c] = X[a][c] + bad;
  double A[P][P];
#pragma unroll
  for (int a = 0; a < P; ++a)
#pragma unroll
    for (int c = 0; c < P; ++c) {
      if (pass == 0) A[a][c] = R[a][c];
      else {
        double s = 0.0;
#pragma unroll
        for (int t = 0; t < P; ++t) s += R[a][t] * Racc[t * P + c];
        A[a][c] = s;
      }
    }
#pragma unroll
  for (int a = 0; a < P; ++a)
#pragma unroll
    for (int c = 0; c < P; ++c) Racc[a * P + c] = A[a][c] + bad;
}

// ---- one block step as one cooperative launch ------------------------------------------------------------------
// Every dot product keeps the summation order of the separate dots / reduce kernels this launch replaced, so the
// results do not depend on the grid: a pass over J basis rows has the virtual grid gv = min(ceil(n / 1024), cap(J P));
// virtual CTA v adds its chunks v, v + gv, ... (per thread a 4-term fma chain, warp_sum, per warp in chunk order),
// then its 8 warps in order into partial[v]; an output is the lane-strided sum over the gv partials, then warp_sum.
// A CTA runs the virtual CTAs blockIdx.x, blockIdx.x + gridDim.x, ...  Axpy, scaling and B W are per element or per
// row and keep their own order (basis rows ascending, CSR order), whatever CTA computes them.
struct StepArgs {
  int64_t n, ld;
  const double* V;            // basis V[0:m] and BV[0:m] (rows, leading dimension ld)
  const double* BV;
  double* W;                  // the new block V[m : m+P] (on entry: the solve's output) and BV[m : m+P]
  double* BW;
  int m, lo, j;               // local pass against rows lo .. m-1, full pass against 0 .. m-1; A_j = rows j .. j+P-1
  int gs;                     // 0: start block (B W and the Cholesky QR only)
  int split;                  // the two partial-sum regions overlap: one barrier more between reading and rewriting
  int gv1, gv2, gvg;          // virtual grids of the local pass, the full pass and the P x P Gram matrices
  double* part_a;             // partial sums of the local pass and of the first Gram matrix
  double* part_b;             // partial sums of the full pass and of the second Gram matrix
  double *H1, *H2, *Aout, *Rout, *scratch;
  const int *bp, *bi;
  const double* bv;
  unsigned long long* ctr;
  unsigned long long base;
};

// this thread's elements i0 + q * 256 of the P rows W[c * ld + i] (zero past n)
template <int P>
__device__ __forceinline__ void load_block(double (&w)[P][BK_EPT], const double* W, int64_t ld, int64_t i0, int64_t n) {
#pragma unroll
  for (int c = 0; c < P; ++c)
#pragma unroll
    for (int q = 0; q < BK_EPT; ++q) {
      const int64_t i = i0 + (int64_t)q * BK_THREADS;
      w[c][q] = (i < n) ? __ldcg(W + (int64_t)c * ld + i) : 0.0;
    }
}

template <int P>
__device__ __forceinline__ void store_block(const double (&w)[P][BK_EPT], double* W, int64_t ld, int64_t i0, int64_t n) {
#pragma unroll
  for (int c = 0; c < P; ++c)
#pragma unroll
    for (int q = 0; q < BK_EPT; ++q) {
      const int64_t i = i0 + (int64_t)q * BK_THREADS;
      if (i < n) W[(int64_t)c * ld + i] = w[c][q];
    }
}

template <int R>
__device__ __forceinline__ void load_rows(double (&v)[R][BK_EPT], const double* __restrict__ Vb, int64_t ld, int a0,
                                          int rows, int64_t i0, int64_t n) {
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const double* row = Vb + (int64_t)(a0 + r) * ld;
    const bool ok = a0 + r < rows;
#pragma unroll
    for (int q = 0; q < BK_EPT; ++q) {
      const int64_t i = i0 + (int64_t)q * BK_THREADS;
      v[r][q] = (ok && i < n) ? __ldg(row + i) : 0.0;
    }
  }
}

// f(v, a0) on this thread's elements of the rows a0 .. a0 + R - 1 of Vb[0:rows], ascending; the loads of the next
// group are issued before f runs on the current one (with one group per trip every trip waited for its own round trip)
template <int R, class F>
__device__ __forceinline__ void sweep_rows(const double* __restrict__ Vb, int64_t ld, int rows, int64_t i0, int64_t n, F&& f) {
  double va[R][BK_EPT], vb[R][BK_EPT];
  load_rows<R>(va, Vb, ld, 0, rows, i0, n);
  for (int a0 = 0; a0 < rows; a0 += 2 * R) {
    const int a1 = a0 + R;
    if (a1 < rows) load_rows<R>(vb, Vb, ld, a1, rows, i0, n);
    f(va, a0);
    if (a1 >= rows) break;
    if (a1 + R < rows) load_rows<R>(va, Vb, ld, a1 + R, rows, i0, n);
    f(vb, a1);
  }
}

// myred[(a0 + r) * P + c] += warp_sum(sum_q v[r][q] w[c][q]) for the rows a0 + r < rows
template <int R, int P>
__device__ __forceinline__ void dot_rows(const double (&v)[R][BK_EPT], const double (&w)[P][BK_EPT], int a0, int rows,
                                         double* myred) {
#pragma unroll
  for (int r = 0; r < R; ++r) {
    if (a0 + r >= rows) break;
#pragma unroll
    for (int c = 0; c < P; ++c) {
      double s = 0.0;
#pragma unroll
      for (int q = 0; q < BK_EPT; ++q) s = fma(v[r][q], w[c][q], s);
      s = warp_sum(s);
      if ((threadIdx.x & 31) == 0) myred[(a0 + r) * P + c] += s;
    }
  }
}

// w[c][q] += hs[(a0 + r) * P + c] * v[r][q] for the rows a0 + r < rows (hs holds -H)
template <int R, int P>
__device__ __forceinline__ void axpy_rows(const double (&v)[R][BK_EPT], double (&w)[P][BK_EPT], int a0, int rows,
                                          const double* hs) {
#pragma unroll
  for (int r = 0; r < R; ++r) {
    if (a0 + r >= rows) break;
#pragma unroll
    for (int c = 0; c < P; ++c) {
      const double h = hs[(a0 + r) * P + c];
#pragma unroll
      for (int q = 0; q < BK_EPT; ++q) w[c][q] = fma(h, v[r][q], w[c][q]);
    }
  }
}

// W <- W Rinv, BW <- BW Rinv (x = Rinv, upper triangular, row-major)
template <int P>
__device__ __forceinline__ void scale_block(double (&w)[P][BK_EPT], double (&b)[P][BK_EPT], const double* x) {
#pragma unroll
  for (int q = 0; q < BK_EPT; ++q)
#pragma unroll
    for (int c = P - 1; c >= 0; --c) {
      double sw = 0.0, sb = 0.0;
#pragma unroll
      for (int t = 0; t <= c; ++t) { sw = fma(w[t][q], x[t * P + c], sw); sb = fma(b[t][q], x[t * P + c], sb); }
      w[c][q] = sw;
      b[c][q] = sb;
    }
}

// b = B W on this thread's rows of the chunk (W of every row from global memory).  The four rows run in lock step,
// two entries each per trip (all index loads, then all gathers); per row and column the products are added in CSR
// order, as in spmm_kernel.
template <int P>
__device__ __forceinline__ void spmm_rows(double (&b)[P][BK_EPT], const int* __restrict__ bp, const int* __restrict__ bi,
                                          const double* __restrict__ bv, const double* W, int64_t ld, int64_t i0, int64_t n) {
  constexpr int U = 2;
  int p[BK_EPT], e[BK_EPT];
#pragma unroll
  for (int q = 0; q < BK_EPT; ++q) {
    const int64_t i = i0 + (int64_t)q * BK_THREADS;
    p[q] = i < n ? bp[i] : 0;
    e[q] = i < n ? bp[i + 1] : 0;
#pragma unroll
    for (int c = 0; c < P; ++c) b[c][q] = 0.0;
  }
  for (int t = 0;; t += U) {
    int idx[BK_EPT][U];
    double val[BK_EPT][U], x[BK_EPT][U][P];
#pragma unroll
    for (int q = 0; q < BK_EPT; ++q)
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int pp = p[q] + t + u;
        idx[q][u] = pp < e[q] ? bi[pp] : 0;
        val[q][u] = pp < e[q] ? bv[pp] : 0.0;
      }
#pragma unroll
    for (int q = 0; q < BK_EPT; ++q)
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int c = 0; c < P; ++c) x[q][u][c] = p[q] + t + u < e[q] ? __ldcg(W + (int64_t)c * ld + idx[q][u]) : 0.0;
    bool more = false;
#pragma unroll
    for (int q = 0; q < BK_EPT; ++q) {
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (p[q] + t + u < e[q])
#pragma unroll
          for (int c = 0; c < P; ++c) b[c][q] = fma(val[q][u], x[q][u][c], b[c][q]);
      more |= p[q] + t + U < e[q];
    }
    if (!more) break;
  }
#pragma unroll
  for (int q = 0; q < BK_EPT; ++q)
#pragma unroll
    for (int c = 0; c < P; ++c) b[c][q] = fma(1.0, b[c][q], 0.0);       // Y = alpha acc + 0 of spmm_kernel
}

// The partial sums of one pass (see above): chunk(i0, myred) adds a chunk's dot products into this warp's row of red.
template <class F>
__device__ __forceinline__ void pass_partials(int gv, int64_t nch, int JP, double* red, double* partial, F&& chunk) {
  const int tid = threadIdx.x;
  for (int v = blockIdx.x; v < gv; v += gridDim.x) {
    for (int e = tid; e < BK_WARPS * JP; e += BK_THREADS) red[e] = 0.0;
    __syncthreads();
    for (int64_t ch = v; ch < nch; ch += gv) chunk(ch * BK_CHUNK + tid, red + (tid >> 5) * JP);
    __syncthreads();
    for (int e = tid; e < JP; e += BK_THREADS) {
      double s = 0.0;
#pragma unroll
      for (int g = 0; g < BK_WARPS; ++g) s += red[g * JP + e];
      partial[(int64_t)v * JP + e] = s;
    }
    __syncthreads();
  }
}

// output e of a pass (after a grid barrier): lanes stride over the gv partials, then warp_sum
__device__ __forceinline__ double reduce_partial(const double* partial, int gv, int JP, int e) {
  double s = 0.0;
  for (int c = threadIdx.x & 31; c < gv; c += 32) s += __ldcg(partial + (int64_t)c * JP + e);
  return warp_sum(s);
}

// every CTA reduces all JP outputs: hs[e] = sign * out[e], and out[e] to global memory when g is set
__device__ __forceinline__ void reduce_all(const double* partial, int gv, int JP, double sign, double* hs, double* g) {
  for (int e = threadIdx.x >> 5; e < JP; e += BK_WARPS) {
    const double s = reduce_partial(partial, gv, JP, e);
    if ((threadIdx.x & 31) == 0) {
      hs[e] = sign * s;
      if (g) g[e] = s;
    }
  }
  __syncthreads();
}

// One block step after the P-column solve ('|' is a grid barrier):
//   1. partial sums of H1 = BV[lo:m] W                                                                   |
//   2. H1; W -= V[lo:m]^T H1 and, in the same sweep over the chunk, partial sums of H2 = BV[0:m] W       |
//      H2, one warp per output across the grid                                                          |
//   3. W -= V[0:m]^T H2 -> V[m : m+P]; A_j = (H1 + H2)[j : j+P]                                          |
//   4. BW = B W -> BV[m : m+P]; partial sums of G1 = BW^T W                                              |
//   5. R1 from G1 (every CTA); W, BW <- W, BW R1^-1; partial sums of G2                                 |
//   6. R2 from G2; W, BW <- W, BW R2^-1; R_j = R2 R1
// The start block runs stages 4 to 6.  W and BW are re-read from L2 in each stage (they are written by other CTAs'
// stages; 2 P n doubles), V[0:m] and BV[0:m] stream from HBM once per pass.
template <int P>
__global__ void __launch_bounds__(BK_THREADS, 2) block_step_kernel(StepArgs a) {
  __shared__ double red[BK_WARPS * BK_RMAX * P];
  __shared__ double hs[BK_RMAX * P];
  __shared__ double rinv[P * P], racc[P * P];
  const int tid = threadIdx.x;
  const int64_t n = a.n, ld = a.ld;
  const int64_t nch = (n + BK_CHUNK - 1) / BK_CHUNK;
  unsigned long long target = a.base;
  auto grid_barrier = [&]() {
    target += gridDim.x;
    coop_grid_barrier(a.ctr, target);
  };
  constexpr int R = P <= 2 ? 4 : 2;           // basis rows per load group (see sweep_rows): registers of 2 CTAs per SM
  using Rows = double[R][BK_EPT];
  if (a.gs) {
    const int J1 = a.m - a.lo, J2 = a.m;
    const double* Vlo = a.V + (int64_t)a.lo * ld;
    const double* BVlo = a.BV + (int64_t)a.lo * ld;
    pass_partials(a.gv1, nch, J1 * P, red, a.part_a, [&](int64_t i0, double* myred) {
      double w[P][BK_EPT];
      load_block<P>(w, a.W, ld, i0, n);
      sweep_rows<R>(BVlo, ld, J1, i0, n, [&](const Rows& v, int a0) { dot_rows<R, P>(v, w, a0, J1, myred); });
    });
    grid_barrier();
    reduce_all(a.part_a, a.gv1, J1 * P, -1.0, hs, blockIdx.x == 0 ? a.H1 : nullptr);
    if (a.split) grid_barrier();
    pass_partials(a.gv2, nch, J2 * P, red, a.part_b, [&](int64_t i0, double* myred) {
      double w[P][BK_EPT];
      load_block<P>(w, a.W, ld, i0, n);
      sweep_rows<R>(Vlo, ld, J1, i0, n, [&](const Rows& v, int a0) { axpy_rows<R, P>(v, w, a0, J1, hs); });
      store_block<P>(w, a.W, ld, i0, n);
      sweep_rows<R>(a.BV, ld, J2, i0, n, [&](const Rows& v, int a0) { dot_rows<R, P>(v, w, a0, J2, myred); });
    });
    grid_barrier();
    for (int e = blockIdx.x * BK_WARPS + (tid >> 5); e < J2 * P; e += gridDim.x * BK_WARPS) {
      const double s = reduce_partial(a.part_b, a.gv2, J2 * P, e);
      if ((tid & 31) == 0) a.H2[e] = s;
    }
    grid_barrier();
    for (int e = tid; e < J2 * P; e += BK_THREADS) hs[e] = -1.0 * __ldcg(a.H2 + e);
    if (blockIdx.x == 0 && tid < P * P) a.Aout[tid] = __ldcg(a.H1 + (a.j - a.lo) * P + tid) + __ldcg(a.H2 + a.j * P + tid);
    __syncthreads();
    for (int64_t ch = blockIdx.x; ch < nch; ch += gridDim.x) {
      const int64_t i0 = ch * BK_CHUNK + tid;
      double w[P][BK_EPT];
      load_block<P>(w, a.W, ld, i0, n);
      sweep_rows<R>(a.V, ld, J2, i0, n, [&](const Rows& v, int a0) { axpy_rows<R, P>(v, w, a0, J2, hs); });
      store_block<P>(w, a.W, ld, i0, n);
    }
    grid_barrier();
  }
  pass_partials(a.gvg, nch, P * P, red, a.part_a, [&](int64_t i0, double* myred) {
    double w[P][BK_EPT], b[P][BK_EPT];
    spmm_rows<P>(b, a.bp, a.bi, a.bv, a.W, ld, i0, n);
    store_block<P>(b, a.BW, ld, i0, n);
    load_block<P>(w, a.W, ld, i0, n);
    dot_rows<P, P>(b, w, 0, P, myred);
  });
  grid_barrier();
  reduce_all(a.part_a, a.gvg, P * P, 1.0, hs, blockIdx.x == 0 ? a.scratch : nullptr);
  if (tid == 0) block_chol<P>(hs, rinv, racc, 0);
  __syncthreads();
  if (blockIdx.x == 0 && tid < P * P) a.scratch[P * P + tid] = rinv[tid];
  if (a.split) grid_barrier();
  pass_partials(a.gvg, nch, P * P, red, a.part_b, [&](int64_t i0, double* myred) {
    double w[P][BK_EPT], b[P][BK_EPT];
    load_block<P>(w, a.W, ld, i0, n);
    load_block<P>(b, a.BW, ld, i0, n);
    scale_block<P>(w, b, rinv);
    store_block<P>(w, a.W, ld, i0, n);
    store_block<P>(b, a.BW, ld, i0, n);
    dot_rows<P, P>(b, w, 0, P, myred);
  });
  grid_barrier();
  reduce_all(a.part_b, a.gvg, P * P, 1.0, hs, blockIdx.x == 0 ? a.scratch : nullptr);
  if (tid == 0) block_chol<P>(hs, rinv, racc, 1);
  __syncthreads();
  if (blockIdx.x == 0 && tid < P * P) {
    a.scratch[P * P + tid] = rinv[tid];
    a.Rout[tid] = racc[tid];
  }
  for (int64_t ch = blockIdx.x; ch < nch; ch += gridDim.x) {
    const int64_t i0 = ch * BK_CHUNK + tid;
    double w[P][BK_EPT], b[P][BK_EPT];
    load_block<P>(w, a.W, ld, i0, n);
    load_block<P>(b, a.BW, ld, i0, n);
    scale_block<P>(w, b, rinv);
    store_block<P>(w, a.W, ld, i0, n);
    store_block<P>(b, a.BW, ld, i0, n);
  }
}

// Launches block_step_kernel<P> for a (its grid, virtual grids, partial-sum regions and barrier base are set here).
// work: the eigd_gemm_tn_workspace buffer, which bounds every virtual grid (gv x outputs must fit) as it bounded the
// grids of the separate dots kernels.
template <int P>
int block_step(StepArgs a, double* work) {
  static int max_grid = 0;
  int rc;
  unsigned long long *ctr = nullptr, *base = nullptr;
  if ((rc = coop_counter(&ctr, &base)) || (rc = coop_max_grid(block_step_kernel<P>, 1 << 20, 1 << 30, &max_grid))) return rc;
  const int64_t ws = eigd_gemm_tn_workspace(32, 32);
  const int64_t nch = (a.n + BK_CHUNK - 1) / BK_CHUNK;
  auto vgrid = [&](int J) {
    const int64_t cap = ws / ((int64_t)J * P);
    return (int)(nch < cap ? nch : cap);
  };
  a.gvg = vgrid(P);
  int64_t size_a = (int64_t)a.gvg * P * P, size_b = size_a;
  if (a.gs) {
    a.gv1 = vgrid(a.m - a.lo);
    a.gv2 = vgrid(a.m);
    if (a.gv2 < 1) { eigd_set_error("block_lanczos: workspace too small"); return 8; }
    size_a = std::max(size_a, (int64_t)a.gv1 * (a.m - a.lo) * P);
    size_b = std::max(size_b, (int64_t)a.gv2 * a.m * P);
  }
  a.part_b = work;
  a.part_a = work + (ws - size_a);
  a.split = size_a + size_b > ws;
  a.ctr = ctr;
  a.base = *base;
  const int grid = (int)(nch < max_grid ? nch : max_grid);
  void* params[] = {(void*)&a};
  EIGD_CUDA(cudaLaunchCooperativeKernel((void*)block_step_kernel<P>, dim3(grid), dim3(BK_THREADS), params, 0, g_eigd_stream));
  ++g_eigd_launches;
  const int barriers = (a.gs ? 6 : 2) + a.split * (a.gs ? 2 : 1);
  *base += (unsigned long long)barriers * (unsigned long long)grid;
  return 0;
}

template <int P>
int extend(eigd_factor* f, int n, const int* bp, const int* bi, const double* bv, double* V, double* BV, int64_t ld, int j0,
           int m0, int ncv, double* Ablk, double* Rblk, double* H1, double* H2, double* scratch, double* work) {
  int rc;
  int step = 0;
  for (int j = j0, m = m0; j < ncv; j += P, m += P, ++step) {
    const double* bvj = BV + (int64_t)j * ld;
    double* W = V + (int64_t)m * ld;
    // W = OP V_j = factor^{-1} (B V_j): the P vectors are rows (stride ld between vectors, 1 inside)
    if ((rc = eigd_factor_apply(f, bvj, 1, ld, W, 1, ld, P))) return rc;
    // Gram-Schmidt in the B inner product: a LOCAL pass against the vectors W is coupled to in exact arithmetic -- the
    // block being expanded and its predecessor (block three-term recurrence), or the whole basis in the first step
    // after a thick restart (the locked Ritz vectors: the arrow) -- then one FULL classical pass against V[0:m].  The
    // local pass takes out the large components (where the cancellation is), the full pass the O(eps)-relative ones
    // left along the older vectors: full reorthogonalisation at half the basis traffic of two full passes.  Then
    // BW = B W and the Cholesky QR (twice) of the block, all in one launch.
    StepArgs a{};
    a.n = n; a.ld = ld; a.V = V; a.BV = BV; a.W = W; a.BW = BV + (int64_t)m * ld;
    a.m = m; a.lo = step == 0 ? 0 : (j - P > 0 ? j - P : 0); a.j = j; a.gs = 1;
    a.H1 = H1; a.H2 = H2; a.Aout = Ablk + (int64_t)step * P * P; a.Rout = Rblk + (int64_t)step * P * P; a.scratch = scratch;
    a.bp = bp; a.bi = bi; a.bv = bv;
    if ((rc = block_step<P>(a, work))) return rc;
  }
  return 0;
}

// scratch: 3 P x P (Gram matrix, inverse factor, R = R2 R1)
template <int P>
int start_block(int n, const int* bp, const int* bi, const double* bv, double* V, double* BV, int64_t ld, double* scratch,
                double* work) {
  StepArgs a{};
  a.n = n; a.ld = ld; a.V = V; a.BV = BV; a.W = V; a.BW = BV; a.gs = 0;
  a.Rout = scratch + 2 * P * P; a.scratch = scratch;
  a.bp = bp; a.bi = bi; a.bv = bv;
  return block_step<P>(a, work);
}

}  // namespace

extern "C" int eigd_block_lanczos_extend(eigd_factor* f, int n, int P, const int* d_b_indptr, const int* d_b_indices,
                                         const double* d_b_vals, double* d_V, double* d_BV, int64_t ld, int j0, int m0, int ncv,
                                         double* d_Ablk, double* d_Rblk, double* d_H1, double* d_H2, double* d_scratch,
                                         double* d_work) {
  if (j0 >= ncv) return 0;
  if ((ncv - j0) % P != 0 || m0 < j0 + P) { eigd_set_error("block_lanczos_extend: the cycle does not end on a block boundary"); return 7; }
  if (m0 + (ncv - j0) > BK_JMAX + BK_PMAX) { eigd_set_error("block_lanczos_extend: basis too large"); return 7; }
  switch (P) {
    case 2: return extend<2>(f, n, d_b_indptr, d_b_indices, d_b_vals, d_V, d_BV, ld, j0, m0, ncv, d_Ablk, d_Rblk, d_H1, d_H2, d_scratch, d_work);
    case 3: return extend<3>(f, n, d_b_indptr, d_b_indices, d_b_vals, d_V, d_BV, ld, j0, m0, ncv, d_Ablk, d_Rblk, d_H1, d_H2, d_scratch, d_work);
    case 4: return extend<4>(f, n, d_b_indptr, d_b_indices, d_b_vals, d_V, d_BV, ld, j0, m0, ncv, d_Ablk, d_Rblk, d_H1, d_H2, d_scratch, d_work);
    default: eigd_set_error("block_lanczos_extend: block size must be 2, 3 or 4"); return 7;
  }
}

// B-orthonormalise the P start vectors V[0:P] (rows) and set BV[0:P] = B V[0:P]; scratch: 3 * P * P doubles
extern "C" int eigd_block_lanczos_start(int n, int P, const int* d_b_indptr, const int* d_b_indices, const double* d_b_vals,
                                        double* d_V, double* d_BV, int64_t ld, double* d_scratch, double* d_work) {
  switch (P) {
    case 2: return start_block<2>(n, d_b_indptr, d_b_indices, d_b_vals, d_V, d_BV, ld, d_scratch, d_work);
    case 3: return start_block<3>(n, d_b_indptr, d_b_indices, d_b_vals, d_V, d_BV, ld, d_scratch, d_work);
    case 4: return start_block<4>(n, d_b_indptr, d_b_indices, d_b_vals, d_V, d_BV, ld, d_scratch, d_work);
    default: eigd_set_error("block_lanczos_start: block size must be 2, 3 or 4"); return 7;
  }
}
