// Tall-skinny fp64 kernels (all HBM-bound): X^T Y, X S, column-wise dots / axpys / scalings.
// They replace the numpy expressions `V.T @ X`, `U @ t`, `x.dot(y)`, `X -= h * W` in
// reference eigd/eigenvector_derivatives.py:26-30 (_project), :502-519 (laa), :616-620 (dl),
// :1228-1260 (sibk Gram-Schmidt), :1529-1538 (Lanczos Gram-Schmidt), :1648 (Rayleigh-Ritz).
//
// Operands are addressed as X[i*rs + c*cs]: (rs=k, cs=1) is the reference's (n, N) row-major
// layout, (rs=1, cs=n) is a Krylov basis stored one vector per row.  Tiles are staged through
// shared memory with the unit-stride index varying fastest across the warp, so global loads
// are coalesced for either layout.  Reductions over n are two-stage and deterministic.
#include "common.cuh"
#include <cstdlib>
#include "../../include/eigd_b200.h"

cudaStream_t g_eigd_stream = 0;
int64_t g_eigd_launches = 0;

extern "C" int eigd_set_stream(void* s) { g_eigd_stream = (cudaStream_t)s; return 0; }
extern "C" int64_t eigd_launch_count(void) { return g_eigd_launches; }
extern "C" int eigd_device_count(int* count) {
  int c = 0;
  cudaError_t e = cudaGetDeviceCount(&c);
  if (e != cudaSuccess) { *count = 0; eigd_set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e)); cudaGetLastError(); return 100 + (int)e; }
  *count = c;
  return 0;
}

namespace {

constexpr int TN_R = 64;        // rows per tile
constexpr int TN_KMAX = 32;     // max columns of either operand per launch
constexpr int TN_THREADS = 256;
constexpr int RED_MAX_CTAS = 296;

// stage a (rows x k) tile of a strided operand into shared memory, tile[r*(k+1) + c]
__device__ __forceinline__ void load_tile(double* tile, const double* __restrict__ X, int64_t rs, int64_t cs,
                                          int64_t row0, int rows, int k, int ldt) {
  int total = rows * k;
  if (cs == 1) {
    for (int e = threadIdx.x; e < total; e += blockDim.x) {
      int r = e / k, c = e - r * k;
      tile[r * ldt + c] = X[(row0 + r) * rs + c];
    }
  } else {
    for (int e = threadIdx.x; e < total; e += blockDim.x) {
      int c = e / rows, r = e - c * rows;
      tile[r * ldt + c] = X[(row0 + r) * rs + (int64_t)c * cs];
    }
  }
}

// partial[cta][a*k2+b] = sum over the CTA's row tiles of X[i,a]*Y[i,b]; 4x4 register tiles
__global__ void __launch_bounds__(TN_THREADS)
gemm_tn_partial(int64_t n, int k1, int k2, const double* __restrict__ X, int64_t xrs, int64_t xcs,
                const double* __restrict__ Y, int64_t yrs, int64_t ycs, double* __restrict__ partial) {
  extern __shared__ double sm[];
  const int ldx = k1 + 1, ldy = k2 + 1;
  double* Xs = sm;
  double* Ys = sm + TN_R * ldx;
  const int nta = (k1 + 3) >> 2, ntb = (k2 + 3) >> 2;
  const int npairs = nta * ntb;
  const int G = TN_THREADS / npairs;  // row groups (npairs <= 64 -> G >= 4)
  const int g = threadIdx.x / npairs, p = threadIdx.x - g * npairs;
  const int a0 = (p / ntb) * 4, b0 = (p % ntb) * 4;
  const bool active = g < G;
  double acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
  const int64_t ntiles = (n + TN_R - 1) / TN_R;
  for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    int64_t row0 = t * TN_R;
    int rows = (int)min((int64_t)TN_R, n - row0);
    load_tile(Xs, X, xrs, xcs, row0, rows, k1, ldx);
    load_tile(Ys, Y, yrs, ycs, row0, rows, k2, ldy);
    __syncthreads();
    if (active) {
      for (int r = g; r < rows; r += G) {
        double xa[4], yb[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) xa[i] = (a0 + i < k1) ? Xs[r * ldx + a0 + i] : 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j) yb[j] = (b0 + j < k2) ? Ys[r * ldy + b0 + j] : 0.0;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fma(xa[i], yb[j], acc[i][j]);
      }
    }
    __syncthreads();
  }
  // reduce over the row groups in a fixed order: group 0 owns the result
  double* red = sm;  // reuse: needs 16 * TN_THREADS doubles = 32 KB <= tile storage? sized by host
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) red[(i * 4 + j) * TN_THREADS + threadIdx.x] = active ? acc[i][j] : 0.0;
  __syncthreads();
  if (g == 0) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (a0 + i < k1 && b0 + j < k2) {
          double s = 0.0;
          for (int gg = 0; gg < G; ++gg) s += red[(i * 4 + j) * TN_THREADS + gg * npairs + p];
          partial[(int64_t)blockIdx.x * (k1 * k2) + (a0 + i) * k2 + (b0 + j)] = s;
        }
      }
  }
}

// C[a*ldc + b] = sum_cta partial[cta][a*k2+b]; one warp per output, lanes stride over the CTAs and meet
// in a shuffle tree (fixed order: deterministic)
__global__ void reduce_partials(int ncta, int k1, int k2, const double* __restrict__ partial, double* __restrict__ C, int ldc) {
  int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (e >= k1 * k2) return;
  double s = 0.0;
  for (int c = lane; c < ncta; c += 32) s += partial[(int64_t)c * (k1 * k2) + e];
  s = warp_sum(s);
  if (lane == 0) C[(e / k2) * ldc + (e % k2)] = s;
}

// ---- Krylov-basis kernels: the basis is stored one vector per row (row a at V + a*ldv), w is a
// contiguous n-vector.  These are the two halves of a classical Gram-Schmidt pass
// (eigd/eigenvector_derivatives.py:1529-1538; ARPACK dsaitr steps 3-4): h = V^T w, w -= V h.
constexpr int BD_THREADS = 256;
constexpr int BD_EPT = 4;                       // elements of w per thread
constexpr int BD_CHUNK = BD_THREADS * BD_EPT;   // per CTA
constexpr int BD_ROWS = 8;                      // basis rows in flight per thread
constexpr int BD_JMAX = 128;

// out[a] = sum_i V[a][i] * w[i], a < j.  CTA c owns elements [c*BD_CHUNK, (c+1)*BD_CHUNK): w lives in
// registers, eight basis rows are streamed at a time (32 independent 8-byte loads per thread).  Partial
// sums go to partial[cta][a]; the last CTA to finish (ticket) adds them in a fixed order, so the result
// is bitwise reproducible and no second launch is needed.
__global__ void __launch_bounds__(BD_THREADS)
basis_dots_kernel(int64_t n, int j, const double* __restrict__ V, int64_t ldv, const double* __restrict__ w,
                  double* __restrict__ partial, double* __restrict__ out, unsigned int* __restrict__ ticket) {
  __shared__ double red[BD_THREADS / 32][BD_JMAX];
  __shared__ bool last;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t i0 = (int64_t)blockIdx.x * BD_CHUNK + tid;
  double wv[BD_EPT];
#pragma unroll
  for (int q = 0; q < BD_EPT; ++q) {
    int64_t i = i0 + (int64_t)q * BD_THREADS;
    wv[q] = (i < n) ? w[i] : 0.0;
  }
  for (int a0 = 0; a0 < j; a0 += BD_ROWS) {
    double v[BD_ROWS][BD_EPT];
#pragma unroll
    for (int r = 0; r < BD_ROWS; ++r) {
      const double* row = V + (int64_t)min(a0 + r, j - 1) * ldv;
#pragma unroll
      for (int q = 0; q < BD_EPT; ++q) {
        int64_t i = i0 + (int64_t)q * BD_THREADS;
        v[r][q] = (i < n) ? __ldg(row + i) : 0.0;
      }
    }
#pragma unroll
    for (int r = 0; r < BD_ROWS; ++r) {
      double s = 0.0;
#pragma unroll
      for (int q = 0; q < BD_EPT; ++q) s = fma(v[r][q], wv[q], s);
      s = warp_sum(s);
      if (lane == 0 && a0 + r < j) red[warp][a0 + r] = s;
    }
  }
  __syncthreads();
  if (tid < j) {
    double s = 0.0;
#pragma unroll
    for (int g = 0; g < BD_THREADS / 32; ++g) s += red[g][tid];
    partial[(int64_t)blockIdx.x * BD_JMAX + tid] = s;
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!last) return;
  __threadfence();
  // 4 lanes per output row, each adds every 4th CTA's partial; rows beyond 64 in a second round
  const int ncta = gridDim.x;
  for (int a = tid >> 2; a < j; a += BD_THREADS >> 2) {
    const int q = tid & 3;
    double s = 0.0;
    for (int c = q; c < ncta; c += 4) s += __ldcg(partial + (int64_t)c * BD_JMAX + a);
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    if (q == 0) out[a] = s;
  }
  if (tid == 0) *ticket = 0u;
}

// w[i] += sign * sum_a h[a] * V[a][i]; optionally also writes the result to a second vector (w2)
__global__ void __launch_bounds__(BD_THREADS)
basis_axpy_kernel(int64_t n, int j, const double* __restrict__ V, int64_t ldv, const double* __restrict__ h, double sign,
                  double* __restrict__ w) {
  __shared__ double hs[BD_JMAX];
  const int tid = threadIdx.x;
  if (tid < j) hs[tid] = sign * h[tid];
  __syncthreads();
  const int64_t i0 = (int64_t)blockIdx.x * BD_CHUNK + tid;
  double acc[BD_EPT];
#pragma unroll
  for (int q = 0; q < BD_EPT; ++q) {
    int64_t i = i0 + (int64_t)q * BD_THREADS;
    acc[q] = (i < n) ? w[i] : 0.0;
  }
  for (int a0 = 0; a0 < j; a0 += BD_ROWS) {
    double v[BD_ROWS][BD_EPT];
#pragma unroll
    for (int r = 0; r < BD_ROWS; ++r) {
      const double* row = V + (int64_t)min(a0 + r, j - 1) * ldv;
#pragma unroll
      for (int q = 0; q < BD_EPT; ++q) {
        int64_t i = i0 + (int64_t)q * BD_THREADS;
        v[r][q] = (i < n) ? __ldg(row + i) : 0.0;
      }
    }
#pragma unroll
    for (int r = 0; r < BD_ROWS; ++r) {
      const double hr = (a0 + r < j) ? hs[a0 + r] : 0.0;
#pragma unroll
      for (int q = 0; q < BD_EPT; ++q) acc[q] = fma(hr, v[r][q], acc[q]);
    }
  }
#pragma unroll
  for (int q = 0; q < BD_EPT; ++q) {
    int64_t i = i0 + (int64_t)q * BD_THREADS;
    if (i < n) w[i] = acc[q];
  }
}

// Same product for the reference's row-major (n, k) operands (unit column stride): no shared-memory staging and
// no block barrier in the row loop -- every CTA owns one contiguous range of rows, a thread (row group g, 4x4
// output tile p) reads its 4 + 4 operand entries of UNR rows straight from global memory (the rows of a warp's
// threads are adjacent, the re-reads by the other tiles of the same row hit L1) before it does the FMAs.
// The staged kernel above spent its time in load -> barrier -> compute -> barrier per 64 rows (63 us for
// 2 x 20 MB at n = 251k); this one is bound by the loads.
__global__ void __launch_bounds__(TN_THREADS)
gemm_tn_rowmajor_partial(int64_t n, int k1, int k2, const double* __restrict__ X, int64_t xrs,
                         const double* __restrict__ Y, int64_t yrs, double* __restrict__ partial) {
  extern __shared__ double sm[];
  constexpr int UNR = 4;
  const int nta = (k1 + 3) >> 2, ntb = (k2 + 3) >> 2;
  const int npairs = nta * ntb;
  const int G = TN_THREADS / npairs;
  const int g = threadIdx.x / npairs, p = threadIdx.x - g * npairs;
  const int a0 = (p / ntb) * 4, b0 = (p % ntb) * 4;
  const bool active = g < G;
  double acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
  const int64_t per = (n + gridDim.x - 1) / gridDim.x;
  const int64_t r0 = (int64_t)blockIdx.x * per, r1 = min(n, r0 + per);
  if (active) {
    for (int64_t rb = r0 + g; rb < r1; rb += (int64_t)G * UNR) {
      double xa[UNR][4], yb[UNR][4];
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        const int64_t r = rb + (int64_t)u * G;
        const bool ok = r < r1;
        const double* xp = X + r * xrs + a0;
        const double* yp = Y + r * yrs + b0;
#pragma unroll
        for (int i = 0; i < 4; ++i) xa[u][i] = (ok && a0 + i < k1) ? __ldg(xp + i) : 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j) yb[u][j] = (ok && b0 + j < k2) ? __ldg(yp + j) : 0.0;
      }
#pragma unroll
      for (int u = 0; u < UNR; ++u)
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fma(xa[u][i], yb[u][j], acc[i][j]);
    }
  }
  // reduce over the row groups in a fixed order: group 0 owns the result
  double* red = sm;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) red[(i * 4 + j) * TN_THREADS + threadIdx.x] = active ? acc[i][j] : 0.0;
  __syncthreads();
  if (g == 0) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (a0 + i < k1 && b0 + j < k2) {
          double s = 0.0;
          for (int gg = 0; gg < G; ++gg) s += red[(i * 4 + j) * TN_THREADS + gg * npairs + p];
          partial[(int64_t)blockIdx.x * (k1 * k2) + (a0 + i) * k2 + (b0 + j)] = s;
        }
      }
  }
}

constexpr int NN_R = 32;
constexpr int NN_K1MAX = 64;
constexpr int NN_K2MAX = 32;

// Y[i,b] = beta*Y[i,b] + alpha*sum_a X[i,a]*S[a,b]
__global__ void __launch_bounds__(256)
gemm_nn_kernel(int64_t n, int k1, int k2, double alpha, const double* __restrict__ X, int64_t xrs, int64_t xcs,
               const double* __restrict__ S, int lds, double beta, double* __restrict__ Y, int64_t yrs, int64_t ycs) {
  __shared__ double Ss[NN_K1MAX * NN_K2MAX];
  __shared__ double Xs[NN_R * (NN_K1MAX + 1)];
  const int ldx = k1 + 1;
  for (int e = threadIdx.x; e < k1 * k2; e += blockDim.x) Ss[e] = S[(e / k2) * lds + (e % k2)];
  const int64_t ntiles = (n + NN_R - 1) / NN_R;
  for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    int64_t row0 = t * NN_R;
    int rows = (int)min((int64_t)NN_R, n - row0);
    __syncthreads();
    load_tile(Xs, X, xrs, xcs, row0, rows, k1, ldx);
    __syncthreads();
    int total = rows * k2;
    for (int e = threadIdx.x; e < total; e += blockDim.x) {
      int r, b;
      if (ycs == 1) { r = e / k2; b = e - r * k2; } else { b = e / rows; r = e - b * rows; }
      double s = 0.0;
      for (int a = 0; a < k1; ++a) s = fma(Xs[r * ldx + a], Ss[a * k2 + b], s);
      int64_t yi = (row0 + r) * yrs + (int64_t)b * ycs;
      double y0 = (beta == 0.0) ? 0.0 : beta * Y[yi];
      Y[yi] = fma(alpha, s, y0);
    }
  }
}

// Same update for row-major X (n, k1) and Y (n, k2): one output entry per thread (coalesced Y), the k1 entries of
// its X row come through L1 (the k2 threads of a row share them), S sits in shared memory; no barrier per tile.
__global__ void __launch_bounds__(256)
gemm_nn_rowmajor_kernel(int64_t n, int k1, int k2, double alpha, const double* __restrict__ X, int64_t xrs,
                        const double* __restrict__ S, int lds, double beta, double* __restrict__ Y, int64_t yrs) {
  __shared__ double Ss[NN_K1MAX * NN_K2MAX];
  for (int e = threadIdx.x; e < k1 * k2; e += blockDim.x) Ss[e] = S[(e / k2) * lds + (e % k2)];
  __syncthreads();
  const int64_t total = n * k2;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / k2;
    const int b = (int)(e - i * k2);
    const double* xp = X + i * xrs;
    const int64_t yi = i * yrs + b;
    const double y0 = (beta == 0.0) ? 0.0 : beta * Y[yi];
    double s = 0.0;
    for (int a = 0; a < k1; ++a) s = fma(__ldg(xp + a), Ss[a * k2 + b], s);
    Y[yi] = fma(alpha, s, y0);
  }
}

// partial[cta][c] = sum_i X[i,c]*Y[i,c] over the CTA's rows
__global__ void __launch_bounds__(256)
col_dot_partial(int64_t n, int k, const double* __restrict__ X, int64_t xrs, int64_t xcs,
                const double* __restrict__ Y, int64_t yrs, int64_t ycs, double* __restrict__ partial) {
  __shared__ double red[256];
  const int RG = 256 / k;  // row lanes per column
  const int rr = threadIdx.x / k, c = threadIdx.x - rr * k;
  // when both operands are unit-stride along rows (k == 1 style) the mapping below is still coalesced
  double acc = 0.0;
  if (rr < RG) {
    for (int64_t i = (int64_t)blockIdx.x * RG + rr; i < n; i += (int64_t)gridDim.x * RG)
      acc = fma(X[i * xrs + (int64_t)c * xcs], Y[i * yrs + (int64_t)c * ycs], acc);
  }
  red[threadIdx.x] = (rr < RG) ? acc : 0.0;
  __syncthreads();
  if (rr == 0) {
    double s = 0.0;
    for (int g = 0; g < RG; ++g) s += red[g * k + c];
    partial[(int64_t)blockIdx.x * k + c] = s;
  }
}

__global__ void col_axpy_kernel(int64_t n, int k, double sign, const double* __restrict__ s, const double* __restrict__ X,
                                int64_t xrs, int64_t xcs, double* __restrict__ Y, int64_t yrs, int64_t ycs) {
  int64_t total = n * k;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t i; int c;
    if (ycs == 1) { i = e / k; c = (int)(e - i * k); } else { c = (int)(e / n); i = e - (int64_t)c * n; }
    int64_t yi = i * yrs + (int64_t)c * ycs;
    Y[yi] = fma(sign * s[c], X[i * xrs + (int64_t)c * xcs], Y[yi]);
  }
}

__global__ void col_scale_kernel(int64_t n, int k, int mode, const double* __restrict__ s, double* __restrict__ X,
                                 int64_t xrs, int64_t xcs) {
  int64_t total = n * k;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t i; int c;
    if (xcs == 1) { i = e / k; c = (int)(e - i * k); } else { c = (int)(e / n); i = e - (int64_t)c * n; }
    double f = s[c];
    if (mode == 1) f = 1.0 / f;
    else if (mode == 2) f = 1.0 / sqrt(f);
    else if (mode == 3) f = (f > 0.0) ? 1.0 / sqrt(f) : 0.0;   // safe normalisation (converged / empty columns)
    else if (mode == 4) f = (f != 0.0) ? 1.0 / f : 0.0;
    X[i * xrs + (int64_t)c * xcs] *= f;
  }
}

// tiled transpose-capable copy: coalesced on both sides
__global__ void copy2d_kernel(int64_t n, int k, const double* __restrict__ X, int64_t xrs, int64_t xcs,
                              double* __restrict__ Y, int64_t yrs, int64_t ycs) {
  __shared__ double tile[32][33];
  int64_t i0 = (int64_t)blockIdx.x * 32;
  int c0 = blockIdx.y * 32;
  // read with the source's unit-stride index fastest
  for (int q = threadIdx.y; q < 32; q += blockDim.y) {
    int64_t i; int c;
    if (xcs == 1) { i = i0 + q; c = c0 + threadIdx.x; } else { i = i0 + threadIdx.x; c = c0 + q; }
    if (i < n && c < k) tile[(int)(i - i0)][c - c0] = X[i * xrs + (int64_t)c * xcs];
  }
  __syncthreads();
  for (int q = threadIdx.y; q < 32; q += blockDim.y) {
    int64_t i; int c;
    if (ycs == 1) { i = i0 + q; c = c0 + threadIdx.x; } else { i = i0 + threadIdx.x; c = c0 + q; }
    if (i < n && c < k) Y[i * yrs + (int64_t)c * ycs] = tile[(int)(i - i0)][c - c0];
  }
}

__global__ void axpby_kernel(int64_t len, double a, const double* __restrict__ x, double b, const double* __restrict__ y,
                             double* __restrict__ out) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < len; e += (int64_t)gridDim.x * blockDim.x)
    out[e] = a * x[e] + (b == 0.0 ? 0.0 : b * y[e]);
}

__device__ unsigned int g_basis_ticket = 0;

inline int tn_grid(int64_t n) {
  int64_t t = (n + TN_R - 1) / TN_R;
  return (int)(t < RED_MAX_CTAS ? (t < 1 ? 1 : t) : RED_MAX_CTAS);
}

}  // namespace

int eigd_basis_dots(int64_t n, int j, const double* V, int64_t ldv, const double* w, double* out, double* work) {
  unsigned int* ticket = nullptr;
  EIGD_CUDA(cudaGetSymbolAddress((void**)&ticket, g_basis_ticket));
  int grid = (int)((n + BD_CHUNK - 1) / BD_CHUNK);
  EIGD_LAUNCH(basis_dots_kernel, grid, BD_THREADS, 0, n, j, V, ldv, w, work, out, ticket);
  EIGD_CHECK_LAUNCH();
  return 0;
}

// w += alpha * sum_a S[a*lds] V[a]
int eigd_basis_axpy(int64_t n, int j, const double* V, int64_t ldv, const double* S, int lds, double alpha, double* w) {
  (void)lds;
  int grid = (int)((n + BD_CHUNK - 1) / BD_CHUNK);
  EIGD_LAUNCH(basis_axpy_kernel, grid, BD_THREADS, 0, n, j, V, ldv, S, alpha, w);
  EIGD_CHECK_LAUNCH();
  return 0;
}

extern "C" int64_t eigd_gemm_tn_workspace(int k1, int k2) {
  (void)k1; (void)k2;
  return (int64_t)RED_MAX_CTAS * TN_KMAX * TN_KMAX;
}

extern "C" int eigd_gemm_tn(int64_t n, int k1, int k2, const double* X, int64_t xrs, int64_t xcs, const double* Y,
                            int64_t yrs, int64_t ycs, double* C, int ldc, double* work) {
  if (n <= 0 || k1 <= 0 || k2 <= 0) return 0;
  if (k2 == 1 && xrs == 1 && yrs == 1 && (ldc == 1 || k1 == 1) && k1 <= BD_JMAX) {     // Krylov basis (one vector per row) times a vector
    int64_t ncta = (n + BD_CHUNK - 1) / BD_CHUNK;
    if (ncta * BD_JMAX <= eigd_gemm_tn_workspace(k1, k2)) return eigd_basis_dots(n, k1, X, xcs, Y, C, work);
  }
  for (int a0 = 0; a0 < k1; a0 += TN_KMAX) {
    int ka = min(TN_KMAX, k1 - a0);
    for (int b0 = 0; b0 < k2; b0 += TN_KMAX) {
      int kb = min(TN_KMAX, k2 - b0);
      int grid = tn_grid(n);
      size_t tile_bytes = (size_t)TN_R * (ka + 1 + kb + 1) * sizeof(double);
      size_t red_bytes = (size_t)16 * TN_THREADS * sizeof(double);
      size_t smem = tile_bytes > red_bytes ? tile_bytes : red_bytes;
      if (xcs == 1 && ycs == 1) {
        EIGD_LAUNCH(gemm_tn_rowmajor_partial, grid, TN_THREADS, red_bytes, n, ka, kb, X + a0, xrs, Y + b0, yrs, work);
      } else {
        EIGD_LAUNCH(gemm_tn_partial, grid, TN_THREADS, smem, n, ka, kb, X + (int64_t)a0 * xcs, xrs, xcs,
                    Y + (int64_t)b0 * ycs, yrs, ycs, work);
      }
      EIGD_CHECK_LAUNCH();
      EIGD_LAUNCH(reduce_partials, (ka * kb + 7) / 8, 256, 0, grid, ka, kb, work, C + (int64_t)a0 * ldc + b0, ldc);
      EIGD_CHECK_LAUNCH();
    }
  }
  return 0;
}

extern "C" int eigd_gemm_nn(int64_t n, int k1, int k2, double alpha, const double* X, int64_t xrs, int64_t xcs,
                            const double* S, int lds, double beta, double* Y, int64_t yrs, int64_t ycs) {
  if (n <= 0 || k2 <= 0) return 0;
  int64_t tiles = (n + NN_R - 1) / NN_R;
  int grid = (int)(tiles < 148 * 8 ? tiles : 148 * 8);
  if (k1 <= 0) {  // Y = beta*Y
    return 0;
  }
  if (k2 == 1 && xrs == 1 && yrs == 1 && beta == 1.0 && k1 <= BD_JMAX && (lds == 1 || k1 == 1)) return eigd_basis_axpy(n, k1, X, xcs, S, lds, alpha, Y);
  for (int b0 = 0; b0 < k2; b0 += NN_K2MAX) {
    int kb = min(NN_K2MAX, k2 - b0);
    for (int a0 = 0; a0 < k1; a0 += NN_K1MAX) {
      int ka = min(NN_K1MAX, k1 - a0);
      if (xcs == 1 && ycs == 1) {
        int64_t ge = (n * kb + 255) / 256;
        int g2 = (int)(ge < 148 * 16 ? ge : 148 * 16);
        EIGD_LAUNCH(gemm_nn_rowmajor_kernel, g2, 256, 0, n, ka, kb, alpha, X + a0, xrs, S + (int64_t)a0 * lds + b0, lds,
                    (a0 == 0 ? beta : 1.0), Y + b0, yrs);
      } else {
        EIGD_LAUNCH(gemm_nn_kernel, grid, 256, 0, n, ka, kb, alpha, X + (int64_t)a0 * xcs, xrs, xcs,
                    S + (int64_t)a0 * lds + b0, lds, (a0 == 0 ? beta : 1.0), Y + (int64_t)b0 * ycs, yrs, ycs);
      }
      EIGD_CHECK_LAUNCH();
    }
  }
  return 0;
}

extern "C" int eigd_col_dot(int64_t n, int k, const double* X, int64_t xrs, int64_t xcs, const double* Y, int64_t yrs,
                            int64_t ycs, double* out, double* work) {
  if (k <= 0) return 0;
  for (int c0 = 0; c0 < k; c0 += 64) {
    int kc = min(64, k - c0);
    int RG = 256 / kc;
    int64_t want = (n + (int64_t)RG * 8 - 1) / ((int64_t)RG * 8);
    int grid = (int)(want < 1 ? 1 : (want > RED_MAX_CTAS ? RED_MAX_CTAS : want));
    EIGD_LAUNCH(col_dot_partial, grid, 256, 0, n, kc, X + (int64_t)c0 * xcs, xrs, xcs, Y + (int64_t)c0 * ycs, yrs, ycs, work);
    EIGD_CHECK_LAUNCH();
    EIGD_LAUNCH(reduce_partials, (kc + 7) / 8, 256, 0, grid, 1, kc, work, out + c0, kc);
    EIGD_CHECK_LAUNCH();
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------------------
// Modified Gram-Schmidt sweep of a block of k columns (the k adjoint systems in lock step) against j stored
// blocks, in ONE cooperative launch:   for t = 0 .. j-1:  h_t[c] = sum_i w[i,c] W_t[i,c];  w[:,c] -= h_t[c] W_t[:,c]
// (reference eigd/eigenvector_derivatives.py:1254-1257 and :1012-1014: one dot / axpy pair per stored vector).
// Every CTA owns a fixed range of rows, so only the k dot products cross CTAs: one software grid barrier per
// stored block; the axpy with W_t and the partial dots with W_{t+1} share one pass over the CTA's rows of w
// (which stay in L2), W_{t+1} is the only stream from HBM.  Partial sums are combined in a fixed order
// (bitwise reproducible); the two halves of `partial` alternate so that a fast CTA never overwrites sums a slow
// one is still reading (to write the sums of step t + 2 it must have passed barrier t + 1).
constexpr int MGS_MAX = 64;     // stored blocks per launch (kernel-parameter space)
constexpr int MGS_KMAX = 64;

struct MgsArgs {
  const double* W[MGS_MAX];
  double* H[MGS_MAX];
};

__global__ void __launch_bounds__(256)
mgs_sweep_kernel(int64_t n, int k, int j, MgsArgs a, double* __restrict__ w, double* __restrict__ partial,
                 unsigned long long* ctr, unsigned long long base) {
  __shared__ double red[256];
  __shared__ double hs[MGS_KMAX];
  const int G = gridDim.x;
  const int RG = 256 / k;                                   // row lanes per column
  const int rr = threadIdx.x / k, c = threadIdx.x - rr * k;
  const bool on = rr < RG;
  const int64_t per = (n + G - 1) / G;
  const int64_t r0 = (int64_t)blockIdx.x * per;
  const int64_t r1 = r0 + per < n ? r0 + per : n;
  double acc = 0.0;
  // row loops run four rows per trip (loads of all four first): with one row per trip every trip waited for its
  // own memory round trip; the summation order is that of the plain loop
  const int64_t st = (int64_t)RG * k;                       // element stride between a thread's consecutive rows
  if (on) {
    const double* W0 = a.W[0];
    int64_t e = (r0 + rr) * k + c;
    const int64_t eend = r1 * k;
    for (; e + 3 * st < eend; e += 4 * st) {
      const double w0 = w[e], w1 = w[e + st], w2 = w[e + 2 * st], w3 = w[e + 3 * st];
      const double x0 = __ldg(W0 + e), x1 = __ldg(W0 + e + st), x2 = __ldg(W0 + e + 2 * st), x3 = __ldg(W0 + e + 3 * st);
      acc = fma(w0, x0, acc); acc = fma(w1, x1, acc); acc = fma(w2, x2, acc); acc = fma(w3, x3, acc);
    }
    for (; e < eend; e += st) acc = fma(w[e], __ldg(W0 + e), acc);
  }
  for (int t = 0; t < j; ++t) {
    red[threadIdx.x] = on ? acc : 0.0;
    __syncthreads();
    double* mine = partial + ((int64_t)(t & 1) * G + blockIdx.x) * k;
    if (threadIdx.x < k) {
      double s = 0.0;
      for (int g = 0; g < RG; ++g) s += red[g * k + threadIdx.x];
      mine[threadIdx.x] = s;
    }
    coop_grid_barrier(ctr, base + (unsigned long long)(t + 1) * (unsigned long long)G);
    const double* all = partial + (int64_t)(t & 1) * G * k;
    double s = 0.0;
    if (on)
      for (int g = rr; g < G; g += RG) s += __ldcg(all + (int64_t)g * k + c);
    red[threadIdx.x] = on ? s : 0.0;
    __syncthreads();
    if (threadIdx.x < k) {
      double h = 0.0;
      for (int g = 0; g < RG; ++g) h += red[g * k + threadIdx.x];
      hs[threadIdx.x] = h;
      if (blockIdx.x == 0) a.H[t][threadIdx.x] = h;
    }
    __syncthreads();
    acc = 0.0;
    if (on) {
      const double h = hs[c];
      const double* Wt = a.W[t];
      int64_t e = (r0 + rr) * k + c;
      const int64_t eend = r1 * k;
      if (t + 1 < j) {
        const double* Wn = a.W[t + 1];
        for (; e + 3 * st < eend; e += 4 * st) {
          const double t0 = __ldg(Wt + e), t1 = __ldg(Wt + e + st), t2 = __ldg(Wt + e + 2 * st), t3 = __ldg(Wt + e + 3 * st);
          const double w0 = w[e], w1 = w[e + st], w2 = w[e + 2 * st], w3 = w[e + 3 * st];
          const double n0 = __ldg(Wn + e), n1 = __ldg(Wn + e + st), n2 = __ldg(Wn + e + 2 * st), n3 = __ldg(Wn + e + 3 * st);
          const double v0 = fma(-h, t0, w0), v1 = fma(-h, t1, w1), v2 = fma(-h, t2, w2), v3 = fma(-h, t3, w3);
          w[e] = v0; w[e + st] = v1; w[e + 2 * st] = v2; w[e + 3 * st] = v3;
          acc = fma(v0, n0, acc); acc = fma(v1, n1, acc); acc = fma(v2, n2, acc); acc = fma(v3, n3, acc);
        }
        for (; e < eend; e += st) {
          const double v = fma(-h, __ldg(Wt + e), w[e]);
          w[e] = v;
          acc = fma(v, __ldg(Wn + e), acc);
        }
      } else {
        for (; e + 3 * st < eend; e += 4 * st) {
          const double t0 = __ldg(Wt + e), t1 = __ldg(Wt + e + st), t2 = __ldg(Wt + e + 2 * st), t3 = __ldg(Wt + e + 3 * st);
          const double w0 = w[e], w1 = w[e + st], w2 = w[e + 2 * st], w3 = w[e + 3 * st];
          w[e] = fma(-h, t0, w0); w[e + st] = fma(-h, t1, w1); w[e + 2 * st] = fma(-h, t2, w2); w[e + 3 * st] = fma(-h, t3, w3);
        }
        for (; e < eend; e += st) w[e] = fma(-h, __ldg(Wt + e), w[e]);
      }
    }
  }
}

static unsigned long long* g_coop_ctr = nullptr;
static unsigned long long g_coop_base = 0;
static int g_coop_dev = -1;

int coop_counter(unsigned long long** ctr, unsigned long long** base) {
  int dev = 0;
  EIGD_CUDA(cudaGetDevice(&dev));
  if (dev != g_coop_dev) {
    EIGD_CUDA(cudaMalloc(&g_coop_ctr, sizeof(unsigned long long)));
    EIGD_CUDA(cudaMemsetAsync(g_coop_ctr, 0, sizeof(unsigned long long), g_eigd_stream));
    g_coop_base = 0;
    g_coop_dev = dev;
  }
  *ctr = g_coop_ctr;
  *base = &g_coop_base;
  return 0;
}

extern "C" int eigd_mgs_sweep(int64_t n, int k, int j, const double* const* W, double* const* H, double* d_w,
                              double* d_work) {
  if (n <= 0 || j <= 0) return 0;
  if (k < 1 || k > MGS_KMAX) { eigd_set_error("mgs_sweep: k = %d outside 1..%d", k, MGS_KMAX); return 7; }
  static int max_grid = 0, per_sm = -1;
  if (per_sm < 0) { const char* e = getenv("EIGD_MGS_CTAS_PER_SM"); per_sm = e ? atoi(e) : 4; if (per_sm < 1) per_sm = 1; }   // developer tuning; measured at C2, 8 blocks: 146 / 130 / 125 us with 2 / 3 / 4
  int rc;
  // the two halves of the partial-sum buffer (2 x grid x k doubles) live in the reduction workspace
  const int cap = (int)(eigd_gemm_tn_workspace(TN_KMAX, TN_KMAX) / (2 * MGS_KMAX));
  unsigned long long *ctr = nullptr, *base = nullptr;
  if ((rc = coop_counter(&ctr, &base)) || (rc = coop_max_grid(mgs_sweep_kernel, per_sm, cap, &max_grid))) return rc;
  const int RG = 256 / k;
  int64_t want = (n + (int64_t)RG * 4 - 1) / ((int64_t)RG * 4);
  int grid = (int)(want < 1 ? 1 : (want > max_grid ? max_grid : want));
  for (int j0 = 0; j0 < j; j0 += MGS_MAX) {
    const int jj = j - j0 < MGS_MAX ? j - j0 : MGS_MAX;
    MgsArgs a;
    for (int t = 0; t < jj; ++t) { a.W[t] = W[j0 + t]; a.H[t] = H[j0 + t]; }
    for (int t = jj; t < MGS_MAX; ++t) { a.W[t] = nullptr; a.H[t] = nullptr; }
    int64_t n_ = n; int k_ = k, jj_ = jj;
    unsigned long long base0 = *base;
    void* params[] = {(void*)&n_, (void*)&k_, (void*)&jj_, (void*)&a, (void*)&d_w, (void*)&d_work, (void*)&ctr, (void*)&base0};
    EIGD_CUDA(cudaLaunchCooperativeKernel((void*)mgs_sweep_kernel, dim3(grid), dim3(256), params, 0, g_eigd_stream));
    ++g_eigd_launches;
    *base += (unsigned long long)jj * (unsigned long long)grid;
  }
  return 0;
}

static inline int ew_grid(int64_t total) {
  int64_t g = (total + 255) / 256;
  return (int)(g < 1 ? 1 : (g > 148 * 16 ? 148 * 16 : g));
}

extern "C" int eigd_col_axpy(int64_t n, int k, double sign, const double* s, const double* X, int64_t xrs, int64_t xcs,
                             double* Y, int64_t yrs, int64_t ycs) {
  if (n <= 0 || k <= 0) return 0;
  EIGD_LAUNCH(col_axpy_kernel, ew_grid(n * k), 256, 0, n, k, sign, s, X, xrs, xcs, Y, yrs, ycs);
  EIGD_CHECK_LAUNCH();
  return 0;
}

extern "C" int eigd_col_scale(int64_t n, int k, int mode, const double* s, double* X, int64_t xrs, int64_t xcs) {
  if (n <= 0 || k <= 0) return 0;
  EIGD_LAUNCH(col_scale_kernel, ew_grid(n * k), 256, 0, n, k, mode, s, X, xrs, xcs);
  EIGD_CHECK_LAUNCH();
  return 0;
}

extern "C" int eigd_copy2d(int64_t n, int k, const double* X, int64_t xrs, int64_t xcs, double* Y, int64_t yrs, int64_t ycs) {
  if (n <= 0 || k <= 0) return 0;
  dim3 grid((unsigned)((n + 31) / 32), (unsigned)((k + 31) / 32));
  dim3 block(32, 8);
  EIGD_LAUNCH(copy2d_kernel, grid, block, 0, n, k, X, xrs, xcs, Y, yrs, ycs);
  EIGD_CHECK_LAUNCH();
  return 0;
}

extern "C" int eigd_axpby(int64_t len, double a, const double* x, double b, const double* y, double* out) {
  if (len <= 0) return 0;
  EIGD_LAUNCH(axpby_kernel, ew_grid(len), 256, 0, len, a, x, b, y, out);
  EIGD_CHECK_LAUNCH();
  return 0;
}
