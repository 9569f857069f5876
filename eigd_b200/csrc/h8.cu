// Unit element matrices of the trilinear hexahedron (H8), computed once per mesh and kept in HBM: the per-design
// assembly and sensitivities of the 3-D solid then run on the stored-matrix kernels of stored_fe.cu, which read each
// 24 x 24 matrix once instead of evaluating 8 Jacobians for each of its 576 entries.
//
//   K0_e = sum_q detJ B^T C B                      (isotropic elasticity, E and nu)
//   M0_e = density sum_q detJ (N N^T (x) I_3)      (consistent mass)
//
// dof order node-major (u_x, u_y, u_z), as fe.element_dofs(conn, 3).  The scalar (heat conduction) element has one
// dof per node and the 8 x 8 unit matrices
//
//   K0_e = sum_q detJ grad N_a . grad N_b          (conductivity 1)
//   M0_e = sum_q detJ N_a N_b                      (heat capacity 1: the scalar block of the solid's M0 at density 1)
//
// Element: h8_element.cuh.
#include "common.cuh"
#include "h8_element.cuh"
#include "../../include/eigd_b200.h"

namespace {

// One warp per element.  Lane b < 24 owns column b (node b / 3, component b % 3) of both matrices; lane l works on
// node l & 7 of the shape-function and Jacobian routine, and the values of node a are read from lane a by shuffles.
// K0 and M0 are stored row-major, row a written by lanes 0..23 at once (coalesced).
__global__ void __launch_bounds__(256)
h8_element_matrices_kernel(int nelems, const int* __restrict__ conn, const double* __restrict__ X, H8C c, double density,
                           double* __restrict__ K0, double* __restrict__ M0) {
  const int lane = threadIdx.x & 31;
  const int64_t e = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (e >= nelems) return;  // whole warps only: blockDim is a multiple of 32
  const int a = lane & 7;
  const H8Node nd = h8_gather(conn, X, e, a);
  const int bn = lane < 24 ? lane / 3 : 0, cb = lane < 24 ? lane % 3 : 0;
  double kc[24], mc[8];
#pragma unroll
  for (int i = 0; i < 24; ++i) kc[i] = 0.0;
#pragma unroll
  for (int i = 0; i < 8; ++i) mc[i] = 0.0;
#pragma unroll 1
  for (int q = 0; q < 8; ++q) {
    double N, Nx, Ny, Nz;
    const double det = h8_point(nd, a, q, N, Nx, Ny, Nz);
    const double nb = __shfl_sync(0xffffffffu, N, bn), nxb = __shfl_sync(0xffffffffu, Nx, bn);
    const double nyb = __shfl_sync(0xffffffffu, Ny, bn), nzb = __shfl_sync(0xffffffffu, Nz, bn);
    double bb[6], s[6];
    h8_strain_rows(cb, nxb, nyb, nzb, bb);
    h8_c_mul(c, bb, s);
#pragma unroll
    for (int an = 0; an < 8; ++an) {
      const double na = __shfl_sync(0xffffffffu, N, an), nxa = __shfl_sync(0xffffffffu, Nx, an);
      const double nya = __shfl_sync(0xffffffffu, Ny, an), nza = __shfl_sync(0xffffffffu, Nz, an);
#pragma unroll
      for (int ca = 0; ca < 3; ++ca) {
        double ba[6];
        h8_strain_rows(ca, nxa, nya, nza, ba);
        double t = 0.0;
#pragma unroll
        for (int i = 0; i < 6; ++i) t = fma(ba[i], s[i], t);
        kc[3 * an + ca] = fma(det, t, kc[3 * an + ca]);
      }
      mc[an] = fma(det, na * nb, mc[an]);
    }
  }
  if (lane >= 24) return;
  double* k = K0 + e * 576 + lane;
  double* m = M0 + e * 576 + lane;
#pragma unroll
  for (int r = 0; r < 24; ++r) {
    k[r * 24] = kc[r];
    m[r * 24] = (r % 3 == cb) ? density * mc[r / 3] : 0.0;
  }
}

// Four elements per warp: lane l is node a = l & 7 of element 4 warp + l / 8 and owns column a of both matrices; the
// values of node an of the same element come from lane an of its 8-lane group.  The shuffles run on the full mask, so
// the lanes past the last element work on element nelems - 1 and skip the store.  M0 accumulates in the order of mc in
// h8_element_matrices_kernel (Gauss points 0..7, one fma each), so it equals the scalar block of the solid's M0 at
// density 1 bit for bit.  Row r of an element is written by its 8 lanes at once (64 contiguous bytes).
__global__ void __launch_bounds__(256)
h8_thermal_element_matrices_kernel(int nelems, const int* __restrict__ conn, const double* __restrict__ X,
                                   double* __restrict__ K0, double* __restrict__ M0) {
  const int64_t eg = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const bool store = eg < nelems;
  const int64_t e = store ? eg : nelems - 1;
  const int a = threadIdx.x & 7;
  const H8Node nd = h8_gather(conn, X, e, a);
  double kc[8], mc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) kc[i] = mc[i] = 0.0;
#pragma unroll 1
  for (int q = 0; q < 8; ++q) {
    double N, Nx, Ny, Nz;
    const double det = h8_point(nd, a, q, N, Nx, Ny, Nz);
#pragma unroll
    for (int an = 0; an < 8; ++an) {
      const double na = __shfl_sync(0xffffffffu, N, an, 8), nxa = __shfl_sync(0xffffffffu, Nx, an, 8);
      const double nya = __shfl_sync(0xffffffffu, Ny, an, 8), nza = __shfl_sync(0xffffffffu, Nz, an, 8);
      const double t = fma(nza, Nz, fma(nya, Ny, nxa * Nx));
      kc[an] = fma(det, t, kc[an]);
      mc[an] = fma(det, na * N, mc[an]);
    }
  }
  if (!store) return;
  double* k = K0 + e * 64 + a;
  double* m = M0 + e * 64 + a;
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    k[r * 8] = kc[r];
    m[r * 8] = mc[r];
  }
}

}  // namespace

extern "C" int eigd_h8_element_matrices(int nelems, const int* d_conn, const double* d_X, double E, double nu, double density,
                                        double* d_K0, double* d_M0) {
  if (nelems <= 0) return 0;
  H8C c;
  if (!h8_isotropic(E, nu, c, "h8_element_matrices")) return 1;
  const int grid = (int)(((int64_t)nelems * 32 + 255) / 256);
  EIGD_LAUNCH(h8_element_matrices_kernel, grid, 256, 0, nelems, d_conn, d_X, c, density, d_K0, d_M0);
  EIGD_CHECK_LAUNCH();
  return 0;
}

extern "C" int eigd_h8_thermal_element_matrices(int nelems, const int* d_conn, const double* d_X, double* d_K0, double* d_M0) {
  if (nelems <= 0) return 0;
  const int grid = (int)(((int64_t)nelems * 8 + 255) / 256);
  EIGD_LAUNCH(h8_thermal_element_matrices_kernel, grid, 256, 0, nelems, d_conn, d_X, d_K0, d_M0);
  EIGD_CHECK_LAUNCH();
  return 0;
}
