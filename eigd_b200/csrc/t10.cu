// Unit element matrices of the quadratic tetrahedron (T10), computed once per mesh and kept in HBM: the per-design
// assembly and sensitivities of the 3-D solid and of heat conduction on tetrahedral meshes then run on the
// stored-matrix kernels of stored_fe.cu (30 x 30 and 10 x 10 element matrices), as those of the H8 elements do.
//
//   K0_e = sum_q w_q detJ B^T C B                      (isotropic elasticity, E and nu)
//   M0_e = density sum_q w_q detJ (N N^T (x) I_3)      (consistent mass)
//
// dof order node-major (u_x, u_y, u_z), as fe.element_dofs(conn, 3).  The scalar (heat conduction) element has one
// dof per node and the 10 x 10 unit matrices
//
//   K0_e = sum_q w_q detJ grad N_a . grad N_b          (conductivity 1)
//   M0_e = sum_q w_q detJ N_a N_b                      (heat capacity 1: the scalar block of the solid's M0 at density 1)
//
// Element and quadrature rule: t10_element.cuh; strain rows and the constitutive product: h8_element.cuh.
#include "common.cuh"
#include "h8_element.cuh"
#include "t10_element.cuh"
#include "../../include/eigd_b200.h"

namespace {

// One warp per element.  Lane b < 30 owns column b (node b / 3, component b % 3) of both matrices; lane l works on
// node l & 15 of the shape-function and Jacobian routine (both half-warps evaluate the same element, lanes 10-15 and
// 26-31 carry zeros), and the values of node a are read from lane a by shuffles.  K0 and M0 are stored row-major, row
// a written by lanes 0..29 at once (coalesced).
__global__ void __launch_bounds__(256)
t10_element_matrices_kernel(int nelems, const int* __restrict__ conn, const double* __restrict__ X, H8C c, double density,
                            double* __restrict__ K0, double* __restrict__ M0) {
  const int lane = threadIdx.x & 31;
  const int64_t e = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (e >= nelems) return;  // whole warps only: blockDim is a multiple of 32
  const int a = lane & 15;
  const T10Node nd = t10_gather(conn, X, e, a);
  const int bn = lane < 30 ? lane / 3 : 0, cb = lane < 30 ? lane % 3 : 0;
  double kc[30], mc[10];
#pragma unroll
  for (int i = 0; i < 30; ++i) kc[i] = 0.0;
#pragma unroll
  for (int i = 0; i < 10; ++i) mc[i] = 0.0;
#pragma unroll 1
  for (int q = 0; q < T10_NQ; ++q) {
    double N, Nx, Ny, Nz;
    const double dv = t10_point(nd, a, q, N, Nx, Ny, Nz);
    const double nb = __shfl_sync(0xffffffffu, N, bn), nxb = __shfl_sync(0xffffffffu, Nx, bn);
    const double nyb = __shfl_sync(0xffffffffu, Ny, bn), nzb = __shfl_sync(0xffffffffu, Nz, bn);
    double bb[6], s[6];
    h8_strain_rows(cb, nxb, nyb, nzb, bb);
    h8_c_mul(c, bb, s);
#pragma unroll
    for (int an = 0; an < 10; ++an) {
      const double na = __shfl_sync(0xffffffffu, N, an), nxa = __shfl_sync(0xffffffffu, Nx, an);
      const double nya = __shfl_sync(0xffffffffu, Ny, an), nza = __shfl_sync(0xffffffffu, Nz, an);
#pragma unroll
      for (int ca = 0; ca < 3; ++ca) {
        double ba[6];
        h8_strain_rows(ca, nxa, nya, nza, ba);
        double t = 0.0;
#pragma unroll
        for (int i = 0; i < 6; ++i) t = fma(ba[i], s[i], t);
        kc[3 * an + ca] = fma(dv, t, kc[3 * an + ca]);
      }
      mc[an] = fma(dv, na * nb, mc[an]);
    }
  }
  if (lane >= 30) return;
  double* k = K0 + e * 900 + lane;
  double* m = M0 + e * 900 + lane;
#pragma unroll
  for (int r = 0; r < 30; ++r) {
    k[r * 30] = kc[r];
    m[r * 30] = (r % 3 == cb) ? density * mc[r / 3] : 0.0;
  }
}

// Two elements per warp: lane l is node a = l & 15 of element 2 warp + l / 16 and owns column a (a < 10) of both
// matrices; the values of node an of the same element come from lane an of its 16-lane group.  The shuffles run on the
// full mask, so the lanes past the last element work on element nelems - 1 and skip the store.  M0 accumulates in the
// order of mc in t10_element_matrices_kernel (points 0..13, one fma each, the same width-16 Jacobian reduction), so it
// equals the scalar block of the solid's M0 at density 1 bit for bit.  Row r of an element is written by its 10 lanes
// at once (80 contiguous bytes).
__global__ void __launch_bounds__(256)
t10_thermal_element_matrices_kernel(int nelems, const int* __restrict__ conn, const double* __restrict__ X,
                                    double* __restrict__ K0, double* __restrict__ M0) {
  const int64_t eg = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
  const bool store = eg < nelems;
  const int64_t e = store ? eg : nelems - 1;
  const int a = threadIdx.x & 15;
  const T10Node nd = t10_gather(conn, X, e, a);
  double kc[10], mc[10];
#pragma unroll
  for (int i = 0; i < 10; ++i) kc[i] = mc[i] = 0.0;
#pragma unroll 1
  for (int q = 0; q < T10_NQ; ++q) {
    double N, Nx, Ny, Nz;
    const double dv = t10_point(nd, a, q, N, Nx, Ny, Nz);
#pragma unroll
    for (int an = 0; an < 10; ++an) {
      const double na = __shfl_sync(0xffffffffu, N, an, 16), nxa = __shfl_sync(0xffffffffu, Nx, an, 16);
      const double nya = __shfl_sync(0xffffffffu, Ny, an, 16), nza = __shfl_sync(0xffffffffu, Nz, an, 16);
      const double t = fma(nza, Nz, fma(nya, Ny, nxa * Nx));
      kc[an] = fma(dv, t, kc[an]);
      mc[an] = fma(dv, na * N, mc[an]);
    }
  }
  if (!store || a >= 10) return;
  double* k = K0 + e * 100 + a;
  double* m = M0 + e * 100 + a;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    k[r * 10] = kc[r];
    m[r * 10] = mc[r];
  }
}

}  // namespace

extern "C" int eigd_t10_element_matrices(int nelems, const int* d_conn, const double* d_X, double E, double nu, double density,
                                         double* d_K0, double* d_M0) {
  if (nelems <= 0) return 0;
  H8C c;
  if (!h8_isotropic(E, nu, c, "t10_element_matrices")) return 1;
  const int grid = (int)(((int64_t)nelems * 32 + 255) / 256);
  EIGD_LAUNCH(t10_element_matrices_kernel, grid, 256, 0, nelems, d_conn, d_X, c, density, d_K0, d_M0);
  EIGD_CHECK_LAUNCH();
  return 0;
}

extern "C" int eigd_t10_thermal_element_matrices(int nelems, const int* d_conn, const double* d_X, double* d_K0, double* d_M0) {
  if (nelems <= 0) return 0;
  const int grid = (int)(((int64_t)nelems * 16 + 255) / 256);
  EIGD_LAUNCH(t10_thermal_element_matrices_kernel, grid, 256, 0, nelems, d_conn, d_X, d_K0, d_M0);
  EIGD_CHECK_LAUNCH();
  return 0;
}
