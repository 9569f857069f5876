// Linearised buckling of the 3-D solid on trilinear hexahedra (H8): the element stresses of the fundamental path, the
// unit stress stiffness G0_e(u) and the displacement derivative of sum_k w_k^T G(u, x) v_k.  The 3-D counterparts of
// the Q4 kernels of buckling.cu; everything else of the buckling pipeline (assembly of K_r and G_r, dG/dx, dK/dx) runs
// on the stored-matrix kernels of stored_fe.cu with G0 and K0 as the resident element matrices.
//
// Voigt order of h8_strain_rows: (xx, yy, zz, yz, xz, xy), engineering shear; S_q is the symmetric 3 x 3 form of the
// stress s_q = C B_q u_e.  With grad w_i the gradient of displacement component i of w at the Gauss point,
//   G0_e[3a+i, 3b+j]              = delta_ij sum_q detJ_q gradN_a^T S_q gradN_b
//   sum_k w_k^T G0_e(u) v_k       = sum_q detJ_q s_q . h_q,
//   h_q = sum_k sum_i (gwx gvx, gwy gvy, gwz gvz, gwy gvz + gwz gvy, gwx gvz + gwz gvx, gwx gvy + gwy gvx)_{i,k}
// and since s_q is linear in u, d/du_e of that form is sum_q detJ_q B_q^T C h_q.
//
// Displacements and the operands W, V are read through a dofmap (nelems, 24): element dof -> row, -1 on a constrained
// dof (contributes zero), so the reduced vectors of the buckling problem are used directly.  Element: h8_element.cuh.
#include "common.cuh"
#include "h8_element.cuh"
#include "../../include/eigd_b200.h"

namespace {

// One warp per element, the layout of h8_element_matrices_kernel: lane b < 24 owns column b (node b / 3, component
// b % 3) of G0_e, lane l evaluates node l & 7 at each Gauss point.  The strain at the point is a width-8 shuffle sum of
// the nodal terms.  G0 couples equal components only, so column b holds the 8 scalars of node b / 3 in rows 3 a + b % 3.
__global__ void __launch_bounds__(256)
h8_stress_stiffness_kernel(int nelems, const int* __restrict__ conn, const double* __restrict__ X, H8C c,
                           const double* __restrict__ kg, const int* __restrict__ dofmap, const double* __restrict__ u,
                           double* __restrict__ stress, double* __restrict__ G0) {
  const int lane = threadIdx.x & 31;
  const int64_t e = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (e >= nelems) return;  // whole warps only: blockDim is a multiple of 32
  const int a = lane & 7;
  const H8Node nd = h8_gather(conn, X, e, a);
  double ua[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const int d = dofmap[e * 24 + 3 * a + i];
    ua[i] = d >= 0 ? u[d] : 0.0;
  }
  const int bn = lane < 24 ? lane / 3 : 0, cb = lane < 24 ? lane % 3 : 0;
  const double kge = kg[e];
  double gc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) gc[i] = 0.0;
#pragma unroll 1
  for (int q = 0; q < 8; ++q) {
    double N, Nx, Ny, Nz;
    const double det = h8_point(nd, a, q, N, Nx, Ny, Nz);
    double eps[6] = {Nx * ua[0], Ny * ua[1], Nz * ua[2], fma(Nz, ua[1], Ny * ua[2]), fma(Nz, ua[0], Nx * ua[2]),
                     fma(Ny, ua[0], Nx * ua[1])};
#pragma unroll
    for (int o = 4; o > 0; o >>= 1)
#pragma unroll
      for (int i = 0; i < 6; ++i) eps[i] += __shfl_xor_sync(0xffffffffu, eps[i], o, 8);
    double s[6];
    h8_c_mul(c, eps, s);
    if (stress && lane == 0) {
#pragma unroll
      for (int i = 0; i < 6; ++i) stress[(e * 8 + q) * 6 + i] = kge * s[i];
    }
    const double nxb = __shfl_sync(0xffffffffu, Nx, bn), nyb = __shfl_sync(0xffffffffu, Ny, bn);
    const double nzb = __shfl_sync(0xffffffffu, Nz, bn);
    const double tx = s[0] * nxb + s[5] * nyb + s[4] * nzb;    // S gradN_b
    const double ty = s[5] * nxb + s[1] * nyb + s[3] * nzb;
    const double tz = s[4] * nxb + s[3] * nyb + s[2] * nzb;
#pragma unroll
    for (int an = 0; an < 8; ++an) {
      const double nxa = __shfl_sync(0xffffffffu, Nx, an), nya = __shfl_sync(0xffffffffu, Ny, an);
      const double nza = __shfl_sync(0xffffffffu, Nz, an);
      gc[an] = fma(det, nxa * tx + nya * ty + nza * tz, gc[an]);
    }
  }
  if (lane >= 24) return;
  double* g = G0 + e * 576 + lane;
#pragma unroll
  for (int r = 0; r < 24; ++r) g[r * 24] = (r % 3 == cb) ? gc[r / 3] : 0.0;
}

// gradients of the three displacement components of w and v at one Gauss point (width-8 sums of the nodal terms of
// this lane group), contracted into the six Voigt entries of h
__device__ __forceinline__ void h8_h_accumulate(const double n[3], const double w[3], const double v[3], double h[6]) {
  double gw[9], gv[9];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int m = 0; m < 3; ++m) {
      gw[3 * i + m] = w[i] * n[m];
      gv[3 * i + m] = v[i] * n[m];
    }
#pragma unroll
  for (int o = 4; o > 0; o >>= 1)
#pragma unroll
    for (int j = 0; j < 9; ++j) {
      gw[j] += __shfl_xor_sync(0xffffffffu, gw[j], o, 8);
      gv[j] += __shfl_xor_sync(0xffffffffu, gv[j], o, 8);
    }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double* x = gw + 3 * i;
    const double* y = gv + 3 * i;
    h[0] = fma(x[0], y[0], h[0]);
    h[1] = fma(x[1], y[1], h[1]);
    h[2] = fma(x[2], y[2], h[2]);
    h[3] += x[1] * y[2] + x[2] * y[1];
    h[4] += x[0] * y[2] + x[2] * y[0];
    h[5] += x[0] * y[1] + x[1] * y[0];
  }
}

// due[e][3 a + i] = kg[e] sum_q detJ_q (B_q^T C h_q)[3 a + i].  One warp per element: lane group g = lane >> 3 takes the
// Gauss points g and g + 4 and lane l the element node l & 7, so h8_point evaluates four points at once and every
// lane keeps only its own node's derivatives at its two points; the modes run in sequence, since each mode's
// gradients are a sum over the 8 nodes of the group anyway.  The B^T C h products of the four groups are summed at
// the end; lanes 0-7 write their node's three entries.
__global__ void __launch_bounds__(256)
h8_gderiv_u_kernel(int nelems, const int* __restrict__ conn, const double* __restrict__ X, H8C c,
                   const double* __restrict__ kg, const int* __restrict__ dofmap, const double* __restrict__ W,
                   const double* __restrict__ V, int N, int64_t ld, double* __restrict__ due) {
  const int lane = threadIdx.x & 31;
  const int64_t e = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (e >= nelems) return;  // whole warps only: blockDim is a multiple of 32
  const int a = lane & 7, grp = lane >> 3;
  const H8Node nd = h8_gather(conn, X, e, a);
  double N0, N1, n0[3], n1[3];
  const double det0 = h8_point(nd, a, grp, N0, n0[0], n0[1], n0[2]);
  const double det1 = h8_point(nd, a, grp + 4, N1, n1[0], n1[1], n1[2]);
  int dof[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) dof[i] = dofmap[e * 24 + 3 * a + i];
  double h0[6], h1[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) h0[i] = h1[i] = 0.0;
#pragma unroll 1
  for (int k = 0; k < N; ++k) {
    double w[3], v[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      w[i] = dof[i] >= 0 ? W[dof[i] * ld + k] : 0.0;
      v[i] = dof[i] >= 0 ? V[dof[i] * ld + k] : 0.0;
    }
    h8_h_accumulate(n0, w, v, h0);
    h8_h_accumulate(n1, w, v, h1);
  }
  double de[3] = {0.0, 0.0, 0.0};
#pragma unroll
  for (int p = 0; p < 2; ++p) {
    const double det = p ? det1 : det0;
    const double* n = p ? n1 : n0;
    const double* h = p ? h1 : h0;
    double f[6], t[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) f[i] = det * h[i];
    h8_c_mul(c, f, t);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      double b[6];
      h8_strain_rows(i, n[0], n[1], n[2], b);
#pragma unroll
      for (int j = 0; j < 6; ++j) de[i] = fma(b[j], t[j], de[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    de[i] += __shfl_xor_sync(0xffffffffu, de[i], 8);
    de[i] += __shfl_xor_sync(0xffffffffu, de[i], 16);
  }
  if (lane >= 8) return;
  const double kge = kg[e];
#pragma unroll
  for (int i = 0; i < 3; ++i) due[e * 24 + 3 * a + i] = kge * de[i];
}

}  // namespace

extern "C" int eigd_h8_stress_stiffness(int nelems, const int* d_conn, const double* d_X, double E, double nu,
                                        const double* d_kg, const int* d_dofmap, const double* d_u, double* d_stress,
                                        double* d_G0) {
  if (nelems <= 0) return 0;
  H8C c;
  if (!h8_isotropic(E, nu, c, "h8_stress_stiffness")) return 1;
  const int grid = (int)(((int64_t)nelems * 32 + 255) / 256);
  EIGD_LAUNCH(h8_stress_stiffness_kernel, grid, 256, 0, nelems, d_conn, d_X, c, d_kg, d_dofmap, d_u, d_stress, d_G0);
  EIGD_CHECK_LAUNCH();
  return 0;
}

extern "C" int eigd_h8_gderiv_u(int nelems, const int* d_conn, const double* d_X, double E, double nu, const double* d_kg,
                                const int* d_dofmap, const double* d_W, const double* d_V, int N, int64_t ld,
                                double* d_due) {
  if (nelems <= 0) return 0;
  H8C c;
  if (!h8_isotropic(E, nu, c, "h8_gderiv_u")) return 1;
  const int grid = (int)(((int64_t)nelems * 32 + 255) / 256);
  EIGD_LAUNCH(h8_gderiv_u_kernel, grid, 256, 0, nelems, d_conn, d_X, c, d_kg, d_dofmap, d_W, d_V, N, ld, d_due);
  EIGD_CHECK_LAUNCH();
  return 0;
}
