// Linearised-buckling element kernels for the plane-stress Q4 column problem of the reference
// (examples/buckling.py): element stresses of the fundamental path, gather-form assembly of the stress
// (geometric) stiffness matrix G(u, x), and the fused sensitivities of  sum_k w_k^T G(u, x) v_k  with
// respect to the element densities and to the displacement u, plus the Dirichlet reduce / expand maps.
//
// Replaces (paths relative to the reference root):
//   get_stress_stiffness_matrix                       examples/buckling.py:220-255
//   intital_stress_stiffness_matrix_deriv             examples/buckling.py:283-310   (dfds)
//   get_stress_stiffness_matrix_uderiv_tensor         examples/buckling.py:312-322
//   get_stress_stiffness_matrix_xderiv_tensor         examples/buckling.py:324-343
//   reduce_vector / full_vector                       examples/buckling.py:499-518
//   Be, Te, detJ                                      examples/fe_utils.py:58-98
#include "common.cuh"
#include "q4_element.cuh"
#include "../../include/eigd_b200.h"

namespace {

// sdet[e][q][i] = detJ_q * ks[e] * (C0 Be(q) u_e)_i : the weights of Te in the element stress stiffness
__global__ void __launch_bounds__(128)
q4_stress_kernel(int nelems, const int* __restrict__ conn, const double* __restrict__ xy, const double* __restrict__ cmat,
                 const double* __restrict__ ks, const double* __restrict__ u, double* __restrict__ sdet) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nelems) return;
  const Q4Nodes el = q4_gather(conn, xy, e);
  const Q4Geom g = q4_geometry(el);
  double ue[8];
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    ue[2 * a] = u[2 * el.nd[a]];
    ue[2 * a + 1] = u[2 * el.nd[a] + 1];
  }
  const Q4C0 c0 = q4_c0_load(cmat);
  const double s = ks[e];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    double eps[3], sig[3];
    q4_strain(g.Nx[q], g.Ny[q], ue, eps);
    q4_c0_mul(c0, eps, sig);
    const double w = g.detJ[q] * s;
#pragma unroll
    for (int i = 0; i < 3; ++i) sdet[(e * 4 + q) * 3 + i] = w * sig[i];
  }
}

// gather-form assembly of G: non-zero p = sum over its (element, a, b) sources of
// sum_q s0 Nxa Nxb + s1 Nya Nyb + s2 (Nxa Nyb + Nya Nxb), non-zero only for equal displacement components
__global__ void q4_assemble_geometric_kernel(int64_t nnz, const int64_t* __restrict__ src_ptr, const int64_t* __restrict__ src,
                                             const int* __restrict__ conn, const double* __restrict__ xy,
                                             const double* __restrict__ sdet, double* __restrict__ Gv) {
  int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nnz) return;
  double gv = 0.0;
  for (int64_t qq = src_ptr[p]; qq < src_ptr[p + 1]; ++qq) {
    int64_t s = src[qq];
    int e = (int)(s / 64);
    int ab = (int)(s - (int64_t)e * 64);
    int a = ab >> 3, b = ab & 7;
    if ((a & 1) != (b & 1)) continue;
    const Q4Nodes el = q4_gather(conn, xy, e);
    double ge = 0.0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const double* sd = sdet + ((int64_t)e * 4 + q) * 3;
      double N[4], Nx[4], Ny[4], na, nxa, nya, nb, nxb, nyb;
      q4_point(el, q, N, Nx, Ny);
      q4_node(a >> 1, N, Nx, Ny, na, nxa, nya);
      q4_node(b >> 1, N, Nx, Ny, nb, nxb, nyb);
      ge += sd[0] * nxa * nxb + sd[1] * nya * nyb + sd[2] * (nxa * nyb + nya * nxb);
    }
    gv += ge;
  }
  Gv[p] = gv;
}

// Per element, with G lanes splitting the modes:
//   dfds[q][i] = detJ_q sum_k sum_d  Te_i(q) : (w_{d,k} v_{d,k}^T)                  (examples/buckling.py:283-310)
//   out_rho[e] += sx * dks[e] * sum_q sum_j (C0 dfds[q])_j (Be(q) u_e)_j             (:324-343)
//   due[e][j8]  = ks[e] * sum_q sum_j Be[j][j8](q) (C0 dfds[q])_j                    (:312-322)
template <int G>
__global__ void __launch_bounds__(256)
q4_gderiv_kernel(int nelems, const int* __restrict__ conn, const double* __restrict__ xy, const double* __restrict__ cmat,
                 const double* __restrict__ W, const double* __restrict__ V, int N, int ldw, const double* __restrict__ ks,
                 const double* __restrict__ dks, const double* __restrict__ u, double sx, double* __restrict__ out_rho,
                 double* __restrict__ due) {
  const int lane = threadIdx.x & (G - 1);
  int e = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G);
  const bool valid = e < nelems;
  if (!valid) e = nelems - 1;
  const Q4Nodes el = q4_gather(conn, xy, e);
  const Q4Geom g = q4_geometry(el);
  double dfds[4][3];
#pragma unroll
  for (int q = 0; q < 4; ++q) dfds[q][0] = dfds[q][1] = dfds[q][2] = 0.0;
  for (int k = lane; k < N; k += G) {
    double w[8], v[8];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      int64_t o = (int64_t)(2 * el.nd[a]) * ldw + k;
      w[2 * a] = W[o];
      w[2 * a + 1] = W[o + ldw];
      v[2 * a] = V[o];
      v[2 * a + 1] = V[o + ldw];
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
#pragma unroll
      for (int d = 0; d < 2; ++d) {
        double gxw = 0, gyw = 0, gxv = 0, gyv = 0;
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          gxw = fma(g.Nx[q][a], w[2 * a + d], gxw);
          gyw = fma(g.Ny[q][a], w[2 * a + d], gyw);
          gxv = fma(g.Nx[q][a], v[2 * a + d], gxv);
          gyv = fma(g.Ny[q][a], v[2 * a + d], gyv);
        }
        dfds[q][0] = fma(gxw, gxv, dfds[q][0]);
        dfds[q][1] = fma(gyw, gyv, dfds[q][1]);
        dfds[q][2] += gxw * gyv + gyw * gxv;
      }
    }
  }
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
      for (int o = G >> 1; o > 0; o >>= 1) dfds[q][i] += __shfl_xor_sync(0xffffffffu, dfds[q][i], o, G);
    }
  if (!valid || lane != 0) return;
  const Q4C0 c0 = q4_c0_load(cmat);
  double ue[8];
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    ue[2 * a] = u[2 * el.nd[a]];
    ue[2 * a + 1] = u[2 * el.nd[a] + 1];
  }
  double drho = 0.0;
  double de[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const double f[3] = {g.detJ[q] * dfds[q][0], g.detJ[q] * dfds[q][1], g.detJ[q] * dfds[q][2]};
    double t[3], eps[3];
    q4_c0_mul(c0, f, t);
    q4_strain(g.Nx[q], g.Ny[q], ue, eps);
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int d = 0; d < 2; ++d) {
        double b[3];
        q4_strain_rows(d, g.Nx[q][a], g.Ny[q][a], b);
        de[2 * a + d] += b[d] * t[d] + b[2] * t[2];  // Be^T t without the zero row 1 - d
      }
    drho += t[0] * eps[0] + t[1] * eps[1] + t[2] * eps[2];
  }
  if (out_rho) out_rho[e] += sx * dks[e] * drho;
  if (due) {
    const double s = ks[e];
#pragma unroll
    for (int j = 0; j < 8; ++j) due[(int64_t)e * 8 + j] = s * de[j];
  }
}

// full[idx[i], :] = red[i, :]   (full_vector, :506-511; the rest of `full` must be zero)
__global__ void expand_rows_kernel(int64_t nr, int k, const int* __restrict__ idx, const double* __restrict__ red,
                                   double* __restrict__ full) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nr * k) return;
  int64_t i = t / k;
  int c = (int)(t - i * k);
  full[(int64_t)idx[i] * k + c] = red[t];
}

// red[i, :] = full[idx[i], :]   (reduce_vector, :499-503)
__global__ void reduce_rows_kernel(int64_t nr, int k, const int* __restrict__ idx, const double* __restrict__ full,
                                   double* __restrict__ red) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nr * k) return;
  int64_t i = t / k;
  int c = (int)(t - i * k);
  red[t] = full[(int64_t)idx[i] * k + c];
}

}  // namespace

extern "C" int eigd_q4_stress(int nelems, const int* d_conn, const double* d_xy, const double* d_cmat6, const double* d_ks,
                              const double* d_u, double* d_sdet) {
  if (nelems <= 0) return 0;
  EIGD_LAUNCH(q4_stress_kernel, (nelems + 127) / 128, 128, 0, nelems, d_conn, d_xy, d_cmat6, d_ks, d_u, d_sdet);
  EIGD_CHECK_LAUNCH();
  return 0;
}

extern "C" int eigd_q4_assemble_geometric(int nelems, const int* d_conn, const double* d_xy, const double* d_sdet,
                                          const int64_t* d_src_ptr, const int64_t* d_src, int64_t nnz, double* d_Gvals) {
  (void)nelems;
  if (nnz <= 0) return 0;
  EIGD_LAUNCH(q4_assemble_geometric_kernel, (int)((nnz + 127) / 128), 128, 0, nnz, d_src_ptr, d_src, d_conn, d_xy, d_sdet, d_Gvals);
  EIGD_CHECK_LAUNCH();
  return 0;
}

extern "C" int eigd_q4_gderiv(int nelems, const int* d_conn, const double* d_xy, const double* d_cmat6, const double* d_W,
                              const double* d_V, int N, int ldw, const double* d_ks, const double* d_dks, const double* d_u,
                              double sx, double* d_out_rho, double* d_due) {
  if (nelems <= 0 || N <= 0) return 0;
  constexpr int G = 8;
  int grid = (int)(((int64_t)nelems * G + 255) / 256);
  EIGD_LAUNCH((q4_gderiv_kernel<G>), grid, 256, 0, nelems, d_conn, d_xy, d_cmat6, d_W, d_V, N, ldw, d_ks, d_dks, d_u, sx,
              d_out_rho, d_due);
  EIGD_CHECK_LAUNCH();
  return 0;
}

extern "C" int eigd_expand_rows(int64_t nr, int k, const int* d_idx, const double* d_red, double* d_full) {
  if (nr <= 0 || k <= 0) return 0;
  EIGD_LAUNCH(expand_rows_kernel, (int)((nr * k + 255) / 256), 256, 0, nr, k, d_idx, d_red, d_full);
  EIGD_CHECK_LAUNCH();
  return 0;
}

extern "C" int eigd_reduce_rows(int64_t nr, int k, const int* d_idx, const double* d_full, double* d_red) {
  if (nr <= 0 || k <= 0) return 0;
  EIGD_LAUNCH(reduce_rows_kernel, (int)((nr * k + 255) / 256), 256, 0, nr, k, d_idx, d_full, d_red);
  EIGD_CHECK_LAUNCH();
  return 0;
}
