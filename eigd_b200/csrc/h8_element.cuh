// Trilinear hexahedron (H8) on the 2x2x2 Gauss rule, for the element kernels of h8.cu: element gather, shape
// functions and Jacobian, the strain column of a displacement dof and the product with the isotropic constitutive
// matrix.  Node numbering: nodes 0-3 counter-clockwise on the zeta = -1 face, nodes 4-7 above them (fe.hex_mesh).
//
// The routines are written for one warp per element: lane l works on element node l & 7, so each aligned group of
// 8 lanes holds the whole element and the Jacobian is a width-8 shuffle reduction.
#pragma once

struct H8Node {
  int nd;
  double x, y, z;
};

// node a of element e (conn row-major (nelems, 8), X row-major (nnodes, 3))
__device__ __forceinline__ H8Node h8_gather(const int* __restrict__ conn, const double* __restrict__ X, int64_t e, int a) {
  H8Node n;
  n.nd = conn[e * 8 + a];
  n.x = X[3 * (int64_t)n.nd];
  n.y = X[3 * (int64_t)n.nd + 1];
  n.z = X[3 * (int64_t)n.nd + 2];
  return n;
}

// shape function of node a and its x / y / z derivatives at Gauss point q (xi: bit 0, eta: bit 1, zeta: bit 2);
// returns detJ.  Every lane of the warp must call it (shuffles); lane l contributes node l & 7 == a.
__device__ __forceinline__ double h8_point(const H8Node& n, int a, int q, double& N, double& Nx, double& Ny, double& Nz) {
  const double gp = 0.57735026918962576451;
  const double xi = (q & 1) ? gp : -gp, eta = (q & 2) ? gp : -gp, zeta = (q & 4) ? gp : -gp;
  const double sa = (a == 1 || a == 2 || a == 5 || a == 6) ? 1.0 : -1.0;
  const double ta = (a == 2 || a == 3 || a == 6 || a == 7) ? 1.0 : -1.0;
  const double ua = a >= 4 ? 1.0 : -1.0;
  const double fx = 1.0 + sa * xi, fy = 1.0 + ta * eta, fz = 1.0 + ua * zeta;
  N = 0.125 * fx * fy * fz;
  const double Nxi = 0.125 * sa * fy * fz, Neta = 0.125 * ta * fx * fz, Nzeta = 0.125 * ua * fx * fy;
  // J[i][j] = d x_i / d xi_j, summed over the 8 nodes of this lane group
  double J[9] = {n.x * Nxi, n.x * Neta, n.x * Nzeta, n.y * Nxi, n.y * Neta, n.y * Nzeta, n.z * Nxi, n.z * Neta, n.z * Nzeta};
#pragma unroll
  for (int o = 4; o > 0; o >>= 1)
#pragma unroll
    for (int i = 0; i < 9; ++i) J[i] += __shfl_xor_sync(0xffffffffu, J[i], o, 8);
  const double c00 = J[4] * J[8] - J[5] * J[7], c01 = J[5] * J[6] - J[3] * J[8], c02 = J[3] * J[7] - J[4] * J[6];
  const double det = J[0] * c00 + J[1] * c01 + J[2] * c02;
  const double r = 1.0 / det;
  // inverse: Jinv[j][i] = d xi_j / d x_i;  dN/dx_i = sum_j Jinv[j][i] dN/dxi_j
  const double i00 = c00 * r, i01 = (J[2] * J[7] - J[1] * J[8]) * r, i02 = (J[1] * J[5] - J[2] * J[4]) * r;
  const double i10 = c01 * r, i11 = (J[0] * J[8] - J[2] * J[6]) * r, i12 = (J[2] * J[3] - J[0] * J[5]) * r;
  const double i20 = c02 * r, i21 = (J[1] * J[6] - J[0] * J[7]) * r, i22 = (J[0] * J[4] - J[1] * J[3]) * r;
  Nx = i00 * Nxi + i10 * Neta + i20 * Nzeta;
  Ny = i01 * Nxi + i11 * Neta + i21 * Nzeta;
  Nz = i02 * Nxi + i12 * Neta + i22 * Nzeta;
  return det;
}

// column of B for displacement component c (0 = u_x, 1 = u_y, 2 = u_z) of a node with derivatives (nx, ny, nz);
// strain order (eps_xx, eps_yy, eps_zz, gamma_yz, gamma_xz, gamma_xy)
__device__ __forceinline__ void h8_strain_rows(int c, double nx, double ny, double nz, double b[6]) {
  b[0] = c == 0 ? nx : 0.0;
  b[1] = c == 1 ? ny : 0.0;
  b[2] = c == 2 ? nz : 0.0;
  b[3] = c == 1 ? nz : (c == 2 ? ny : 0.0);
  b[4] = c == 0 ? nz : (c == 2 ? nx : 0.0);
  b[5] = c == 0 ? ny : (c == 1 ? nx : 0.0);
}

// isotropic elasticity: C = lambda 1 1^T + mu diag(2, 2, 2, 1, 1, 1)
struct H8C {
  double lam, mu;
};

// Lame constants of (E, nu) on the host; false (error set, prefixed with `what`) for nu outside (-1, 0.5).
// Include common.cuh first.
inline bool h8_isotropic(double E, double nu, H8C& c, const char* what) {
  if (!(nu > -1.0 && nu < 0.5)) {
    eigd_set_error("%s: Poisson ratio %g outside (-1, 0.5)", what, nu);
    return false;
  }
  c = {E * nu / ((1.0 + nu) * (1.0 - 2.0 * nu)), E / (2.0 * (1.0 + nu))};
  return true;
}

// s = C e
__device__ __forceinline__ void h8_c_mul(const H8C& c, const double e[6], double s[6]) {
  const double tr = c.lam * (e[0] + e[1] + e[2]);
  s[0] = fma(2.0 * c.mu, e[0], tr);
  s[1] = fma(2.0 * c.mu, e[1], tr);
  s[2] = fma(2.0 * c.mu, e[2], tr);
  s[3] = c.mu * e[3];
  s[4] = c.mu * e[4];
  s[5] = c.mu * e[5];
}
