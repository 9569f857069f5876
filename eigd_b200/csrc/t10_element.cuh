// Quadratic tetrahedron (T10) for the element kernels of t10.cu: element gather, quadratic shape functions in
// barycentric coordinates, their gradients and the Jacobian at a quadrature point.  Node order is VTK's quadratic tetra:
// corners 0-3 (positive corner volume), then the midside nodes of the edges (0,1), (1,2), (2,0), (0,3), (1,3), (2,3).
//
// With barycentric coordinates l0 = 1 - xi - eta - zeta, l1 = xi, l2 = eta, l3 = zeta of the reference tetrahedron:
//   corner a:      N_a = l_a (2 l_a - 1)
//   edge (i, j):   N   = 4 l_i l_j
// The Jacobian is evaluated in full at every point (not taken as constant), so curved midside nodes are integrated
// correctly.  One quadrature rule serves K and M: the 14-point degree-5 rule with positive weights (Walkington), which
// is exact for M = N N^T (degree 4) on straight-sided elements.
//
// The routines are written for 16-lane groups: lane l works on element node l & 15, lanes with l & 15 >= 10 carry
// zeros, and the Jacobian is a width-16 shuffle reduction.
#pragma once

// T10_RULE: rows {l1, l2, l3, w} of the 14 points; the weights sum to 1/6, the volume of the reference tetrahedron, so
// that the integral over an element is sum_q w_q detJ_q f(q).  tests/t10_oracle.py reads this table from here.
__constant__ double t10_rule[14][4] = {
    {0.3108859192633006097973, 0.3108859192633006097973, 0.3108859192633006097973, 0.01878132095300264179986},
    {0.06734224221009817060796, 0.3108859192633006097973, 0.3108859192633006097973, 0.01878132095300264179986},
    {0.3108859192633006097973, 0.06734224221009817060796, 0.3108859192633006097973, 0.01878132095300264179986},
    {0.3108859192633006097973, 0.3108859192633006097973, 0.06734224221009817060796, 0.01878132095300264179986},
    {0.09273525031089122640232, 0.09273525031089122640232, 0.09273525031089122640232, 0.01224884051939365825729},
    {0.721794249067326320793, 0.09273525031089122640232, 0.09273525031089122640232, 0.01224884051939365825729},
    {0.09273525031089122640232, 0.721794249067326320793, 0.09273525031089122640232, 0.01224884051939365825729},
    {0.09273525031089122640232, 0.09273525031089122640232, 0.721794249067326320793, 0.01224884051939365825729},
    {0.4544962958743503505081, 0.04550370412564964949188, 0.04550370412564964949188, 0.007091003462846911073012},
    {0.04550370412564964949188, 0.4544962958743503505081, 0.04550370412564964949188, 0.007091003462846911073012},
    {0.04550370412564964949188, 0.04550370412564964949188, 0.4544962958743503505081, 0.007091003462846911073012},
    {0.4544962958743503505081, 0.4544962958743503505081, 0.04550370412564964949188, 0.007091003462846911073012},
    {0.4544962958743503505081, 0.04550370412564964949188, 0.4544962958743503505081, 0.007091003462846911073012},
    {0.04550370412564964949188, 0.4544962958743503505081, 0.4544962958743503505081, 0.007091003462846911073012},
};
constexpr int T10_NQ = 14;

struct T10Node {
  double x, y, z;
};

// node a of element e (conn row-major (nelems, 10), X row-major (nnodes, 3)); zeros for a >= 10
__device__ __forceinline__ T10Node t10_gather(const int* __restrict__ conn, const double* __restrict__ X, int64_t e, int a) {
  T10Node n = {0.0, 0.0, 0.0};
  if (a < 10) {
    const int64_t nd = conn[e * 10 + a];
    n.x = X[3 * nd];
    n.y = X[3 * nd + 1];
    n.z = X[3 * nd + 2];
  }
  return n;
}

__device__ __forceinline__ double t10_pick(int k, double l0, double l1, double l2, double l3) {
  return k == 0 ? l0 : (k == 1 ? l1 : (k == 2 ? l2 : l3));
}

// shape function of node a and its x / y / z derivatives at quadrature point q; returns w_q detJ (the volume weight of
// the point).  Every lane of the warp must call it (shuffles); lane l contributes node l & 15 == a (nothing if a >= 10).
__device__ __forceinline__ double t10_point(const T10Node& n, int a, int q, double& N, double& Nx, double& Ny, double& Nz) {
  const double l1 = t10_rule[q][0], l2 = t10_rule[q][1], l3 = t10_rule[q][2];
  const double l0 = 1.0 - l1 - l2 - l3;
  // the node's barycentric pair (i, j): i == j for a corner; dN/dl_i = gi, dN/dl_j = gj
  const int i = a < 4 ? a : (a == 4 || a == 7) ? 0 : (a == 5 || a == 8) ? 1 : 2;
  const int j = a < 4 ? a : a == 4 ? 1 : a == 5 ? 2 : a == 6 ? 0 : 3;
  const double li = t10_pick(i, l0, l1, l2, l3), lj = t10_pick(j, l0, l1, l2, l3);
  double gi, gj;
  if (a < 4) {
    N = li * (2.0 * li - 1.0);
    gi = 4.0 * li - 1.0;
    gj = 0.0;
  } else if (a < 10) {
    N = 4.0 * li * lj;
    gi = 4.0 * lj;
    gj = 4.0 * li;
  } else {
    N = gi = gj = 0.0;
  }
  // dN/dxi_k = dN/dl_k - dN/dl_0 (k = 1, 2, 3)
  const double g0 = (i == 0 ? gi : 0.0) + (j == 0 ? gj : 0.0);
  const double Nxi = (i == 1 ? gi : 0.0) + (j == 1 ? gj : 0.0) - g0;
  const double Neta = (i == 2 ? gi : 0.0) + (j == 2 ? gj : 0.0) - g0;
  const double Nzeta = (i == 3 ? gi : 0.0) + (j == 3 ? gj : 0.0) - g0;
  // J[i][j] = d x_i / d xi_j, summed over the 10 nodes of this lane group
  double J[9] = {n.x * Nxi, n.x * Neta, n.x * Nzeta, n.y * Nxi, n.y * Neta, n.y * Nzeta, n.z * Nxi, n.z * Neta, n.z * Nzeta};
#pragma unroll
  for (int o = 8; o > 0; o >>= 1)
#pragma unroll
    for (int k = 0; k < 9; ++k) J[k] += __shfl_xor_sync(0xffffffffu, J[k], o, 16);
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
  return t10_rule[q][3] * det;
}
