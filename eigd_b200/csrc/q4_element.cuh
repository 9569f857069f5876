// Bilinear quadrilateral (Q4) element on the 2x2 Gauss rule, shared by the element kernels of fe.cu and
// buckling.cu: element gather, shape functions and Jacobian (examples/fe_utils.py:4-16, 26-44), plane-stress
// strain, the product with the constitutive matrix C0 and the strain rows of a displacement dof.
//
// The kernels' results are reproducible bit for bit across changes of this file only as long as each helper
// keeps its operand order, fma nesting and summation order.
#pragma once

struct Q4Nodes {
  int nd[4];
  double x[4], y[4];
};

// node ids and coordinates of element e
__device__ __forceinline__ Q4Nodes q4_gather(const int* __restrict__ conn, const double* __restrict__ xy, int e) {
  Q4Nodes el;
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    el.nd[a] = conn[e * 4 + a];
    el.x[a] = xy[2 * el.nd[a]];
    el.y[a] = xy[2 * el.nd[a] + 1];
  }
  return el;
}

// shape functions N and their x / y derivatives at Gauss point q; returns detJ.
// q = 2*j + i with xi = pts[i], eta = pts[j] (examples/thermal.py:117); element sums do not depend on it.
__device__ __forceinline__ double q4_point(const Q4Nodes& el, int q, double N[4], double Nx[4], double Ny[4]) {
  const double gp = 0.57735026918962576451;
  const double xi = (q & 1) ? gp : -gp;
  const double eta = (q & 2) ? gp : -gp;
  const double Nxi[4] = {-0.25 * (1.0 - eta), 0.25 * (1.0 - eta), 0.25 * (1.0 + eta), -0.25 * (1.0 + eta)};
  const double Neta[4] = {-0.25 * (1.0 - xi), -0.25 * (1.0 + xi), 0.25 * (1.0 + xi), 0.25 * (1.0 - xi)};
  N[0] = 0.25 * (1.0 - xi) * (1.0 - eta);
  N[1] = 0.25 * (1.0 + xi) * (1.0 - eta);
  N[2] = 0.25 * (1.0 + xi) * (1.0 + eta);
  N[3] = 0.25 * (1.0 - xi) * (1.0 + eta);
  double J00 = 0, J10 = 0, J01 = 0, J11 = 0;
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    J00 = fma(el.x[a], Nxi[a], J00);
    J10 = fma(el.y[a], Nxi[a], J10);
    J01 = fma(el.x[a], Neta[a], J01);
    J11 = fma(el.y[a], Neta[a], J11);
  }
  const double det = J00 * J11 - J01 * J10;
  const double i00 = J11 / det, i01 = -J01 / det, i10 = -J10 / det, i11 = J00 / det;
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    Nx[a] = i00 * Nxi[a] + i10 * Neta[a];
    Ny[a] = i01 * Nxi[a] + i11 * Neta[a];
  }
  return det;
}

struct Q4Geom {
  double N[4][4], Nx[4][4], Ny[4][4], detJ[4];  // [gauss point][node]
};

__device__ __forceinline__ Q4Geom q4_geometry(const Q4Nodes& el) {
  Q4Geom g;
#pragma unroll
  for (int q = 0; q < 4; ++q) g.detJ[q] = q4_point(el, q, g.N[q], g.Nx[q], g.Ny[q]);
  return g;
}

// the values of node n at one Gauss point, selected without dynamic register indexing
__device__ __forceinline__ void q4_node(int n, const double N[4], const double Nx[4], const double Ny[4], double& nn,
                                        double& nx, double& ny) {
  nn = nx = ny = 0.0;
#pragma unroll
  for (int i = 0; i < 4; ++i)
    if (i == n) { nn = N[i]; nx = Nx[i]; ny = Ny[i]; }
}

// plane-stress strain (eps_x, eps_y, gamma_xy) at one Gauss point of the nodal vector u = (u_x, u_y) per node
__device__ __forceinline__ void q4_strain(const double Nx[4], const double Ny[4], const double u[8], double eps[3]) {
  eps[0] = eps[1] = eps[2] = 0.0;
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    eps[0] = fma(Nx[a], u[2 * a], eps[0]);
    eps[1] = fma(Ny[a], u[2 * a + 1], eps[1]);
    eps[2] = fma(Ny[a], u[2 * a], fma(Nx[a], u[2 * a + 1], eps[2]));
  }
}

// column of Be for displacement component c (0 = u, 1 = v) of a node: u -> [Nx, 0, Ny], v -> [0, Ny, Nx].
// Row 1 - c is zero.
__device__ __forceinline__ void q4_strain_rows(int c, double nx, double ny, double b[3]) {
  b[0] = c ? 0.0 : nx;
  b[1] = c ? ny : 0.0;
  b[2] = c ? nx : ny;
}

// symmetric plane-stress constitutive matrix from its 6 entries c00 c01 c02 c11 c12 c22
struct Q4C0 {
  double c00, c01, c02, c11, c12, c22;
};

__device__ __forceinline__ Q4C0 q4_c0_load(const double* __restrict__ cmat) {
  return {cmat[0], cmat[1], cmat[2], cmat[3], cmat[4], cmat[5]};
}

// s = C0 e
__device__ __forceinline__ void q4_c0_mul(const Q4C0& c, const double e[3], double s[3]) {
  s[0] = c.c00 * e[0] + c.c01 * e[1] + c.c02 * e[2];
  s[1] = c.c01 * e[0] + c.c11 * e[1] + c.c12 * e[2];
  s[2] = c.c02 * e[0] + c.c12 * e[1] + c.c22 * e[2];
}
