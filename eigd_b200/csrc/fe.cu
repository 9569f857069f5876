// Q4 element kernels: per-element bilinear forms w_e^T (dK_e/ds) v_e, w_e^T (dM_e/dm) v_e summed
// over modes (warp-shuffle segmented reduction, one lane group per element), gather-form
// assembly of K and M through the (element, a, b) -> CSR map, the element -> node gather and the element -> dof gather
// of the buckling problems.
//
// Replaces the numpy einsum callbacks of the reference examples:
//   thermal      examples/thermal.py:126-148 (K), :150-190 (dK), :192-214 (M), :216-246 (dM)
//   plane stress examples/natural_frequency.py:134-160 (K), :162-203 (dK), :205-236 (M), :238-284 (dM)
//   node scatter examples/thermal.py:612-615, examples/natural_frequency.py:509-512
// Shape functions, Jacobian and strain: q4_element.cuh.
#include "common.cuh"
#include "q4_element.cuh"
#include "../../include/eigd_b200.h"

namespace {

// G lanes per element; lane l handles modes l, l+G, ...
template <int KIND, int G>
__global__ void __launch_bounds__(256)
q4_quadforms_kernel(int nelems, const int* __restrict__ conn, const double* __restrict__ xy,
                    const double* __restrict__ cmat, const double* __restrict__ WA, const double* __restrict__ WB,
                    const double* __restrict__ V, int N, int ldw, const double* __restrict__ dk,
                    const double* __restrict__ dm, double sA, double sB, double* __restrict__ out) {
  const int lane = threadIdx.x & (G - 1);
  int e = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G);
  const bool valid = e < nelems;
  if (!valid) e = nelems - 1;  // keep the whole warp converged for the shuffles
  const Q4Nodes el = q4_gather(conn, xy, e);
  const Q4Geom g = q4_geometry(el);
  const Q4C0 c0 = KIND == 1 ? q4_c0_load(cmat) : Q4C0{};  // cmat may be NULL for kind 0
  double sumK = 0.0, sumM = 0.0;
  for (int k = lane; k < N; k += G) {
    if (KIND == 0) {
      double wa[4], wb[4], v[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        int64_t o = (int64_t)el.nd[a] * ldw + k;
        v[a] = V[o];
        wa[a] = WA ? WA[o] : 0.0;
        wb[a] = WB ? WB[o] : 0.0;
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        double gxw = 0, gyw = 0, gxv = 0, gyv = 0, nw = 0, nv = 0;
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          gxw = fma(g.Nx[q][a], wa[a], gxw);
          gyw = fma(g.Ny[q][a], wa[a], gyw);
          gxv = fma(g.Nx[q][a], v[a], gxv);
          gyv = fma(g.Ny[q][a], v[a], gyv);
          nw = fma(g.N[q][a], wb[a], nw);
          nv = fma(g.N[q][a], v[a], nv);
        }
        sumK = fma(g.detJ[q], gxw * gxv + gyw * gyv, sumK);
        sumM = fma(g.detJ[q], nw * nv, sumM);
      }
    } else {
      double wa[8], wb[8], v[8];
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        int64_t o = (int64_t)(2 * el.nd[a]) * ldw + k;
        v[2 * a] = V[o];
        v[2 * a + 1] = V[o + ldw];
        wa[2 * a] = WA ? WA[o] : 0.0;
        wa[2 * a + 1] = WA ? WA[o + ldw] : 0.0;
        wb[2 * a] = WB ? WB[o] : 0.0;
        wb[2 * a + 1] = WB ? WB[o + ldw] : 0.0;
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        double ew[3], ev[3], s[3], hw[2] = {0, 0}, hv[2] = {0, 0};
        q4_strain(g.Nx[q], g.Ny[q], wa, ew);
        q4_strain(g.Nx[q], g.Ny[q], v, ev);
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          hw[0] = fma(g.N[q][a], wb[2 * a], hw[0]);
          hw[1] = fma(g.N[q][a], wb[2 * a + 1], hw[1]);
          hv[0] = fma(g.N[q][a], v[2 * a], hv[0]);
          hv[1] = fma(g.N[q][a], v[2 * a + 1], hv[1]);
        }
        q4_c0_mul(c0, ev, s);
        sumK = fma(g.detJ[q], ew[0] * s[0] + ew[1] * s[1] + ew[2] * s[2], sumK);
        sumM = fma(g.detJ[q], hw[0] * hv[0] + hw[1] * hv[1], sumM);
      }
    }
  }
  // segmented reduction over the G lanes of this element
#pragma unroll
  for (int o = G >> 1; o > 0; o >>= 1) {
    sumK += __shfl_xor_sync(0xffffffffu, sumK, o, G);
    sumM += __shfl_xor_sync(0xffffffffu, sumM, o, G);
  }
  if (valid && lane == 0) {
    double r = 0.0;
    if (WA) r += sA * (dk ? dk[e] : 1.0) * sumK;
    if (WB) r -= sB * (dm ? dm[e] : 1.0) * sumM;
    out[e] += r;
  }
}

// gather-form assembly: value of CSR non-zero p = sum over its (element, a, b) sources
template <int KIND>
__global__ void q4_assemble_kernel(int64_t nnz, const int64_t* __restrict__ src_ptr, const int64_t* __restrict__ src,
                                   const int* __restrict__ conn, const double* __restrict__ xy,
                                   const double* __restrict__ ks, const double* __restrict__ ms,
                                   const double* __restrict__ cmat, double* __restrict__ Kv, double* __restrict__ Mv) {
  int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nnz) return;
  constexpr int NE = (KIND == 0) ? 4 : 8;
  const Q4C0 c0 = KIND == 1 ? q4_c0_load(cmat) : Q4C0{};  // cmat may be NULL for kind 0
  double kv = 0.0, mv = 0.0;
  for (int64_t q = src_ptr[p]; q < src_ptr[p + 1]; ++q) {
    int64_t s = src[q];
    int e = (int)(s / (NE * NE));
    int ab = (int)(s - (int64_t)e * NE * NE);
    int a = ab / NE, b = ab - a * NE;
    const int ia = KIND == 0 ? a : a >> 1, ib = KIND == 0 ? b : b >> 1;  // element nodes of dofs a, b
    const Q4Nodes el = q4_gather(conn, xy, e);
    double ke = 0.0, me = 0.0;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      double N[4], Nx[4], Ny[4], na, nxa, nya, nb, nxb, nyb;
      const double det = q4_point(el, g, N, Nx, Ny);
      q4_node(ia, N, Nx, Ny, na, nxa, nya);
      q4_node(ib, N, Nx, Ny, nb, nxb, nyb);
      if (KIND == 0) {
        ke = fma(det, nxa * nxb + nya * nyb, ke);
        me = fma(det, na * nb, me);
      } else {
        const int ca = a & 1, cb = b & 1;
        double ba[3], bb[3], t[3];
        q4_strain_rows(ca, nxa, nya, ba);
        q4_strain_rows(cb, nxb, nyb, bb);
        q4_c0_mul(c0, bb, t);
        ke = fma(det, ba[0] * t[0] + ba[1] * t[1] + ba[2] * t[2], ke);
        if (ca == cb) me = fma(det, na * nb, me);
      }
    }
    kv = fma(ks[e], ke, kv);
    mv = fma(ms[e], me, mv);
  }
  if (Kv) Kv[p] = kv;
  if (Mv) Mv[p] = mv;
}

__global__ void node_gather_kernel(int nnodes, const int* __restrict__ nptr, const int* __restrict__ nelem,
                                   const double* __restrict__ ev, double scale, double* __restrict__ out) {
  int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nnodes) return;
  double s = 0.0;
  for (int p = nptr[v]; p < nptr[v + 1]; ++p) s += ev[nelem[p]];
  out[v] = scale * s;
}

// out[NC v + i] = sum over the elements e around node v of due[e][NC local(v, e) + i], due (nelems, npe * NC): the
// gather form of the dof scatter np.add.at (examples/buckling.py:318-320), deterministic and without atomics
template <int NC>
__global__ void dof_gather_kernel(int nnodes, int npe, const int* __restrict__ nptr, const int* __restrict__ nelem,
                                  const int* __restrict__ nlocal, const double* __restrict__ due, double* __restrict__ out) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nnodes) return;
  double s[NC];
#pragma unroll
  for (int i = 0; i < NC; ++i) s[i] = 0.0;
  for (int p = nptr[v]; p < nptr[v + 1]; ++p) {
    const double* d = due + (int64_t)nelem[p] * (npe * NC) + NC * nlocal[p];
#pragma unroll
    for (int i = 0; i < NC; ++i) s[i] += d[i];
  }
#pragma unroll
  for (int i = 0; i < NC; ++i) out[NC * (int64_t)v + i] = s[i];
}

}  // namespace

extern "C" int eigd_q4_assemble(int kind, int nelems, const int* d_conn, const double* d_xy, const double* d_ks,
                                const double* d_ms, const double* d_cmat6, const int64_t* d_src_ptr,
                                const int64_t* d_src, int64_t nnz, double* d_Kvals, double* d_Mvals) {
  (void)nelems;
  if (nnz <= 0) return 0;
  int grid = (int)((nnz + 127) / 128);
  if (kind == 0) EIGD_LAUNCH(q4_assemble_kernel<0>, grid, 128, 0, nnz, d_src_ptr, d_src, d_conn, d_xy, d_ks, d_ms, d_cmat6, d_Kvals, d_Mvals);
  else if (kind == 1) EIGD_LAUNCH(q4_assemble_kernel<1>, grid, 128, 0, nnz, d_src_ptr, d_src, d_conn, d_xy, d_ks, d_ms, d_cmat6, d_Kvals, d_Mvals);
  else { eigd_set_error("q4_assemble: unknown kind %d", kind); return 1; }
  EIGD_CHECK_LAUNCH();
  return 0;
}

extern "C" int eigd_q4_quadforms(int kind, int nelems, const int* d_conn, const double* d_xy, const double* d_cmat6,
                                 const double* d_WA, const double* d_WB, const double* d_V, int N, int ldw,
                                 const double* d_dk, const double* d_dm, double sA, double sB, double* d_out) {
  if (nelems <= 0 || N <= 0) return 0;
  constexpr int G = 8;
  int grid = (int)(((int64_t)nelems * G + 255) / 256);
  if (kind == 0) EIGD_LAUNCH((q4_quadforms_kernel<0, G>), grid, 256, 0, nelems, d_conn, d_xy, d_cmat6, d_WA, d_WB, d_V, N, ldw, d_dk, d_dm, sA, sB, d_out);
  else if (kind == 1) EIGD_LAUNCH((q4_quadforms_kernel<1, G>), grid, 256, 0, nelems, d_conn, d_xy, d_cmat6, d_WA, d_WB, d_V, N, ldw, d_dk, d_dm, sA, sB, d_out);
  else { eigd_set_error("q4_quadforms: unknown kind %d", kind); return 1; }
  EIGD_CHECK_LAUNCH();
  return 0;
}

extern "C" int eigd_node_gather(int nnodes, const int* d_nptr, const int* d_nelem, const double* d_evals, double scale,
                                double* d_out) {
  if (nnodes <= 0) return 0;
  EIGD_LAUNCH(node_gather_kernel, (nnodes + 255) / 256, 256, 0, nnodes, d_nptr, d_nelem, d_evals, scale, d_out);
  EIGD_CHECK_LAUNCH();
  return 0;
}

extern "C" int eigd_dof_gather(int nnodes, int ncomp, int npe, const int* d_nptr, const int* d_nelem, const int* d_nlocal,
                               const double* d_due, double* d_out) {
  if (nnodes <= 0) return 0;
  const int grid = (nnodes + 255) / 256;
  if (ncomp == 2) EIGD_LAUNCH(dof_gather_kernel<2>, grid, 256, 0, nnodes, npe, d_nptr, d_nelem, d_nlocal, d_due, d_out);
  else if (ncomp == 3) EIGD_LAUNCH(dof_gather_kernel<3>, grid, 256, 0, nnodes, npe, d_nptr, d_nelem, d_nlocal, d_due, d_out);
  else { eigd_set_error("dof_gather: %d components per node not instantiated (2: Q4 plane stress, 3: H8)", ncomp); return 1; }
  EIGD_CHECK_LAUNCH();
  return 0;
}

// ---- smooth Heaviside projection of the filtered density (examples/node_filter.py:174-181, 193-203) ------------
// forward : out = (tanh(beta eta) + tanh(beta (rho - eta))) / (tanh(beta eta) + tanh(beta (1 - eta)))
// gradient: out = g * (beta / denom) / cosh(beta (rho - eta))^2          (rho = the filtered, unprojected field)
namespace {
__global__ void filter_project_kernel(int n, double beta, double eta, const double* __restrict__ rho,
                                      const double* __restrict__ g, double* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double denom = tanh(beta * eta) + tanh(beta * (1.0 - eta));
  const double t = beta * (rho[i] - eta);
  if (g) {
    const double c = cosh(t);
    out[i] = g[i] * (beta / denom) / (c * c);
  } else {
    out[i] = (tanh(beta * eta) + tanh(t)) / denom;
  }
}
}  // namespace

extern "C" int eigd_filter_project(int n, double beta, double eta, const double* d_rho, const double* d_g, double* d_out) {
  if (n <= 0) return 0;
  EIGD_LAUNCH(filter_project_kernel, (n + 255) / 256, 256, 0, n, beta, eta, d_rho, d_g, d_out);
  EIGD_CHECK_LAUNCH();
  return 0;
}

// ---- element density and material interpolation ----------------------------------------------
// rhoE[e] = 1/npe sum_a rho[conn[e, a]]        (examples/thermal.py:348-353, natural_frequency.py:399-404)
//   npe = 4 (Q4), 8 (H8) or 10 (T10) nodes per element
// law 0 (thermal.py:132,198,175-188,236-244): ks = k0((1-b) r^p + b), ms = c0((1-b) r + b)
// law 1 (natural_frequency.py:140-143,219-220 "simp"): ks = r^p + r0, ms = c0 r
// law 2 (RAMP, natural_frequency.py:142-143): ks = r/(1+q(1-r)) + r0, ms = c0 r
// par = {p or q, k0, c0, b or r0}
namespace {
__global__ void q4_material_kernel(int law, int nelems, int npe, const int* __restrict__ conn, const double* __restrict__ rho,
                                   double p0, double k0, double c0, double b, double* __restrict__ rhoE,
                                   double* __restrict__ ks, double* __restrict__ ms, double* __restrict__ dk,
                                   double* __restrict__ dm) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nelems) return;
  double r;
  if (conn) {
    const int* c = conn + (int64_t)npe * e;
    if (npe == 4)
      r = 0.25 * (rho[c[0]] + rho[c[1]] + rho[c[2]] + rho[c[3]]);
    else if (npe == 8)
      r = 0.125 * (rho[c[0]] + rho[c[1]] + rho[c[2]] + rho[c[3]] + rho[c[4]] + rho[c[5]] + rho[c[6]] + rho[c[7]]);
    else
      r = 0.1 * (rho[c[0]] + rho[c[1]] + rho[c[2]] + rho[c[3]] + rho[c[4]] + rho[c[5]] + rho[c[6]] + rho[c[7]] + rho[c[8]] +
                 rho[c[9]]);
    if (rhoE) rhoE[e] = r;
  } else {
    r = rho[e];
  }
  double vk, vm, gk, gm;
  if (law == 0) {
    vk = k0 * ((1.0 - b) * pow(r, p0) + b);
    gk = (1.0 - b) * k0 * p0 * pow(r, p0 - 1.0);
    vm = c0 * ((1.0 - b) * r + b);
    gm = (1.0 - b) * c0;
  } else if (law == 1) {
    vk = k0 * pow(r, p0) + b;
    gk = k0 * p0 * pow(r, p0 - 1.0);
    vm = c0 * r;
    gm = c0;
  } else {
    double den = 1.0 + p0 * (1.0 - r);
    vk = k0 * r / den + b;
    gk = k0 * (1.0 + p0) / (den * den);
    vm = c0 * r;
    gm = c0;
  }
  if (ks) ks[e] = vk;
  if (ms) ms[e] = vm;
  if (dk) dk[e] = gk;
  if (dm) dm[e] = gm;
}
}  // namespace

extern "C" int eigd_q4_material(int law, int nelems, int npe, const int* d_conn, const double* d_rho, const double* par4,
                                double* d_rhoE, double* d_ks, double* d_ms, double* d_dk, double* d_dm) {
  if (nelems <= 0) return 0;
  if (law < 0 || law > 2) { eigd_set_error("q4_material: unknown law %d", law); return 1; }
  if (npe != 4 && npe != 8 && npe != 10) {
    eigd_set_error("q4_material: %d nodes per element (4: Q4, 8: H8, 10: T10)", npe);
    return 1;
  }
  EIGD_LAUNCH(q4_material_kernel, (nelems + 255) / 256, 256, 0, law, nelems, npe, d_conn, d_rho, par4[0], par4[1], par4[2],
              par4[3], d_rhoE, d_ks, d_ms, d_dk, d_dm);
  EIGD_CHECK_LAUNCH();
  return 0;
}
