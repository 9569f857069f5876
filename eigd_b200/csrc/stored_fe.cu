// Finite-element operators on STORED unit element matrices (ne x ne per element, ne <= 32 element dofs), for
// models whose element matrices are an affine combination of a few geometry-only matrices with per-element
// design coefficients:  K_e = c1[e] E1_e + c3[e] E3_e  (flat shell: membrane + transverse shear ~ t, bending ~ t^3;
// mass: translation ~ t, rotary inertia ~ t^3).  With 180 GB of HBM the unit matrices of a 1M-DOF shell model
// (167k elements x 576 x 4 arrays = 3 GB) simply stay resident; per design only the coefficients change.  The H8
// and T10 elements (h8.cu, t10.cu) use them with one term per matrix: K_e = ks[e] K0_e, M_e = ms[e] M0_e.
//
// Replaces, for the CRM-like driver (reference examples/crm.py:122-142, 331-355), what TACS does on the host:
//   assembleMatType(STIFFNESS_MATRIX / MASS_MATRIX)            -> eigd_stored_assemble (gather form, no atomics)
//   addMatDVSensInnerProduct(w, v) per mode ("vector" form)    -> eigd_stored_quadform + eigd_segment_sum
// The per-component sums are warp-shuffle segmented reductions over elements sorted by component.
#include "common.cuh"
#include "../../include/eigd_b200.h"

namespace {

// vals[p] = sum over the sources s of CSR non-zero p of c1[e] * E1[s] + c3[e] * E3[s],  e = s / ne2
// (s = e * ne2 + a * ne + b: the flattened element-matrix order, as in eigd_q4_assemble); second pair (F1, F3, d1, d3)
// optional: a second matrix on the same pattern (the mass matrix) assembled in the same pass.  T3 = false: models
// without the t^3 terms (E3, c3, F3, d3 unused).
template <bool T3>
__global__ void __launch_bounds__(256)
stored_assemble_kernel(int64_t nnz, const int64_t* __restrict__ src_ptr, const int64_t* __restrict__ src, int ne2,
                       const double* __restrict__ E1, const double* __restrict__ E3, const double* __restrict__ c1,
                       const double* __restrict__ c3, double* __restrict__ vals, const double* __restrict__ F1,
                       const double* __restrict__ F3, const double* __restrict__ d1, const double* __restrict__ d3,
                       double* __restrict__ vals2) {
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < nnz; p += (int64_t)gridDim.x * blockDim.x) {
    double a = 0.0, b = 0.0;
    const int64_t s0 = src_ptr[p], s1 = src_ptr[p + 1];
    for (int64_t q = s0; q < s1; ++q) {
      const int64_t s = src[q];
      const int64_t e = s / ne2;
      a = fma(c1[e], E1[s], a);
      if (T3) a = fma(c3[e], E3[s], a);
      if (vals2) {
        b = fma(d1[e], F1[s], b);
        if (T3) b = fma(d3[e], F3[s], b);
      }
    }
    vals[p] = a;
    if (vals2) vals2[p] = b;
  }
}

// out[e] = sum_k sum_{a,b} W[dof(e,a), k] (c1[e] E1[e][a][b] + c3[e] E3[e][a][b]) V[dof(e,b), k]
// One warp per element: lane b holds column b of the combined element matrix in registers (coalesced loads of the rows),
// then loops over the modes; dof < 0 marks a constrained dof (contributes nothing).  W, V row-major (n, N), leading
// dimension ld.  NE = element dofs (<= 32).  T3 = false: no c3 E3 term.  TWO: a second term on the same gathered V,
//   out[e] = s1 * sum_k W_k^T (c1 E1 [+ c3 E3]) V_k + s2 * sum_k W2_k^T (d1 F1) V_k,
// both reduced together (the fused dA/dx, dB/dx form of the tensor derivative).
template <int NE, bool T3, bool TWO>
__global__ void __launch_bounds__(256)
stored_quadform_kernel(int nelems, const int* __restrict__ dofmap, const double* __restrict__ E1, const double* __restrict__ E3,
                       const double* __restrict__ c1, const double* __restrict__ c3, const double* __restrict__ W,
                       const double* __restrict__ V, int N, int64_t ld, double* __restrict__ out,
                       const double* __restrict__ F1, const double* __restrict__ d1, const double* __restrict__ W2, double s1,
                       double s2) {
  const int lane = threadIdx.x & 31;
  const int e = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (e >= nelems) return;
  const double a1 = c1[e], a3 = T3 ? c3[e] : 0.0;
  const double* p1 = E1 + (int64_t)e * NE * NE;
  const double* p3 = T3 ? E3 + (int64_t)e * NE * NE : nullptr;
  double col[NE];
#pragma unroll
  for (int a = 0; a < NE; ++a)
    col[a] = lane < NE ? (T3 ? fma(a3, __ldg(p3 + a * NE + lane), a1 * __ldg(p1 + a * NE + lane)) : a1 * __ldg(p1 + a * NE + lane))
                       : 0.0;
  double col2[TWO ? NE : 1];
  if (TWO) {
    const double b1 = d1[e];
    const double* q1 = F1 + (int64_t)e * NE * NE;
#pragma unroll
    for (int a = 0; a < NE; ++a) col2[a] = lane < NE ? b1 * __ldg(q1 + a * NE + lane) : 0.0;
  }
  const int mydof = lane < NE ? dofmap[(int64_t)e * NE + lane] : -1;
  double total = 0.0, total2 = 0.0;
  for (int k = 0; k < N; ++k) {
    const double wv = mydof >= 0 ? W[(int64_t)mydof * ld + k] : 0.0;      // w_a for a = lane
    const double vv = mydof >= 0 ? V[(int64_t)mydof * ld + k] : 0.0;      // v_b for b = lane
    double s = 0.0;
#pragma unroll
    for (int a = 0; a < NE; ++a) s = fma(__shfl_sync(0xffffffffu, wv, a), col[a], s);   // (w^T E)[b]
    total = fma(s, vv, total);
    if (TWO) {
      const double w2 = mydof >= 0 ? W2[(int64_t)mydof * ld + k] : 0.0;
      double t = 0.0;
#pragma unroll
      for (int a = 0; a < NE; ++a) t = fma(__shfl_sync(0xffffffffu, w2, a), col2[TWO ? a : 0], t);
      total2 = fma(t, vv, total2);
    }
  }
  if (TWO) total = fma(s2, total2, s1 * total);
  total = warp_sum(total);
  if (lane == 0) out[e] = total;
}

// out[c] = scale * sum_{i in [seg_ptr[c], seg_ptr[c+1])} x[perm[i]]   (elements sorted by component): one warp per segment
__global__ void __launch_bounds__(256)
segment_sum_kernel(int nseg, const int* __restrict__ seg_ptr, const int* __restrict__ perm, const double* __restrict__ x,
                   double scale, double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int c = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (c >= nseg) return;
  double s = 0.0;
  for (int i = seg_ptr[c] + lane; i < seg_ptr[c + 1]; i += 32) s += x[perm ? perm[i] : i];
  s = warp_sum(s);
  if (lane == 0) out[c] = scale * s;
}

}  // namespace

extern "C" int eigd_stored_assemble(int64_t nnz, const int64_t* d_src_ptr, const int64_t* d_src, int ne,
                                    const double* d_E1, const double* d_E3, const double* d_c1, const double* d_c3,
                                    double* d_vals, const double* d_F1, const double* d_F3, const double* d_d1,
                                    const double* d_d3, double* d_vals2) {
  if (nnz <= 0) return 0;
  int64_t g = (nnz + 255) / 256;
  int grid = (int)(g < 148 * 32 ? g : 148 * 32);
  const bool t3 = d_E3 != nullptr;
  if (t3 != (d_c3 != nullptr) || (d_vals2 && (t3 != (d_F3 != nullptr) || t3 != (d_d3 != nullptr)))) {
    eigd_set_error("stored_assemble: give all of the t^3 terms (E3, c3 and, with a second matrix, F3, d3) or none");
    return 1;
  }
  if (t3)
    EIGD_LAUNCH(stored_assemble_kernel<true>, grid, 256, 0, nnz, d_src_ptr, d_src, ne * ne, d_E1, d_E3, d_c1, d_c3, d_vals, d_F1,
                d_F3, d_d1, d_d3, d_vals2);
  else
    EIGD_LAUNCH(stored_assemble_kernel<false>, grid, 256, 0, nnz, d_src_ptr, d_src, ne * ne, d_E1, d_E3, d_c1, d_c3, d_vals, d_F1,
                d_F3, d_d1, d_d3, d_vals2);
  EIGD_CHECK_LAUNCH();
  return 0;
}

template <int NE>
static void stored_quadform_launch(int grid, bool t3, bool two, int nelems, const int* d_dofmap, const double* d_E1,
                                   const double* d_E3, const double* d_c1, const double* d_c3, const double* d_W,
                                   const double* d_V, int N, int64_t ld, double* d_out, const double* d_F1, const double* d_d1,
                                   const double* d_W2, double s1, double s2) {
  if (t3 && !two)
    EIGD_LAUNCH((stored_quadform_kernel<NE, true, false>), grid, 256, 0, nelems, d_dofmap, d_E1, d_E3, d_c1, d_c3, d_W, d_V, N, ld,
                d_out, d_F1, d_d1, d_W2, s1, s2);
  else if (t3)
    EIGD_LAUNCH((stored_quadform_kernel<NE, true, true>), grid, 256, 0, nelems, d_dofmap, d_E1, d_E3, d_c1, d_c3, d_W, d_V, N, ld,
                d_out, d_F1, d_d1, d_W2, s1, s2);
  else if (!two)
    EIGD_LAUNCH((stored_quadform_kernel<NE, false, false>), grid, 256, 0, nelems, d_dofmap, d_E1, d_E3, d_c1, d_c3, d_W, d_V, N, ld,
                d_out, d_F1, d_d1, d_W2, s1, s2);
  else
    EIGD_LAUNCH((stored_quadform_kernel<NE, false, true>), grid, 256, 0, nelems, d_dofmap, d_E1, d_E3, d_c1, d_c3, d_W, d_V, N, ld,
                d_out, d_F1, d_d1, d_W2, s1, s2);
}

extern "C" int eigd_stored_quadform(int nelems, int ne, const int* d_dofmap, const double* d_E1, const double* d_E3,
                                    const double* d_c1, const double* d_c3, const double* d_W, const double* d_V, int N,
                                    int64_t ld, double* d_out, const double* d_F1, const double* d_d1, const double* d_W2,
                                    double s1, double s2) {
  if (nelems <= 0) return 0;
  const bool t3 = d_E3 != nullptr, two = d_F1 != nullptr;
  if (t3 != (d_c3 != nullptr) || (two && (!d_d1 || !d_W2))) {
    eigd_set_error("stored_quadform: E3 needs c3, and a second term needs F1, d1 and W2");
    return 1;
  }
  const int grid = (int)(((int64_t)nelems * 32 + 255) / 256);
  switch (ne) {
    case 24: stored_quadform_launch<24>(grid, t3, two, nelems, d_dofmap, d_E1, d_E3, d_c1, d_c3, d_W, d_V, N, ld, d_out, d_F1, d_d1, d_W2, s1, s2); break;
    case 8: stored_quadform_launch<8>(grid, t3, two, nelems, d_dofmap, d_E1, d_E3, d_c1, d_c3, d_W, d_V, N, ld, d_out, d_F1, d_d1, d_W2, s1, s2); break;
    case 30: stored_quadform_launch<30>(grid, t3, two, nelems, d_dofmap, d_E1, d_E3, d_c1, d_c3, d_W, d_V, N, ld, d_out, d_F1, d_d1, d_W2, s1, s2); break;
    case 10: stored_quadform_launch<10>(grid, t3, two, nelems, d_dofmap, d_E1, d_E3, d_c1, d_c3, d_W, d_V, N, ld, d_out, d_F1, d_d1, d_W2, s1, s2); break;
    default:
      eigd_set_error("stored_quadform: element size %d not instantiated (24: shell Q4 and H8, 8: membrane Q4 and scalar H8, "
                     "30: T10, 10: scalar T10)", ne);
      return 7;
  }
  EIGD_CHECK_LAUNCH();
  return 0;
}

extern "C" int eigd_segment_sum(int nseg, const int* d_seg_ptr, const int* d_perm, const double* d_x, double scale, double* d_out) {
  if (nseg <= 0) return 0;
  const int grid = (int)(((int64_t)nseg * 32 + 255) / 256);
  EIGD_LAUNCH(segment_sum_kernel, grid, 256, 0, nseg, d_seg_ptr, d_perm, d_x, scale, d_out);
  EIGD_CHECK_LAUNCH();
  return 0;
}
