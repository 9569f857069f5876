// Device-resident shift-and-invert Lanczos recurrence: one C-ABI call runs the steps j0 .. j1-1 of a
// (restarted) Lanczos cycle without returning to the host -- solve, two classical Gram-Schmidt passes
// (DGKS), B-product, B-norm, normalisation -- so the Python layer only sequences restart cycles.
// Replaces the reverse-communication loop `params.iterate()` of reference eigd/arpack.py:438-442
// (ARPACK dsaupd / dsaitr: one OP application, one or two B-products and the CGS / DGKS
// orthogonalisation per step) and the per-step body of BasicLanczos.solve
// (eigd/eigenvector_derivatives.py:1496-1545).
//
// Storage: the bases V and BV = B V are (ncv + 1) x n row-major (one vector per contiguous row, leading
// dimension ld); w, h, g are work vectors; ab is 2 x ldab: row 0 receives alpha_j, row 1 beta_j^2.
#include "common.cuh"
#include "../../include/eigd_b200.h"

int eigd_basis_dots(int64_t n, int j, const double* V, int64_t ldv, const double* w, double* out, double* work);
int eigd_basis_axpy(int64_t n, int j, const double* V, int64_t ldv, const double* S, int lds, double alpha, double* w);
int eigd_csr_spmv_dot(int n, const int* indptr, const int* indices, const double* vals, const double* x, double* y,
                      double* out, double* work);

namespace {

// v_next = w / sqrt(beta2), bv_next /= sqrt(beta2), alpha_j = h_j + g_j (second Gram-Schmidt pass included)
__global__ void lanczos_finish_kernel(int64_t n, const double* __restrict__ w, const double* __restrict__ beta2,
                                      double* __restrict__ vnext, double* __restrict__ bvnext,
                                      const double* __restrict__ hj, const double* __restrict__ gj, double* __restrict__ alpha) {
  const double b2 = *beta2;
  const double s = 1.0 / sqrt(b2);
  if (blockIdx.x == 0 && threadIdx.x == 0) *alpha = *hj + *gj;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    vnext[i] = w[i] * s;
    bvnext[i] *= s;
  }
}

inline int ew_grid(int64_t n) {
  int64_t g = (n + 255) / 256;
  return (int)(g < 1 ? 1 : (g > 148 * 8 ? 148 * 8 : g));
}

}  // namespace

extern "C" int eigd_lanczos_extend(eigd_factor* f, int n, const int* d_b_indptr, const int* d_b_indices,
                                   const double* d_b_vals, double* d_V, double* d_BV, int64_t ld, int j0, int j1,
                                   double* d_w, double* d_h, double* d_g, double* d_ab, int ldab, double* d_work) {
  if (j1 <= j0) return 0;
  int rc;
  for (int j = j0; j < j1; ++j) {
    const double* bvj = d_BV + (int64_t)j * ld;
    // w = OP v_j = (A - sigma B)^{-1} (B v_j)
    if ((rc = eigd_factor_apply(f, bvj, 1, 1, d_w, 1, 1, 1))) return rc;
    // classical Gram-Schmidt against v_0 .. v_j in the B inner product, second pass unconditional (DGKS)
    if ((rc = eigd_basis_dots(n, j + 1, d_BV, ld, d_w, d_h, d_work))) return rc;
    if ((rc = eigd_basis_axpy(n, j + 1, d_V, ld, d_h, 1, -1.0, d_w))) return rc;
    if ((rc = eigd_basis_dots(n, j + 1, d_BV, ld, d_w, d_g, d_work))) return rc;
    if ((rc = eigd_basis_axpy(n, j + 1, d_V, ld, d_g, 1, -1.0, d_w))) return rc;
    // B-norm of the new direction and the next basis vector
    double* bvn = d_BV + (int64_t)(j + 1) * ld;
    if ((int64_t)(n + 63) / 64 <= eigd_gemm_tn_workspace(32, 32)) {
      if ((rc = eigd_csr_spmv_dot(n, d_b_indptr, d_b_indices, d_b_vals, d_w, bvn, d_ab + ldab + j, d_work))) return rc;
    } else {
      if ((rc = eigd_csr_spmm(n, d_b_indptr, d_b_indices, d_b_vals, d_w, 1, 1, bvn, 1, 1, 1, 1.0, 0.0))) return rc;
      if ((rc = eigd_basis_dots(n, 1, bvn, ld, d_w, d_ab + ldab + j, d_work))) return rc;
    }
    EIGD_LAUNCH(lanczos_finish_kernel, ew_grid(n), 256, 0, (int64_t)n, d_w, d_ab + ldab + j, d_V + (int64_t)(j + 1) * ld, bvn,
                d_h + j, d_g + j, d_ab + j);
    EIGD_CHECK_LAUNCH();
  }
  return 0;
}
