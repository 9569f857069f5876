/*
 * eigd_b200 -- C-ABI of the B200-native gradient path of smdogroup/eigd.
 *
 * The reference is pure Python (no FFI of its own); the drop-in boundary is the public
 * surface of `eigd/eigenvector_derivatives.py` + `eigd/arpack.py`.  This header declares
 * the entry points that sit directly beneath that surface.  Each group cites the reference
 * code whose arithmetic it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; `eigd_last_error()` gives
 *     a message for the last failure on the calling thread;
 *   - pointers named d_* are DEVICE pointers (fp64 / int32 unless said otherwise), all
 *     others are host pointers; no ownership ever passes across the boundary except for
 *     the opaque handles created/destroyed here;
 *   - dense multi-vectors are addressed as X[i*rs + c*cs] (row stride, column stride in
 *     elements), which covers both the reference's (n, N) row-major arrays
 *     (rs = N, cs = 1; eigd/eigenvector_derivatives.py:56-65) and Krylov bases stored one
 *     vector per row (rs = 1, cs = n);
 *   - all kernels are launched on the stream set with eigd_set_stream (default: stream 0).
 */
#ifndef EIGD_B200_H
#define EIGD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- library / context --------------------------------------------------------------- */
int eigd_version(void);
const char* eigd_last_error(void);
int eigd_device_count(int* count);
int eigd_set_stream(void* cuda_stream);
/* number of kernels this library has launched since load (bench.py "gpu_launches") */
int64_t eigd_launch_count(void);

/* ---- sparse products: replaces scipy `B @ x`, `A @ x` (csr_matvec[s]) used at
 *      eigd/eigenvector_derivatives.py:255-265,519,609,800-857,975-1010,1173-1252,1500 --- */
/* Y = alpha * A @ X + beta * Y,  A CSR (n rows), X and Y with (rs, cs) strides, k columns */
int eigd_csr_spmm(int n, const int* d_indptr, const int* d_indices, const double* d_vals,
                  const double* d_X, int64_t xrs, int64_t xcs,
                  double* d_Y, int64_t yrs, int64_t ycs, int k, double alpha, double beta);
/* out = a*va + b*vb on the value arrays of two matrices sharing one pattern
 * (K - sigma*M at examples/natural_frequency.py:338, Kr + sigma*Gr at examples/buckling.py:582) */
int eigd_axpby(int64_t len, double a, const double* d_x, double b, const double* d_y, double* d_out);

/* ---- tall-skinny dense kernels: replaces numpy `V.T @ X`, `U @ t`, `.dot`, axpy loops
 *      (eigd/eigenvector_derivatives.py:26-30,502,519,616-620,1254-1260,1529-1538,1648,1979) */
/* C[a*ldc + b] = sum_i X[i*xrs + a*xcs] * Y[i*yrs + b*ycs]; k1,k2 <= 64; workspace >= eigd_gemm_tn_workspace() doubles */
int64_t eigd_gemm_tn_workspace(int k1, int k2);
int eigd_gemm_tn(int64_t n, int k1, int k2, const double* d_X, int64_t xrs, int64_t xcs,
                 const double* d_Y, int64_t yrs, int64_t ycs, double* d_C, int ldc, double* d_work);
/* Y[i,b] = beta*Y[i,b] + alpha * sum_a X[i,a] * S[a*lds + b]; S on device; k1 <= 128, k2 <= 64 */
int eigd_gemm_nn(int64_t n, int k1, int k2, double alpha, const double* d_X, int64_t xrs, int64_t xcs,
                 const double* d_S, int lds, double beta, double* d_Y, int64_t yrs, int64_t ycs);
/* out[c] = sum_i X[i,c]*Y[i,c] (column-wise dots, k <= 64) */
int eigd_col_dot(int64_t n, int k, const double* d_X, int64_t xrs, int64_t xcs,
                 const double* d_Y, int64_t yrs, int64_t ycs, double* d_out, double* d_work);
/* Y[i,c] += sign * s[c] * X[i,c]   (s on device) */
int eigd_col_axpy(int64_t n, int k, double sign, const double* d_s, const double* d_X, int64_t xrs, int64_t xcs,
                  double* d_Y, int64_t yrs, int64_t ycs);
/* Modified Gram-Schmidt sweep of the k columns of w (n x k, row-major, contiguous) against j stored blocks of the same
 * layout, in the order given: h_t[c] = sum_i w[i,c] W_t[i,c]; w[:,c] -= h_t[c] W_t[:,c]; h_t is written to H[t] (k
 * doubles on the device).  W and H are HOST arrays of j device pointers.  One cooperative launch per 64 blocks.
 * Replaces the dot / axpy loops of eigd/eigenvector_derivatives.py:1254-1257 (sibk) and :1012-1014 (pgmres).
 * d_work: the eigd_gemm_tn_workspace buffer.  k <= 64. */
int eigd_mgs_sweep(int64_t n, int k, int j, const double* const* W, double* const* H, double* d_w, double* d_work);
/* X[i,c] *= s[c]  (mode 0)   or   X[i,c] /= s[c]  (mode 1)   or X[i,c] /= sqrt(s[c]) (mode 2);
 * modes 3 / 4 are the zero-safe forms of 2 / 1 (a zero scale leaves a zero column) */
int eigd_col_scale(int64_t n, int k, int mode, const double* d_s, double* d_X, int64_t xrs, int64_t xcs);
/* Y[i,c] = X[i,c] (strided copy / transpose) */
int eigd_copy2d(int64_t n, int k, const double* d_X, int64_t xrs, int64_t xcs, double* d_Y, int64_t yrs, int64_t ycs);

/* ---- sparse LDL^T of the shifted matrix: replaces scipy.sparse.linalg.splu + SuperLU.solve
 *      behind SpLuOperator (eigd/eigenvector_derivatives.py:11-23) ------------------------ */
typedef struct eigd_symbolic eigd_symbolic;
typedef struct eigd_factor eigd_factor;

/* Symbolic analysis of a structurally symmetric CSR pattern (host arrays).
 * coords: optional (n_nodes x dim) node coordinates for geometric nested dissection, with
 * dof_per_node consecutive rows per node (NULL -> graph-based dissection).
 * opts: optional int[8] {leaf_cols, max_super_cols, nd_leaf, relax, 0...}; NULL -> defaults. */
int eigd_symbolic_create(int n, const int* indptr, const int* indices,
                         const double* coords, int dim, int dof_per_node,
                         const int* opts, eigd_symbolic** out);
void eigd_symbolic_destroy(eigd_symbolic* s);
/* scalar queries: what = 0 n, 1 nsuper, 2 nlevels, 3 nnz(L) (strict lower, dense fronts),
 * 4 front storage doubles, 5 sum of front sizes, 6 max front size, 7 max supernode cols,
 * 8 flops of the factorisation, 9 nnz of exact (unrelaxed) L, 10 doubles of the pooled front workspace
 * (eigd_factor_numeric_pool) */
int64_t eigd_symbolic_query(const eigd_symbolic* s, int what);
/* array getters (host copies): which = 0 perm[n] (new->old), 1 etree parent[n], 2 sn_first[nsuper+1],
 * 3 sn_rowptr[nsuper+1], 4 sn_rows[...], 5 sn_parent[nsuper], 6 sn_level[nsuper],
 * 7 front_off[nsuper+1], 8 rel[...] (aligned with sn_rows), 9 colcount[n], 10 level_ptr[nlevels+1],
 * 11 level_sn[nsuper], 12 pool_off[nsuper] (offset of every front in the pooled front workspace: front k is live
 * from level sn_level[k] through sn_level[sn_parent[k]], and fronts live at one level never overlap).
 * Returns the element count; copies min(count, cap) int64 values. */
int64_t eigd_symbolic_get(const eigd_symbolic* s, int which, int64_t* out, int64_t cap);
/* assembly map nz -> slot in front storage (or -1), computed by host code */
int eigd_symbolic_assembly_map_host(const eigd_symbolic* s, int n, const int* indptr, const int* indices, int64_t* out_map);
/* the same map computed by the CUDA integer kernel (device CSR in, device map out) */
int eigd_symbolic_assembly_map_device(eigd_symbolic* s, int n, const int* d_indptr, const int* d_indices, int64_t* d_map);

/* inspection of the host-built plan of the persistent solve kernel (tests): which = 0 soff[nsuper+1],
 * 1 ovf_row[sum_front] (-1 or offset into the overflow list), 2 overflow list (count, sources...),
 * 3 tile records (8 values each: first, nc, nb, tile, soff, w_off, row_off, link), 4 phases (5 values
 * each: dir, ws, ntiles, level, tile_off; ws == 0 marks a subtree phase), 5 subtree tables (slot x local
 * level -> first tile), 6 owning slot of every supernode (-1 above the cut), 7 {cut_level, nslots, nfwd},
 * 8 child slab of every supernode (0, 1, 2 = overflow, 255 = root).
 * target_warps = resident warps the level phases are balanced for, nslots = CTA slots of the subtree
 * phases, cut = -2 automatic / -1 no subtree phases / >= 0 forced cut level.
 * Returns the element count; copies min(count, cap) values. */
int64_t eigd_solve_plan_get(const eigd_symbolic* s, int target_warps, int nslots, int cut, int which, int64_t* out,
                            int64_t cap);

int eigd_factor_create(eigd_symbolic* s, int max_rhs, eigd_factor** out);
/* same, with every device array carved out of a caller-owned buffer of eigd_factor_workspace_bytes()
 * bytes (a torch tensor, so that the caching allocator recycles it: no cudaMalloc / cudaFree per design) */
int64_t eigd_factor_workspace_bytes(eigd_symbolic* s, int max_rhs);
int eigd_factor_create_in(eigd_symbolic* s, int max_rhs, void* d_workspace, int64_t workspace_bytes, eigd_factor** out);
/* the same two with a choice of front memory: fronts = 0 resident (as above: one f x f front per supernode in the
 * workspace, kept for the factor's life), 1 pooled (no fronts in the workspace: every eigd_factor_numeric_pool call
 * borrows a pool of eigd_symbolic_query(s, 10) doubles from the caller, so factors can take turns on one pool).  The
 * factor is the same bit for bit in both modes.  Any other mode fails. */
int64_t eigd_factor_workspace_bytes_fronts(eigd_symbolic* s, int max_rhs, int fronts);
int eigd_factor_create_in_fronts(eigd_symbolic* s, int max_rhs, int fronts, void* d_workspace, int64_t workspace_bytes,
                                 eigd_factor** out);
void eigd_factor_destroy(eigd_factor* f);
/* measured FP64 tensor-pipe (DMMA, mma.sync.m8n8k4.f64) peak of the current device in TFLOP/s: register-resident
 * micro-benchmark on all SMs, best of `reps` launches of `iters` x 8 MMAs per warp (denominator of bench.py's
 * roofline_fp64_tensor) */
int eigd_dmma_peak(int iters, int reps, double* tflops_out);
/* numeric factorisation from device CSR values + device assembly map (resident fronts only) */
int eigd_factor_numeric(eigd_factor* f, int64_t nnz, const double* d_vals, const int64_t* d_map);
/* the same for a factor with pooled fronts.  d_ent: int32 pairs (CSR index p, slot of entry p inside its front,
 * i.e. assembly map[p] - front_off[k]) of every mapped entry, grouped by front and sorted by slot inside a front;
 * d_seg[nsuper + 1] (int64): the pairs of front k are d_ent[2 d_seg[k] .. 2 d_seg[k + 1]).  d_pool: a 256-byte
 * aligned device buffer of pool_bytes >= 8 * eigd_symbolic_query(s, 10) bytes, used only until the kernels queued by
 * this call have run (returns 3 when it is smaller). */
int eigd_factor_numeric_pool(eigd_factor* f, int64_t nnz, const double* d_vals, const int64_t* d_seg, const int* d_ent,
                             void* d_pool, int64_t pool_bytes);
/* info[0] = #negative pivots (inertia), info[1] = #perturbed pivots, info[2] = #non-finite */
int eigd_factor_info(eigd_factor* f, int64_t* info3);
/* pivoting of the following eigd_factor_numeric calls: 0 = static (default; tiny pivots perturbed to +-1e-11 max|A|),
 * 1 = restricted Bunch-Kaufman (1x1 / 1x1 interchanged / 2x2 pivots chosen inside every 32-column pivot block,
 * 2x2 blocks rotated to diagonal form; tiny pivots still perturbed and counted).  Returns 1 for another mode. */
int eigd_factor_set_pivoting(eigd_factor* f, int mode);
/* out[0] = #2x2 pivots, out[1] = #row/column interchanges of the last restricted Bunch-Kaufman factorisation
 * (0, 0 for a static one) */
int eigd_factor_pivot_counts(eigd_factor* f, int64_t* out2);
/* X = (L D L^T)^{-1} B in the original ordering; k columns, (rs, cs) strides; X may alias B */
int eigd_factor_solve(eigd_factor* f, const double* d_B, int64_t brs, int64_t bcs,
                      double* d_X, int64_t xrs, int64_t xcs, int k);
/* iterative refinement of eigd_factor_apply: `steps` rounds of x += F (b - A x) against the device CSR A (the
 * factorised matrix; may be NULL when steps == 0), with d_work >= 2 * n * work_cols doubles of scratch (may be NULL when
 * work_cols == 0).  Both stay owned by the caller and must outlive their registration.  A new factor has steps = 0. */
int eigd_factor_set_refinement(eigd_factor* f, int steps, const int* d_indptr, const int* d_indices, const double* d_vals,
                               double* d_work, int work_cols);
/* X = A^{-1} B as the operator applies it: eigd_factor_solve followed by the registered refinement steps, over all k
 * columns; X may alias B.  Fails when the refinement depth is not 0 and k exceeds the registered work_cols. */
int eigd_factor_apply(eigd_factor* f, const double* d_B, int64_t brs, int64_t bcs,
                      double* d_X, int64_t xrs, int64_t xcs, int k);
/* live timing of every solve launch between begin and end (CUDA events on the launching stream, used by
 * bench.py for the roofline of the dominant kernel): calls_by_k / ms_by_k have 33 entries, index = number
 * of right-hand sides of the launch */
int eigd_solve_timing_begin(void);
int eigd_solve_timing_end(int64_t* calls_by_k, double* ms_by_k);
/* developer profiling of the persistent solve kernel: d_buf (device, (nphases + 1) x uint64) receives the
 * %globaltimer of CTA 0 at kernel start and after every phase of the following solves; NULL switches it off */
int eigd_solve_set_phase_times(void* d_buf);
/* developer profiling: d_buf (device, 8 x nphases int64) receives clock64 stamps of CTA 0 / warp 0 inside its first
 * tile of every level phase (start, dependencies met, product done, partials reduced, stored, signalled) */
int eigd_solve_set_trace(void* d_buf);
/* developer profiling: d_buf = 4 * nphases * (number of SMs) u64, %globaltimer of every CTA's first tile of every level
 * phase of the pipelined level kernel (start, slot there, dependencies complete, signalled); NULL switches it off */
int eigd_solve_set_skew(void* d_buf);
int eigd_solve_num_phases(const eigd_factor* f);
int64_t eigd_factor_bytes(const eigd_factor* f);

/* ---- device-resident Lanczos recurrence: replaces the reverse-communication loop around ARPACK dsaupd
 *      (eigd/arpack.py:438-442) and the step body of BasicLanczos.solve
 *      (eigd/eigenvector_derivatives.py:1496-1545).  Runs steps j0 .. j1-1 without returning to the host:
 *      w = factor^{-1} BV[j] (eigd_factor_apply: the refinement registered with the factor, whose
 *      scratch must hold one column), two classical Gram-Schmidt passes against V[0..j] in the B inner
 *      product, BV[j+1] = B w, beta_j^2 = w . B w, V[j+1] = w / beta_j, BV[j+1] /= beta_j.
 *      V, BV: (ncv + 1) x n row-major with leading dimension ld; w, h, g: n, ncv + 1, ncv + 1 doubles;
 *      ab: 2 x ldab, row 0 <- alpha_j, row 1 <- beta_j^2; work >= eigd_gemm_tn_workspace() doubles. ------- */
int eigd_lanczos_extend(eigd_factor* f, int n, const int* d_b_indptr, const int* d_b_indices,
                        const double* d_b_vals, double* d_V, double* d_BV, int64_t ld, int j0, int j1,
                        double* d_w, double* d_h, double* d_g, double* d_ab, int ldab, double* d_work);

/* ---- operators on stored unit element matrices (csrc/stored_fe.cu): the CRM-like shell driver, replacing what TACS
 *      does on the host in reference examples/crm.py:122-142 (assembleMatType) and :331-355 (addMatDVSensInnerProduct,
 *      the per-mode "vector" derivative form).  Element matrices K_e = c1[e] E1_e + c3[e] E3_e, ne x ne row-major,
 *      ne element dofs.  Assembly is gather-form through the (element, a, b) -> CSR source lists of
 *      eigd_q4_assemble; a second matrix on the same pattern (F1, F3, d1, d3 -> vals2) is optional (NULL), and so
 *      are the t^3 terms (E3, c3, F3, d3 all NULL: K_e = c1[e] E1_e, the H8 solid). ---- */
int eigd_stored_assemble(int64_t nnz, const int64_t* d_src_ptr, const int64_t* d_src, int ne, const double* d_E1,
                         const double* d_E3, const double* d_c1, const double* d_c3, double* d_vals, const double* d_F1,
                         const double* d_F3, const double* d_d1, const double* d_d3, double* d_vals2);
/* out[e] = sum_k W[dof(e,:), k]^T (c1[e] E1_e + c3[e] E3_e) V[dof(e,:), k]; dofmap (nelems x ne, -1 = constrained);
 * W, V row-major (n, N) with leading dimension ld; ne in {8, 24}; E3 and c3 may both be NULL.  With a second term
 * (F1, d1, W2 non-NULL; W2 shares the layout of W and V) both are evaluated in the same pass over V:
 *   out[e] = s1 * sum_k W_k^T (c1[e] E1_e + c3[e] E3_e) V_k + s2 * sum_k W2_k^T (d1[e] F1_e) V_k
 * (s1, s2 are ignored without it). */
int eigd_stored_quadform(int nelems, int ne, const int* d_dofmap, const double* d_E1, const double* d_E3, const double* d_c1,
                         const double* d_c3, const double* d_W, const double* d_V, int N, int64_t ld, double* d_out,
                         const double* d_F1, const double* d_d1, const double* d_W2, double s1, double s2);
/* out[c] = scale * sum_{i in [seg_ptr[c], seg_ptr[c+1])} x[perm[i]] (perm NULL: identity): warp-shuffle segmented sum */
int eigd_segment_sum(int nseg, const int* d_seg_ptr, const int* d_perm, const double* d_x, double scale, double* d_out);

/* ---- BLOCK version of the recurrence (block size P = 2 .. 4; csrc/block_krylov.cu): one call runs the block steps
 *      j = j0, j0 + P, ... < ncv of a restart cycle on the device.  V, BV: (ncv + P) x n row-major (leading dimension
 *      ld) holding m0 >= j0 + P B-orthonormal vectors on entry and ncv + P on exit.  Per step s the P x P diagonal
 *      block (H1 + H2)[j : j + P] goes to Ablk[s] and the sub-diagonal block R (W = V_new R) to Rblk[s] (row-major);
 *      a rank-deficient block (breakdown) is flagged by NaNs in Rblk.  H1, H2: (ncv + P) * P doubles; scratch: 3 P^2;
 *      work >= eigd_gemm_tn_workspace().  The P-column solves are eigd_factor_apply: the refinement
 *      registered with the factor, whose scratch must hold P columns. -------------------------------------------- */
int eigd_block_lanczos_extend(eigd_factor* f, int n, int P, const int* d_b_indptr, const int* d_b_indices,
                              const double* d_b_vals, double* d_V, double* d_BV, int64_t ld, int j0, int m0, int ncv,
                              double* d_Ablk, double* d_Rblk, double* d_H1, double* d_H2, double* d_scratch,
                              double* d_work);
/* B-orthonormalise the P start vectors V[0:P] (rows) in place and set BV[0:P] = B V[0:P]; scratch: 3 P^2 doubles */
int eigd_block_lanczos_start(int n, int P, const int* d_b_indptr, const int* d_b_indices, const double* d_b_vals,
                             double* d_V, double* d_BV, int64_t ld, double* d_scratch, double* d_work);

/* ---- element kernels: replaces the numpy einsum callbacks and assembly in
 *      examples/thermal.py:126-246, examples/natural_frequency.py:134-284 ------------------ */
/* kind: 0 = thermal Q4 (1 dof/node), 1 = plane-stress Q4 (2 dof/node), ne = 4*dof.
 * Gather-form assembly (deterministic, no atomics): CSR non-zero p receives the sum of its
 * sources d_src[d_src_ptr[p] .. d_src_ptr[p+1]), each encoded as e*ne*ne + a*ne + b (the
 * flattened `Ke.flatten()` order of examples/thermal.py:79-92, natural_frequency.py:90-104).
 * ks[e], ms[e]: per-element penalised material factors. cmat6 = C0 {c00,c01,c02,c11,c12,c22}
 * (device, may be NULL for kind 0).  d_Kvals / d_Mvals may be NULL. */
int eigd_q4_assemble(int kind, int nelems, const int* d_conn, const double* d_xy,
                     const double* d_ks, const double* d_ms, const double* d_cmat6,
                     const int64_t* d_src_ptr, const int64_t* d_src, int64_t nnz,
                     double* d_Kvals, double* d_Mvals);
/* out[e] += sA * dk[e] * sum_k wA_e^T Ke1 v_e  -  sB * dm[e] * sum_k wB_e^T Me1 v_e  per element,
 * Ke1 / Me1 the unit-material element matrices, dk / dm the penalisation derivatives (NULL -> 1).
 * WA, WB, V are (ndof, N) row-major with leading dimension ldw; WA or WB may be NULL. */
int eigd_q4_quadforms(int kind, int nelems, const int* d_conn, const double* d_xy, const double* d_cmat6,
                      const double* d_WA, const double* d_WB, const double* d_V, int N, int ldw,
                      const double* d_dk, const double* d_dm, double sA, double sB, double* d_out);
/* Element density rhoE[e] = 1/npe sum_a rho[conn[e,a]], npe = 4 (Q4), 8 (H8) or 10 (T10) nodes per element (d_conn NULL:
 * d_rho is already per element) and the
 * penalised material factors / derivatives of the examples (thermal.py:132,175-188,198,236-244;
 * natural_frequency.py:140-143,198-201,219-220).  law 0 thermal SIMP, 1 structural SIMP, 2 RAMP;
 * par4 = {p or q, k0, c0, beta or rho0} (host).  Any output may be NULL. */
int eigd_q4_material(int law, int nelems, int npe, const int* d_conn, const double* d_rho, const double* par4,
                     double* d_rhoE, double* d_ks, double* d_ms, double* d_dk, double* d_dm);
/* ---- 3-D solid (csrc/h8.cu): unit element matrices of the trilinear hexahedron on the 2x2x2 Gauss rule, once per
 *      mesh.  conn (nelems, 8): nodes 0-3 counter-clockwise on the zeta = -1 face, 4-7 above them; X (nnodes, 3).
 *      K0, M0: (nelems, 24, 24) row-major, dof order node-major (u_x, u_y, u_z);
 *      K0_e = sum_q detJ B^T C(E, nu) B, M0_e = density sum_q detJ (N N^T (x) I_3). */
int eigd_h8_element_matrices(int nelems, const int* d_conn, const double* d_X, double E, double nu, double density,
                             double* d_K0, double* d_M0);
/* Scalar (heat conduction) H8, one dof per node in node order (fe.element_dofs(conn, 1)), same element and rule:
 * K0, M0 (nelems, 8, 8) row-major, K0_e = sum_q detJ grad N_a . grad N_b, M0_e = sum_q detJ N_a N_b (unit material;
 * M0 is bitwise the scalar block of eigd_h8_element_matrices' M0 at density 1). */
int eigd_h8_thermal_element_matrices(int nelems, const int* d_conn, const double* d_X, double* d_K0, double* d_M0);
/* ---- quadratic tetrahedra (csrc/t10.cu): unit element matrices on the 14-point degree-5 rule, once per mesh.
 *      conn (nelems, 10), VTK quadratic-tetra order: corners 0-3 (positive volume), then the midside nodes of the edges
 *      (0,1), (1,2), (2,0), (0,3), (1,3), (2,3); X (nnodes, 3).  Solid: K0, M0 (nelems, 30, 30) row-major, dof order
 *      node-major (u_x, u_y, u_z); K0_e = sum_q w_q detJ B^T C(E, nu) B, M0_e = density sum_q w_q detJ (N N^T (x) I_3). */
int eigd_t10_element_matrices(int nelems, const int* d_conn, const double* d_X, double E, double nu, double density,
                              double* d_K0, double* d_M0);
/* Scalar (heat conduction) T10, one dof per node in node order: K0, M0 (nelems, 10, 10) row-major,
 * K0_e = sum_q w_q detJ grad N_a . grad N_b, M0_e = sum_q w_q detJ N_a N_b (M0 is bitwise the scalar block of
 * eigd_t10_element_matrices' M0 at density 1). */
int eigd_t10_thermal_element_matrices(int nelems, const int* d_conn, const double* d_X, double* d_K0, double* d_M0);
/* node_out[v] = scale * sum_{e in adj(v)} e_vals[e]   (gather form of np.add.at, thermal.py:612-615) */
int eigd_node_gather(int nnodes, const int* d_nptr, const int* d_nelem, const double* d_evals, double scale, double* d_out);
/* out[ncomp v + i] = sum_{e around v} due[e][ncomp local + i], due (nelems, npe * ncomp), local = d_nlocal (the node's
 * index inside each adjacent element): the dof scatter np.add.at of examples/buckling.py:318-320 in gather form, for
 * the element terms of eigd_q4_gderiv (ncomp 2, npe 4) and eigd_h8_gderiv_u (ncomp 3, npe 8) */
int eigd_dof_gather(int nnodes, int ncomp, int npe, const int* d_nptr, const int* d_nelem, const int* d_nlocal,
                    const double* d_due, double* d_out);

/* tanh projection of the filtered density (examples/node_filter.py:174-181) and its gradient factor (:193-203):
 * d_g == NULL: out = projected rho; otherwise out = g * d(projection)/d(rho) evaluated at the UNPROJECTED rho */
int eigd_filter_project(int n, double beta, double eta, const double* d_rho, const double* d_g, double* d_out);

/* ---- linearised buckling (examples/buckling.py): stress stiffness G(u, x) and its sensitivities ---------
 * All vectors are in the FULL dof numbering (2 dof per node); eigd_expand_rows / eigd_reduce_rows are the
 * Dirichlet maps full_vector / reduce_vector (examples/buckling.py:499-518). */
/* sdet[e][q][i] = detJ_q ks[e] (C0 Be(q) u_e)_i, q = 4 Gauss points, i = 3 stress components (:241-247) */
int eigd_q4_stress(int nelems, const int* d_conn, const double* d_xy, const double* d_cmat6, const double* d_ks,
                   const double* d_u, double* d_sdet);
/* gather-form assembly of G through the same (element, a, b) -> CSR source lists as K (:249-255) */
int eigd_q4_assemble_geometric(int nelems, const int* d_conn, const double* d_xy, const double* d_sdet,
                               const int64_t* d_src_ptr, const int64_t* d_src, int64_t nnz, double* d_Gvals);
/* fused sensitivities of sum_k w_k^T G(u, x) v_k: out_rho[e] += sx * dks[e] * (...) (:324-343, per element, before
 * the node scatter) and due[e][8] = ks[e] * (...) (:312-322, before the dof scatter); either output may be NULL.
 * W, V: (2*nnodes, N) row-major with leading dimension ldw. */
int eigd_q4_gderiv(int nelems, const int* d_conn, const double* d_xy, const double* d_cmat6, const double* d_W,
                   const double* d_V, int N, int ldw, const double* d_ks, const double* d_dks, const double* d_u,
                   double sx, double* d_out_rho, double* d_due);
/* ---- linearised buckling of the 3-D solid (csrc/h8_buckling.cu), H8 elements as eigd_h8_element_matrices.
 *      dofmap (nelems, 24): element dof (node-major u_x, u_y, u_z) -> row of u, W and V; -1 = constrained (zero).
 *      Voigt order (xx, yy, zz, yz, xz, xy), engineering shear; C = C(E, nu) of K0. ---- */
/* per design: stress[e][q][6] = kg[e] C B_q u_e (NULL: not written) and the unit stress stiffness
 * G0[e] (24 x 24 row-major) = [delta_ij sum_q detJ_q gradN_a^T S_q gradN_b], S_q the 3 x 3 form of C B_q u_e */
int eigd_h8_stress_stiffness(int nelems, const int* d_conn, const double* d_X, double E, double nu, const double* d_kg,
                             const int* d_dofmap, const double* d_u, double* d_stress, double* d_G0);
/* due[e][24] = kg[e] sum_q detJ_q B_q^T C h_q, h_q = sum_k sum_i Voigt(grad w_{i,k} (x) grad v_{i,k}) with both shear
 * products: d/du_e of sum_k w_k^T G(u) v_k.  W, V row-major with leading dimension ld, N columns. */
int eigd_h8_gderiv_u(int nelems, const int* d_conn, const double* d_X, double E, double nu, const double* d_kg,
                     const int* d_dofmap, const double* d_W, const double* d_V, int N, int64_t ld, double* d_due);
/* full[idx[i], :] = red[i, :] and red[i, :] = full[idx[i], :], k columns, row-major */
int eigd_expand_rows(int64_t nr, int k, const int* d_idx, const double* d_red, double* d_full);
int eigd_reduce_rows(int64_t nr, int k, const int* d_idx, const double* d_full, double* d_red);

#ifdef __cplusplus
}
#endif
#endif
