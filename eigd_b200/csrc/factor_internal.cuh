// Internal declarations shared by factor.cu (device mirror of the symbolic analysis + numeric
// LDL^T + solve panels) and solve.cu (persistent multi-RHS triangular solve).
#pragma once
#include "common.cuh"
#include "solve_plan.hpp"
#include "symbolic.hpp"

#include <vector>

constexpr int NB = 32;        // pivot block width
constexpr int TRSM_ROWS = 128;
constexpr int UPD_TILE = 64;
constexpr int EA_TILE = 32;
constexpr int POOL_CHUNK = 16384;   // doubles of a front zeroed and assembled by one CTA (pooled fronts)

struct SymDev {
  int n, nsuper;
  int *perm, *iperm, *col2sn;
  int* sn_first;
  int64_t* sn_rowptr;
  int* sn_rows;
  int* rel;
  int64_t* front_off;
  int64_t* w_off;
  int64_t* linv_off;
  int64_t* soff;      // solve-panel offsets (prefix of f * nc)
  int64_t* xoff;      // full-inverse offsets (prefix of nc * nc)
  int* sn_parent;
  int *child_ptr, *child_idx;
  int *th_f, *th_b;   // per supernode: tile height of the tile-major S / S^T solve panel (solve_plan.hpp), 0 = column-major
};

struct Launch {
  int kind;      // 0 extend-add, 1 diag, 2 trsm, 3 update, 4 inverse-init, 5 inverse GEMM (C A^-1), 6 inverse GEMM (-B^-1 T),
                 // 7 panel build, 8 zero + assemble fronts (pooled fronts)
  int kb;        // pivot block index (kinds 1-3) / doubling stage (kinds 5, 6)
  int64_t off;   // offset into the task array (int2 entries)
  int count;
};

// device copy of the solve plan (solve_plan.hpp)
struct SolvePlanDev {
  TileRec* tiles = nullptr;
  TileDep* deps = nullptr;      // parallel to tiles
  int* dep_ovf = nullptr;
  PhaseRec* phases = nullptr;
  int* ovf_row = nullptr;
  int* ovf = nullptr;
  int* sub_ptr = nullptr;
  int nphases = 0;
  int grid = 0;               // CTAs of the cooperative launch
  std::vector<PhaseRec> host_phases;
};

struct SymDevHolder {
  SymDev d;
  std::vector<void*> allocs;
  int2* tasks = nullptr;
  std::vector<Launch> factor_plan;
  int64_t linv_total = 0;     // 32x32 diagonal-block inverses
  int64_t xinv_total = 0;     // full nc x nc inverses of the unit-lower pivot blocks
  int64_t panel_total = 0;    // sum f * nc
  SolvePlanDev solve;
  // pooled fronts (build_pool_plan, on first use)
  int64_t* pool_off = nullptr;        // device copy of eigd_symbolic::pool_off
  int2* pool_tasks = nullptr;
  std::vector<Launch> pool_plan;
};

struct eigd_factor {
  eigd_symbolic* sym = nullptr;
  SymDevHolder* h = nullptr;
  int max_rhs = 1;
  double* fronts = nullptr;   // f x f frontal matrices (factorisation workspace); NULL with pooled fronts
  bool pooled = false;        // fronts borrowed per eigd_factor_numeric_pool call (pool_off layout) instead of resident
  double* linv = nullptr;     // inverses of the 32x32 unit-lower diagonal blocks (pivoted: of the dense blocks M, see
                              // diag_factor_bk_kernel)
  double* xinv = nullptr;     // full inverse of every L11 (nc x nc, column-major)
  double* xtmp = nullptr;     // scratch of the same size (recursive-doubling products)
  double* sfwd = nullptr;     // solve panels S = [L11^-1 ; -L21 L11^-1], f x nc: column-major below the cut of the solve
                              // plan, tile-major above it (solve_plan.hpp)
  double* sbwd = nullptr;     // S^T, nc x f, likewise
  double* dval = nullptr;
  double* dinv = nullptr;
  double* wbuf = nullptr;     // forward-sweep update vectors: 3 slabs x kmax planes x (sum of front sizes)
  double* bperm = nullptr;    // right-hand side in the permuted ordering, n x k
  double* ybuf = nullptr;     // D^-1 L^-1 b in the permuted ordering, n x k
  double* xperm = nullptr;    // solution in the permuted ordering, n x k
  unsigned long long* amax = nullptr;   // 1 value
  unsigned long long* info = nullptr;   // 4 values
  unsigned long long* barrier = nullptr;  // arrival counter of the grid barrier (monotone)
  unsigned long long bar_base = 0;        // arrivals issued so far (host mirror)
  unsigned* cnt = nullptr;                // per-front completion counters of the solve (2 per supernode), monotone
  unsigned epoch = 0;                     // cooperative solve launches issued so far (host mirror)
  double piv_tol = 1e-11;
  int pivoting = 0;                       // 0 static pivots, 1 restricted Bunch-Kaufman (eigd_factor_set_pivoting)
  struct {                                // iterative refinement of eigd_factor_apply (eigd_factor_set_refinement)
    int steps, cols;                      // depth; right-hand sides the scratch holds
    const int *indptr, *indices;          // the caller's device CSR of the factorised matrix
    const double* vals;
    double* work;                         // the caller's scratch, 2 x n x cols doubles
  } refine = {};
  int64_t bytes = 0;
  char* base = nullptr;
  bool owns = true;
};

int build_symdev(eigd_symbolic* S);
int build_pool_plan(eigd_symbolic* S);
int build_solve_plan_dev(eigd_symbolic* S, SymDevHolder* h);
void free_solve_plan_dev(SymDevHolder* h);
