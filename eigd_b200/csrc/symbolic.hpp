// Host-side symbolic analysis for the supernodal multifrontal LDL^T.
// No reference counterpart: the reference hides this step inside SuperLU (scipy splu,
// eigd/eigenvector_derivatives.py:13).  See DESIGN.md "Symbolic analysis".
#pragma once
#include <cstdint>
#include <vector>

struct eigd_symbolic {
  int n = 0;
  // perm[new] = old, iperm[old] = new
  std::vector<int> perm, iperm;
  std::vector<int> parent;    // column elimination tree (permuted, postordered)
  std::vector<int> colcount;  // strict-lower column counts of the exact factor
  int nsuper = 0;
  std::vector<int> sn_first;        // nsuper+1
  std::vector<int> col2sn;          // n
  std::vector<int64_t> sn_rowptr;   // nsuper+1, offsets into sn_rows / rel
  std::vector<int> sn_rows;         // below-diagonal rows of each front (permuted, ascending)
  std::vector<int> rel;             // position of each of those rows in the parent's front
  std::vector<int> sn_parent;       // supernodal elimination tree
  std::vector<int> sn_level;        // height above the leaves
  std::vector<int64_t> front_off;   // nsuper+1, offsets (doubles) of the f x f fronts
  std::vector<int64_t> pool_off;    // nsuper, offsets (doubles) of the fronts in the pooled front workspace
  int64_t pool_doubles = 0;         // size of that workspace
  std::vector<int64_t> w_off;       // nsuper+1, prefix sum of front sizes
  std::vector<int> child_ptr, child_idx;  // children of each supernode (ascending)
  int nlevels = 0;
  std::vector<int> level_ptr, level_sn;   // supernodes grouped by level
  int64_t nnzL = 0, exact_nnzL = 0, flops = 0;
  int maxfront = 0, maxcols = 0;
  // options actually used
  int leaf_cols = 16, max_super_cols = 256, nd_leaf = 8, relax = 1;
  // opaque device mirror owned by factor.cu
  void* dev = nullptr;
  void (*dev_free)(void*) = nullptr;
};

inline int sn_ncols(const eigd_symbolic* s, int k) { return s->sn_first[k + 1] - s->sn_first[k]; }
inline int sn_nbelow(const eigd_symbolic* s, int k) { return (int)(s->sn_rowptr[k + 1] - s->sn_rowptr[k]); }
inline int sn_fsize(const eigd_symbolic* s, int k) { return sn_ncols(s, k) + sn_nbelow(s, k); }

void eigd_set_error(const char* fmt, ...);
