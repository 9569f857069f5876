// Multi-RHS sparse triangular solves x = (L D L^T)^{-1} b as ONE persistent kernel.
// Replaces SuperLU.solve behind SpLuOperator._matvec (reference eigd/eigenvector_derivatives.py:18-23),
// which the reference calls once per right-hand-side column.
//
// Formulation.  The factorisation leaves, for every front (supernode with nc pivot columns and nb
// rows below them, f = nc + nb), the dense solve panel S = [L11^{-1} ; -L21 L11^{-1}] (f x nc) and
// its transpose.  With w1 = (b restricted to the pivot rows) + (updates gathered from the children):
//     forward :  [y1 ; u2] = S w1,   z1 = D^{-1} y1 kept, u2 (+ gathered child rows) passed up;
//     backward:  x1 = S^T [z1 ; x2], x2 = solution entries of the front's below rows (ancestors).
// Neither sweep has a dependency inside a front, so a level of the assembly tree is one batch of
// independent dense products.  Above the cut the persistent kernel walks the 2 * nlevels level phases in order,
// but there is NO grid barrier between them: every front owns a forward and a backward completion counter, a tile
// waits (ld.acquire spin of one lane per dependency) only for the fronts it actually reads from -- its children
// in the forward sweep, its parent in the backward sweep -- and the panel entries of its first chunk are already
// in flight while it waits (TileDep in solve_plan.hpp).
//
// Mapping.  512-thread CTAs (16 tile warps), one per SM, cooperative launch.  A warp tile is 32 (16, 8 on the upper
// levels) consecutive outputs of one front (lane = output), the reduction dimension is streamed in chunks of 32 whose
// input vectors are staged in shared memory ([k][32] per warp).  Panels of the fronts above the cut are stored
// tile-major (solve_plan.hpp): for one- and two-column solves a 17th PRODUCER warp streams every warp's panel slices
// into shared-memory rings ahead of time (cp.async.bulk + mbarriers, section "ASYNCHRONOUS PANEL PIPELINE" below);
// wider solves read the entries straight from HBM, coalesced across the lanes.  On the upper levels, where a level
// has few tiles, ws warps share a tile and split its reduction dimension; partial sums meet in shared memory.  Update
// vectors are gathered (pull lists built on the host), never scattered: no atomics, bitwise reproducible sums.
//
// Algorithmic bytes per call (SURVEY.md 8d): 2*(nnz(L)*8 + idx) + n*8 + 4*n*k*8.
#include "factor_internal.cuh"
#include "../../include/eigd_b200.h"

#include <algorithm>
#include <vector>

namespace {

constexpr int MAX_PHASES_SMEM = 96;
constexpr int MAX_SUB_LEVELS = 32;

struct SolveArgs {
  const TileRec* tiles;
  const PhaseRec* phases;
  int nphases;
  const int* ovf_row;
  const int* ovf;
  const int* sub_ptr;
  const int* perm;
  const int* sn_rows;
  const int* rel;
  const double* sfwd;
  const double* sbwd;
  const double* dinv;
  double* wbuf;          // three slabs x kmax planes x sumf rows
  int64_t sumf;          // rows per plane
  int64_t slab_stride;   // kmax * sumf
  double* bperm;         // permuted right-hand side, n x k
  double* ybuf;
  double* xperm;
  const double* B;
  int64_t brs, bcs;
  double* X;
  int64_t xrs, xcs;
  int n, k;
  const TileDep* deps;            // per-tile completion-counter dependencies (level phases)
  const int* dep_ovf;
  unsigned long long* barrier;    // arrival counter of the (rare) grid barriers, monotone
  unsigned long long bar_base;
  unsigned* cnt;                  // completion counters: 2 * supernode + direction, monotone over the solves of a factor
  unsigned epoch;                 // number of this solve (1, 2, ...): counter c is complete at epoch * tiles(c)
  int p_begin, p_end;             // phases run by the cooperative kernel
  int ring_w;                     // bytes of shared-memory panel buffer per warp (front mode of the subtree phases)
  int lring_w;                    // bytes of shared-memory panel ring per warp in the level kernel (KT <= 2; 0 otherwise)
  int rec_cap;                    // tile records of a slot that fit in shared memory
  unsigned long long* times;      // developer profiling: %globaltimer of CTA 0 after every phase (NULL: off)
  unsigned long long* skew;       // developer profiling: %globaltimer of EVERY CTA's warp 0 in its first tile of every level
                                  // phase of the pipelined kernel, 4 slots per (phase, CTA): tile start, slot there,
                                  // dependencies complete, signalled (NULL: off)
  long long* trace;               // developer profiling: clock64 of CTA 0 / warp 0 inside its first tile of every level
                                  // phase, 16 slots per phase: 0 start, 1 waited, 2 product done, 3 reduced, 4 stored,
                                  // 5 signalled, 6 slot (record + panel slice) there, 7 end of tile, 8 top of the phase loop,
                                  // 9 dispatch
  int blk_mask;                   // 31 for a factor with restricted Bunch-Kaufman pivoting, else 0: its pivot blocks of S are
                                  // block lower triangular at 32-row granularity (dense 32 x 32 diagonal blocks), so the
                                  // triangular skip bounds of a thin tile (TH < 32) are widened to the 32-row block
};

// vectors produced earlier in the same launch by other SMs are read through L2 (ld.global.cg): L1 is
// not coherent across SMs and a line fetched in an earlier phase may be stale
template <int KT>
__device__ __forceinline__ void add_row(const double* __restrict__ base, int64_t row, int k, double* v) {
  const double* p = base + row * k;
#pragma unroll
  for (int r = 0; r < KT; ++r)
    if (r < k) v[r] += __ldcg(p + r);
}

// v += the updates addressed to w-row t by third and later children (overflow slab), via the row's source list
template <int KT>
__device__ __forceinline__ void ovf_add(const SolveArgs& a, int64_t t, double* v) {
  const int o = __ldg(&a.ovf_row[t]);
  if (o < 0) return;
  const int cnt = __ldg(&a.ovf[o]);
  const double* p2 = a.wbuf + 2 * a.slab_stride;
  for (int q = 0; q < cnt; ++q) {
    const int64_t src = __ldg(&a.ovf[o + 1 + q]);
#pragma unroll
    for (int r = 0; r < KT; ++r)
      if (r < a.k) v[r] += __ldcg(p2 + (int64_t)r * a.sumf + src);
  }
}

// v += the forward-sweep updates addressed to w-row t: slab 0 + slab 1 (+ overflow list), fixed order
template <int KT>
__device__ __forceinline__ void child_add(const SolveArgs& a, int64_t t, int64_t link, double* v) {
  if (!(link & LINK_HAS_CHILDREN)) return;
  const double* p0 = a.wbuf + t;
  const double* p1 = p0 + a.slab_stride;
#pragma unroll
  for (int r = 0; r < KT; ++r)
    if (r < a.k) v[r] += __ldcg(p0 + (int64_t)r * a.sumf) + __ldcg(p1 + (int64_t)r * a.sumf);
  if (link & LINK_HAS_OVF) ovf_add<KT>(a, t, v);
}

// v += w1 entry c of a front in the forward sweep: the right-hand side (gathered from B through perm in the first phase,
// else the permuted copy) + the children's updates; v is zero on entry
template <int KT>
__device__ __forceinline__ void fwd_operand(const SolveArgs& a, bool use_perm, const TileRec& tr, int c, double* v) {
  if (use_perm) {
    const int64_t po = __ldg(&a.perm[tr.first + c]);
    const double* bp = a.B + po * a.brs;
#pragma unroll
    for (int r = 0; r < KT; ++r)
      if (r < a.k) v[r] = bp[(int64_t)r * a.bcs];
  } else {
    add_row<KT>(a.bperm, tr.first + c, a.k, v);
  }
  child_add<KT>(a, tr.w_off + c, tr.link, v);
}

// v += input entry i of a front in the backward sweep: z1 for a pivot row, the solution x2 (through sn_rows) below them
template <int KT>
__device__ __forceinline__ void bwd_operand(const SolveArgs& a, const TileRec& tr, int i, double* v) {
  if (i < tr.nc) add_row<KT>(a.ybuf, tr.first + i, a.k, v);
  else add_row<KT>(a.xperm, __ldg(&a.sn_rows[tr.row_off + i - tr.nc]), a.k, v);
}

// thin tile (TH < 32): the 32 / TH lane groups that shared the columns of every chunk add up their sums
template <int KT, int TH>
__device__ __forceinline__ void group_reduce(double* acc) {
  if (TH < 32) {
#pragma unroll
    for (int o = TH; o < 32; o <<= 1)
#pragma unroll
      for (int r = 0; r < KT; ++r) acc[r] += __shfl_xor_sync(0xffffffffu, acc[r], o);
  }
}

// permuted copy of the right-hand side for the later phases (coalesced writes, gathered reads); thread t of nt
__device__ __forceinline__ void permute_rhs(const SolveArgs& a, int64_t t, int64_t nt) {
  const int k = a.k;
  for (int64_t e = t; e < (int64_t)a.n * k; e += nt) {
    const int64_t i = e / k;
    const int r = (int)(e - i * k);
    a.bperm[e] = a.B[(int64_t)__ldg(&a.perm[i]) * a.brs + (int64_t)r * a.bcs];
  }
}

__device__ __forceinline__ TileRec unpack_tile(int4 a, int4 b, int4 c) {
  TileRec t;
  t.first = a.x; t.nc = a.y; t.nb = a.z; t.tile = a.w;
  t.soff = ((int64_t)(unsigned)b.x) | ((int64_t)b.y << 32);
  t.w_off = ((int64_t)(unsigned)b.z) | ((int64_t)b.w << 32);
  t.row_off = ((int64_t)(unsigned)c.x) | ((int64_t)c.y << 32);
  t.link = ((int64_t)(unsigned)c.z) | ((int64_t)c.w << 32);
  return t;
}

__device__ __forceinline__ TileRec load_tile(const TileRec* p) {
  const int4* q = reinterpret_cast<const int4*>(p);
  return unpack_tile(__ldg(q), __ldg(q + 1), __ldg(q + 2));
}

// acc += M[out, c0:c1) * in[c0:c1) for this lane's output; M column-major with leading dimension ld.
// stage_fn(c, v) fills v[0:k) with input vector entry c (lane-parallel over the chunk of 32 columns),
// the chunk is then shared through the warp's staging buffer.  Memory-level parallelism comes from the
// instruction stream, not from occupancy: the panel entries of a sub-chunk are requested back to back
// (MC independent 8-byte loads per lane, 256 B per warp each) BEFORE the gather of the input vector, so
// one DRAM round trip covers MC columns.
template <int KT>
struct DefaultMC {
  static constexpr int value = KT <= 2 ? 32 : (KT <= 10 ? 16 : 8);
};

// Completion-counter wait of one tile: lane d < 2 polls inline dependency d, further dependencies are polled
// lane-strided from the overflow list; the warp leaves together.  Called at most once per tile (first use).
struct DepWait {
  const unsigned* cnt;
  const int* ovf;
  unsigned epoch;
  TileDep td;
  bool pending;
  __device__ __forceinline__ void arm(int4 d0, int4 d1) {     // the tile's TileDep, read as two 16-byte words
    td.self = d0.x; td.ndep = d0.y; td.d0 = d0.z; td.n0 = d0.w;
    td.d1 = d1.x; td.n1 = d1.y; td.ovf = d1.z; td.pad = 0;
    pending = td.ndep > 0;
  }
  __device__ __forceinline__ static void spin(const unsigned* c, unsigned need) {
    unsigned v;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(c) : "memory");
    } while ((int)(v - need) < 0);
  }
  __device__ __forceinline__ void operator()(int lane) {
    if (!pending) return;
    pending = false;
    if (lane < 2 && lane < td.ndep) spin(cnt + (lane ? td.d1 : td.d0), epoch * (unsigned)(lane ? td.n1 : td.n0));
    for (int q = 2 + lane; q < td.ndep; q += 32) {
      const int* e = ovf + td.ovf + 2 * (q - 2);
      spin(cnt + __ldg(e), epoch * (unsigned)__ldg(e + 1));
    }
    __syncwarp();
  }
};
struct NoWait {
  __device__ __forceinline__ void operator()(int) {}
};

__device__ __forceinline__ void signal_done(unsigned* c) {
  // the warp's stores happen-before lane 0's release through the warp barrier (cumulativity)
  __syncwarp();
  if ((threadIdx.x & 31) == 0) asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(c) : "memory");
}

// TH = tile height (outputs per warp tile): 32 (lane = output), or 16 / 8 on the upper levels, where a level has too few
// 32-output tiles to occupy the SMs and a 32-row slice of a wide front would make ONE SM stream 64 - 128 KB (its
// load path, ~64 B per clock, is then the bound).  With TH < 32 the lanes form 32 / TH groups that share the
// columns of a chunk (group g takes columns g, g + 32 / TH, ...) and meet in a shuffle reduction at the end.
template <int KT, int MC, int TH, class StageFn, class WaitFn>
__device__ __forceinline__ void warp_panel_product(const double* __restrict__ M, int64_t ld, int c0, int c1, int lane,
                                                   double* stage, double* acc, StageFn stage_fn, WaitFn& wait) {
  constexpr int nks = 32 / TH;
  const int g = lane / TH;
  for (int cc = c0; cc < c1; cc += 32) {
    const int ncol = min(32, c1 - cc);
    const double* Mc = M + (int64_t)(cc + g) * ld;
    const int64_t step = (int64_t)nks * ld;
    double m[MC];
#pragma unroll
    for (int j = 0; j < MC; ++j) m[j] = (g + j * nks < ncol) ? __ldg(Mc + j * step) : 0.0;
    double v[KT];
#pragma unroll
    for (int r = 0; r < KT; ++r) v[r] = 0.0;
    wait(lane);                     // the panel loads above are in flight while the producers of the operands finish
    if (lane < ncol) stage_fn(cc + lane, v);
#pragma unroll
    for (int r = 0; r < KT; ++r) stage[r * 32 + lane] = v[r];
    __syncwarp();
#pragma unroll
    for (int j = 0; j < MC; ++j)
#pragma unroll
      for (int r = 0; r < KT; ++r) acc[r] = fma(m[j], stage[r * 32 + ((g + j * nks) & 31)], acc[r]);
    if (MC * nks < 32) {
      for (int j0 = MC; g + j0 * nks < ncol; j0 += MC) {          // warp-uniform trip count is not needed: no sync inside
#pragma unroll
        for (int j = 0; j < MC; ++j) m[j] = (g + (j0 + j) * nks < ncol) ? __ldg(Mc + (j0 + j) * step) : 0.0;
#pragma unroll
        for (int j = 0; j < MC; ++j)
#pragma unroll
          for (int r = 0; r < KT; ++r) acc[r] = fma(m[j], stage[r * 32 + ((g + (j0 + j) * nks) & 31)], acc[r]);
      }
    }
    __syncwarp();
  }
}

// Grid-wide barrier, only behind phase 0 of a plan without subtree phases: the later phases read the permuted copy of
// the right-hand side that all CTAs write during phase 0, which no completion counter covers.
// (the caller puts a CTA barrier -- of all its participating warps -- on both sides)
__device__ __forceinline__ void grid_barrier_arrive_wait(unsigned long long* ctr, unsigned long long target) {
  if (threadIdx.x == 0) {
    unsigned long long v;
    asm volatile("red.release.gpu.global.add.u64 [%0], 1;" ::"l"(ctr) : "memory");
    do {
      asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(ctr) : "memory");
    } while (v < target);
  }
}

// the products of one warp tile: slice `slice` of `ws` of the reduction dimension.
// use_perm: the right-hand side is gathered from B through perm (first phase; later phases read the
// permuted copy written during the first one)
// TILED: the front's panels are stored tile-major with tile height TH (fronts above the cut, solve_plan.hpp); column-major
// below the cut (the tile path of fronts_phase)
template <int KT, int MC = DefaultMC<KT>::value, int TH = SOLVE_TILE, bool TILED = false, class WaitFn>
__device__ __forceinline__ void tile_compute(const SolveArgs& a, int dir, bool use_perm, const TileRec& tr, int lane,
                                             int slice, int ws, double* stage, double* acc, WaitFn& wait) {
  constexpr int to = TH;
  constexpr int MCT = MC < TH ? MC : TH;               // loads in flight per lane and chunk: a chunk has TH columns per lane group
  const int nc = tr.nc, f = tr.nc + tr.nb;
  const int o0 = tr.tile * to;
  const int out = o0 + (lane % to);
  if (dir == 0) {
    // ---- forward: outputs are front rows; acc = S[row, 0:cend) w1 (+ the children's updates of the row)
    // S is lower triangular inside the pivot rows (a pivoted factor: at 32-row granularity; TH = 32 tiles start on a
    // 32-row edge, thin tiles read on to the end of their 32-row block)
    const int cend = min(nc, TH < 32 ? (o0 + to + a.blk_mask) & ~a.blk_mask : o0 + to);
    const int per = solve_slice_len(cend, ws);
    const int c0 = min(cend, slice * per), c1 = min(cend, c0 + per);
    const int th = min(to, f - o0);                     // rows of this row tile
    const double* M = TILED ? a.sfwd + tr.soff + (int64_t)o0 * nc + min(lane % to, th - 1) : a.sfwd + tr.soff + min(out, f - 1);
    warp_panel_product<KT, MCT, TH>(M, TILED ? th : f, c0, c1, lane, stage, acc,
                                    [&](int c, double* v) { fwd_operand<KT>(a, use_perm, tr, c, v); }, wait);
    wait(lane);
    group_reduce<KT, TH>(acc);
    if (slice == 0 && lane < to && out >= nc && out < f) {
      double cu[KT];                                    // the children's updates of this output row
#pragma unroll
      for (int r = 0; r < KT; ++r) cu[r] = 0.0;
      child_add<KT>(a, tr.w_off + out, tr.link, cu);
#pragma unroll
      for (int r = 0; r < KT; ++r) acc[r] += cu[r];
    }
  } else {
    // ---- backward: outputs are pivot columns; acc = S^T[col, ob:f) [z1 ; x2], ob = o0 (pivoted factor, thin tile: the
    // first row of o0's 32-row block)
    const int ob = TH < 32 ? o0 & ~a.blk_mask : o0;
    const int len = f - ob;
    const int per = solve_slice_len(len, ws);
    const int i0 = min(f, ob + slice * per), i1 = min(f, i0 + per);
    const int tw = min(to, nc - o0);                    // pivot columns of this column tile
    const double* M = TILED ? a.sbwd + tr.soff + (int64_t)o0 * f + min(lane % to, tw - 1) : a.sbwd + tr.soff + min(out, nc - 1);
    warp_panel_product<KT, MCT, TH>(M, TILED ? tw : nc, i0, i1, lane, stage, acc,
                                    [&](int i, double* v) { bwd_operand<KT>(a, tr, i, v); }, wait);
    wait(lane);
    group_reduce<KT, TH>(acc);
  }
}

// The stores of a tile's outputs: z1 = D^-1 y1 (forward, pivot rows), the update rows into the parent's slab (forward,
// below the pivots), the solution into xperm and X (backward).  tile_store_request loads the index / scaling operands
// (the D^-1 entry, the parent row position or the original index of the output); the pipelined level kernel requests
// them BEFORE the tile waits for its dependencies, so that they sit in registers when the sums are ready instead of
// adding a dependent look-up (an L2 or DRAM round trip) between the last FMA and the stores.
struct StoreOps {
  double di;
  int64_t dst;
};
template <int TH>
__device__ __forceinline__ StoreOps tile_store_request(const SolveArgs& a, int dir, const TileRec& tr, int lane) {
  StoreOps o;
  o.di = 0.0;
  o.dst = 0;
  const int nc = tr.nc, f = tr.nc + tr.nb;
  const int out = tr.tile * TH + lane;
  if (TH < 32 && lane >= TH) return o;
  if (dir == 0) {
    if (out < nc) o.di = __ldg(&a.dinv[tr.first + out]);
    else if (out < f) {
      const int slab = (int)((tr.link >> LINK_SLAB_SHIFT) & 0xff);
      if (slab < 2) o.dst = slab * a.slab_stride + (tr.link & LINK_WOFF_MASK) + __ldg(&a.rel[tr.row_off + out - nc]);
      else o.dst = 2 * a.slab_stride + tr.w_off + out;
    }
  } else if (out < nc) {
    o.dst = (int64_t)__ldg(&a.perm[tr.first + out]) * a.xrs;
  }
  return o;
}
template <int KT, int TH>
__device__ __forceinline__ void tile_store_with(const SolveArgs& a, int dir, const TileRec& tr, int lane, const double* acc,
                                                const StoreOps& o) {
  const int k = a.k;
  const int nc = tr.nc, f = tr.nc + tr.nb;
  const int out = tr.tile * TH + lane;
  if (TH < 32 && lane >= TH) return;
  if (dir == 0) {
    if (out < nc) {
      double* y = a.ybuf + (int64_t)(tr.first + out) * k;
#pragma unroll
      for (int r = 0; r < KT; ++r)
        if (r < k) y[r] = o.di * acc[r];
    } else if (out < f) {
      double* w = a.wbuf + o.dst;
#pragma unroll
      for (int r = 0; r < KT; ++r)
        if (r < k) w[(int64_t)r * a.sumf] = acc[r];
    }
  } else if (out < nc) {
    double* xp = a.xperm + (int64_t)(tr.first + out) * k;
    double* xo = a.X + o.dst;
#pragma unroll
    for (int r = 0; r < KT; ++r)
      if (r < k) { xp[r] = acc[r]; xo[(int64_t)r * a.xcs] = acc[r]; }
  }
}

template <int KT, int TH = SOLVE_TILE>
__device__ __forceinline__ void tile_store(const SolveArgs& a, int dir, const TileRec& tr, int lane, const double* acc) {
  tile_store_with<KT, TH>(a, dir, tr, lane, acc, tile_store_request<TH>(a, dir, tr, lane));
}

// ---------------------------------------------------------------------------------------------------------
// FRONT MODE of the subtree phases.  Below the cut the fronts are small (nc ~ 4 - 30 pivot columns, f ~ 20 - 110
// rows: a 2 - 10 KB panel) and there are thousands of them per SM; with one warp tile per 32 outputs the solve
// was bound by the load/store path (every lane fetching 8 bytes of panel per instruction, all 16 warps at
// once) and by per-tile overhead, not by DRAM (DESIGN.md section 5).  Here the unit of work is a FRONT: lane 0
// of the warp brings the whole panel -- one contiguous, 16-byte aligned run of f x nc doubles -- into the warp's
// shared-memory buffer with ONE bulk copy (cp.async.bulk, completion on an mbarrier), the next front's panel is
// requested before the current one is consumed (two half-buffers), the operand vector is gathered once per
// front instead of once per tile, and all row tiles run out of shared memory.  Fronts that do not fit (panel
// larger than FRONT_PANEL_MAX, or more than 32 pivot columns; for k >= 2 in the backward sweep also a panel and
// operand block larger than the warp's buffer) take the tile path below, record by record.
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void bulk_load(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  unsigned ok;
  do {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok)
                 : "r"(smem_u32(bar)), "r"(parity)
                 : "memory");
  } while (!ok);
}

// per-lane asynchronous copies into shared memory (LDGSTS): they hold no register while in flight, and each lane
// has its own source address, so they serve the gathers through perm, rel and sn_rows as well
__device__ __forceinline__ void cp_async8(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

constexpr int FRONT_TILES_MAX = 8;   // row tiles / row chunks of a front in front mode (k >= 2): f <= 256
constexpr int FRONT_RT = 3;    // row tiles (forward) / row chunks (backward) of a front in the k = 1 pipeline: f <= 96
// Largest panel that takes front mode.  Not the ring size: the forward front path adds the children's updates of a row
// before its products, the tile path after them, so moving this bound would change the bits of the result.
constexpr int FRONT_PANEL_MAX = 10240;

// Operands of one front, REQUESTED one front ahead (software pipeline in registers, k = 1): by the time the
// front is processed its loads have landed, so a front costs no exposed memory round trip in the forward sweep
// and one (index -> value) in the backward sweep.
struct FrontOps {
  double b, s0, s1;                  // forward: w1 entry of lane c = b + (s0 + s1)
  double u0[FRONT_RT], u1[FRONT_RT];   // forward: children's updates of row t*32 + lane
  double auxd[FRONT_RT];             // forward: D^-1 of pivot row t*32 + lane
  int auxi[FRONT_RT];                // forward: position of update row t*32 + lane in the parent; backward:
                                     // row index of input entry t*32 + lane (auxi[t]) ...
  int perm0;                         // ... backward: original index of pivot column `lane`
};

__device__ __forceinline__ void front_request(const SolveArgs& a, int dir, bool use_perm, const TileRec& tr, int lane,
                                              FrontOps& o) {
  const int nc = tr.nc, f = tr.nc + tr.nb;
  const bool kids = (tr.link & LINK_HAS_CHILDREN) != 0;
  if (dir == 0) {
    const int64_t col = tr.first + min(lane, nc - 1);
    const double* bp = use_perm ? a.B + (int64_t)__ldg(&a.perm[col]) * a.brs : a.bperm + col;
    const double* w0 = a.wbuf + tr.w_off + lane;
    const bool ok = lane < nc;
    o.b = ok ? __ldcg(bp) : 0.0;
    o.s0 = (ok && kids) ? __ldcg(w0) : 0.0;
    o.s1 = (ok && kids) ? __ldcg(w0 + a.slab_stride) : 0.0;
#pragma unroll
    for (int t = 0; t < FRONT_RT; ++t) {
      const int row = t * SOLVE_TILE + lane;
      o.auxd[t] = row < nc ? __ldg(&a.dinv[tr.first + row]) : 0.0;
      o.auxi[t] = (row >= nc && row < f) ? __ldg(&a.rel[tr.row_off + row - nc]) : 0;
      const bool upd = kids && row >= nc && row < f;
      o.u0[t] = upd ? __ldcg(w0 + t * SOLVE_TILE) : 0.0;
      o.u1[t] = upd ? __ldcg(w0 + t * SOLVE_TILE + a.slab_stride) : 0.0;
    }
  } else {
    o.perm0 = lane < nc ? __ldg(&a.perm[tr.first + lane]) : 0;
#pragma unroll
    for (int t = 0; t < FRONT_RT; ++t) {
      const int i = t * SOLVE_TILE + lane;
      o.auxi[t] = i < nc ? tr.first + i : (i < f ? __ldg(&a.sn_rows[tr.row_off + i - nc]) : 0);
    }
  }
}

// one front of a one-column solve out of shared memory (buf = its panel, copy completion on `bar`), with the operands
// prefetched into registers
__device__ __forceinline__ void front_compute_k1(const SolveArgs& a, int dir, const TileRec& tr, const double* buf,
                                                 unsigned long long* bar, unsigned parity, const FrontOps& ops, int lane,
                                                 double* stage) {
  const int nc = tr.nc, f = tr.nc + tr.nb;
  const int ntile = (f + SOLVE_TILE - 1) / SOLVE_TILE;
  if (dir == 0) {
    // ---- forward: w1 (nc <= 32 entries) staged once, then every row tile of S w1 out of shared memory
    double v = ops.b + (ops.s0 + ops.s1);
    if ((tr.link & LINK_HAS_OVF) && lane < nc) {
      double z = 0.0;
      ovf_add<1>(a, tr.w_off + lane, &z);
      v += z;
    }
    stage[lane] = v;
    __syncwarp();
    mbar_wait(bar, parity);
#pragma unroll
    for (int t = 0; t < FRONT_RT; ++t) {
      if (t >= ntile) break;
      const int row = t * SOLVE_TILE + lane;
      double acc = 0.0;
      const int cend = min(nc, (t + 1) * SOLVE_TILE);
      const double* col = buf + min(row, f - 1);
#pragma unroll 4
      for (int c = 0; c < cend; ++c) acc = fma(col[c * f], stage[c], acc);
      acc += ops.u0[t] + ops.u1[t];
      if ((tr.link & LINK_HAS_OVF) && row >= nc && row < f) ovf_add<1>(a, tr.w_off + row, &acc);
      // store with the prefetched D^-1 / parent position (tile_store without its look-up)
      if (row < nc) {
        a.ybuf[tr.first + row] = ops.auxd[t] * acc;
      } else if (row < f) {
        const int sl = (int)((tr.link >> LINK_SLAB_SHIFT) & 0xff);
        const int64_t dst = sl < 2 ? sl * a.slab_stride + (tr.link & LINK_WOFF_MASK) + ops.auxi[t]
                                   : 2 * a.slab_stride + tr.w_off + row;
        a.wbuf[dst] = acc;
      }
    }
  } else {
    // ---- backward: x1 = S^T [z1 ; x2], lane = pivot column (nc <= 32), front rows streamed in chunks of 32; all
    // chunks' values are requested at once (their indices arrived with the previous front)
    double vv[FRONT_RT];
#pragma unroll
    for (int t = 0; t < FRONT_RT; ++t) {
      const int i = t * SOLVE_TILE + lane;
      vv[t] = i < f ? __ldcg((i < nc ? a.ybuf : a.xperm) + ops.auxi[t]) : 0.0;
    }
    mbar_wait(bar, parity);
    double acc = 0.0;
    const double* colp = buf + min(lane, nc - 1);
#pragma unroll
    for (int t = 0; t < FRONT_RT; ++t) {
      const int cc = t * SOLVE_TILE;
      if (cc >= f) break;
      const int nrow = min(32, f - cc);
      stage[lane] = vv[t];
      __syncwarp();
      const double* rowp = colp + cc * nc;
#pragma unroll 4
      for (int j = 0; j < nrow; ++j) acc = fma(rowp[j * nc], stage[j], acc);
      __syncwarp();
    }
    if (lane < nc) {
      a.xperm[tr.first + lane] = acc;
      a.X[(int64_t)ops.perm0 * a.xrs] = acc;
    }
  }
}

// ---- OPERAND STAGING of a multi-column front (KT >= 2).  The operands travel in shared memory, in the warp's ring
// right behind the front's panel (same allocation), requested one front ahead with per-lane cp.async:
//   forward : b [nc][k] (right-hand side of the pivot rows) | s0, s1 [k][f] (slabs 0 and 1 of every row; fronts with
//             children only) | D^-1 [nc] | rel [nb] (int, parent positions of the update rows)
//   backward: v [f][KT] (the input [z1 ; x2], gathered at the front's start through the indices) | sn_rows [nb] (int)
//             | perm [nc] (int)
// The request is split in two: the early part goes out before the current front is computed; the late part needs an
// index loaded by the early part (forward, first phase: B through perm) and closes the front's copy group.
// The forward sweep stages its operands at KT = 2 only.  C2 on a B200 (forward subtree phase, CTA-0 timestamps, staging
// in every forward front that fits): k = 2 55.6 -> 52.4 us, but k = 4 69.7 -> 71.9 us and k = 10 135.1 -> 144.1 us;
// there the direct loads stay (profiles/r3_subtree_staging.txt).
template <int KT>
constexpr bool FWD_STAGE = KT == 2;

__host__ __device__ __forceinline__ int front_ops_doubles(const TileRec& t, int dir, int k, int kt) {
  const int nc = t.nc, nb = t.nb, f = nc + nb;
  if (dir == 0) return k * nc + ((t.link & LINK_HAS_CHILDREN) ? 2 * k * f : 0) + nc + (nb + 1) / 2;
  return f * kt + (nb + nc + 1) / 2;
}

template <int KT>
__device__ __forceinline__ int front_ops_early(const SolveArgs& a, int dir, bool use_perm, const TileRec& tr, int lane,
                                               double* ops) {
  if (dir != 0 || !FWD_STAGE<KT>) return 0;
  const int k = a.k;
  const int nc = tr.nc, f = tr.nc + tr.nb;
  if (!use_perm)
    for (int e = lane; e < nc * k; e += 32) cp_async8(ops + e, a.bperm + (int64_t)tr.first * k + e);
  double* d = ops + k * nc;
  if (tr.link & LINK_HAS_CHILDREN) {
    for (int r = 0; r < k; ++r)
      for (int row = lane; row < f; row += 32) {
        const double* s = a.wbuf + tr.w_off + row + (int64_t)r * a.sumf;
        cp_async8(d + r * f + row, s);
        cp_async8(d + (k + r) * f + row, s + a.slab_stride);
      }
    d += 2 * k * f;
  }
  if (lane < nc) cp_async8(d + lane, a.dinv + tr.first + lane);
  int* rel = reinterpret_cast<int*>(d + nc);
  for (int i = lane; i < tr.nb; i += 32) cp_async4(rel + i, a.rel + tr.row_off + i);
  return (use_perm && lane < nc) ? __ldg(&a.perm[tr.first + lane]) : 0;
}

template <int KT>
__device__ __forceinline__ void front_ops_late(const SolveArgs& a, int dir, bool use_perm, const TileRec& tr, int lane,
                                               double* ops, int po) {
  const int nc = tr.nc, f = tr.nc + tr.nb;
  if (dir == 0) {
    if (FWD_STAGE<KT> && use_perm && lane < nc) {
      const double* bp = a.B + (int64_t)po * a.brs;
#pragma unroll
      for (int r = 0; r < KT; ++r)
        if (r < a.k) cp_async8(ops + lane * a.k + r, bp + (int64_t)r * a.bcs);
    }
  } else {
    int* idx = reinterpret_cast<int*>(ops + f * KT);
    for (int i = lane; i < tr.nb; i += 32) cp_async4(idx + i, a.sn_rows + tr.row_off + i);
    if (lane < nc) cp_async4(idx + tr.nb + lane, a.perm + tr.first + lane);
  }
  cp_async_commit();
}

// acc[0:KT) = fma(m, s[0:KT), acc) with 16-byte shared loads, two right-hand sides each (s 16-byte aligned)
template <int KT>
__device__ __forceinline__ void fma_row(double m, const double* s, double* acc) {
  static_assert(KT % 2 == 0, "the paired operand layout needs an even KT");
  const double2* s2 = reinterpret_cast<const double2*>(s);
#pragma unroll
  for (int r = 0; r < KT / 2; ++r) {
    const double2 q = s2[r];
    acc[2 * r] = fma(m, q.x, acc[2 * r]);
    acc[2 * r + 1] = fma(m, q.y, acc[2 * r + 1]);
  }
}

// forward sweep of one front of a multi-column solve out of shared memory (buf = its panel, copy completion on `bar`).
// ops = its staged operand block, or NULL (it did not fit in the ring): the operands are then loaded directly, in the
// same summation order.  next_late() issues the late part of the next front's request once w1 is staged.
template <int KT, class NextFn>
__device__ __forceinline__ void front_forward(const SolveArgs& a, bool use_perm, const TileRec& tr, const double* buf,
                                              unsigned long long* bar, unsigned parity, const double* ops, int lane,
                                              double* stage, NextFn next_late) {
  const int k = a.k;
  const int nc = tr.nc, f = tr.nc + tr.nb;
  const bool kids = (tr.link & LINK_HAS_CHILDREN) != 0;
  const double* s0 = nullptr;    // the staged slabs, D^-1 and parent positions
  const double* dv = nullptr;
  const int* rel = nullptr;
  if (ops) {
    s0 = ops + k * nc;
    dv = s0 + (kids ? 2 * k * f : 0);
    rel = reinterpret_cast<const int*>(dv + nc);
    cp_async_wait<0>();           // this front's copy group (the next front's early part is not committed yet)
    __syncwarp();
  }
  // w1 entry of lane c: b + (s0 + s1) (+ overflow); stage[c][KT]
  double v[KT];
#pragma unroll
  for (int r = 0; r < KT; ++r) v[r] = 0.0;
  if (lane < nc) {
    if (ops) {
#pragma unroll
      for (int r = 0; r < KT; ++r)
        if (r < k) {
          const double b = ops[lane * k + r];
          v[r] = use_perm ? b : v[r] + b;
          if (kids) v[r] += s0[r * f + lane] + s0[(k + r) * f + lane];
        }
      if (tr.link & LINK_HAS_OVF) ovf_add<KT>(a, tr.w_off + lane, v);
    } else {
      fwd_operand<KT>(a, use_perm, tr, lane, v);
    }
  }
#pragma unroll
  for (int r = 0; r < KT; ++r) stage[lane * KT + r] = v[r];
  __syncwarp();
  next_late();
  mbar_wait(bar, parity);
  const int ntile = (f + SOLVE_TILE - 1) / SOLVE_TILE;
#pragma unroll 1
  for (int t = 0; t < FRONT_TILES_MAX; ++t) {
    if (t >= ntile) break;
    const int row = t * SOLVE_TILE + lane;
    double acc[KT];
#pragma unroll
    for (int r = 0; r < KT; ++r) acc[r] = 0.0;
    if (row >= nc && row < f) {
      if (!ops) {
        child_add<KT>(a, tr.w_off + row, tr.link, acc);
      } else if (kids) {
#pragma unroll
        for (int r = 0; r < KT; ++r)
          if (r < k) acc[r] += s0[r * f + row] + s0[(k + r) * f + row];
        if (tr.link & LINK_HAS_OVF) ovf_add<KT>(a, tr.w_off + row, acc);
      }
    }
    const int cend = min(nc, (t + 1) * SOLVE_TILE);
    const double* col = buf + min(row, f - 1);
#pragma unroll 4
    for (int c = 0; c < cend; ++c) fma_row<KT>(col[c * f], stage + c * KT, acc);
    if (!ops) {
      TileRec tt = tr;
      tt.tile = t;
      tile_store<KT>(a, 0, tt, lane, acc);
    } else if (row < nc) {
      double* y = a.ybuf + (int64_t)(tr.first + row) * k;
      const double di = dv[row];
#pragma unroll
      for (int r = 0; r < KT; ++r)
        if (r < k) y[r] = di * acc[r];
    } else if (row < f) {
      const int sl = (int)((tr.link >> LINK_SLAB_SHIFT) & 0xff);
      const int64_t dst = sl < 2 ? sl * a.slab_stride + (tr.link & LINK_WOFF_MASK) + rel[row - nc]
                                 : 2 * a.slab_stride + tr.w_off + row;
      double* w = a.wbuf + dst;
#pragma unroll
      for (int r = 0; r < KT; ++r)
        if (r < k) w[(int64_t)r * a.sumf] = acc[r];
    }
  }
}

// backward sweep of one front of a multi-column solve: x1 = S^T [z1 ; x2], lane = pivot column (nc <= 32).  The
// indices arrived with the previous front; the values go into v[f][KT] with one gather, while the next front's
// indices are requested, and the product runs over all f rows out of shared memory.
template <int KT, class NextFn>
__device__ __forceinline__ void front_backward(const SolveArgs& a, const TileRec& tr, const double* buf,
                                               unsigned long long* bar, unsigned parity, double* ops, int lane,
                                               NextFn next_late) {
  const int k = a.k;
  const int nc = tr.nc, f = tr.nc + tr.nb;
  const int* idx = reinterpret_cast<const int*>(ops + f * KT);
  cp_async_wait<0>();
  __syncwarp();
  for (int i = lane; i < f; i += 32) {
    const double* src = i < nc ? a.ybuf + (int64_t)(tr.first + i) * k : a.xperm + (int64_t)idx[i - nc] * k;
#pragma unroll
    for (int r = 0; r < KT; ++r)
      if (r < k) cp_async8(ops + i * KT + r, src + r);
  }
  cp_async_commit();
  next_late();
  cp_async_wait<1>();             // the gather (the next front's indices may stay in flight)
  __syncwarp();
  mbar_wait(bar, parity);
  double acc[KT];
#pragma unroll
  for (int r = 0; r < KT; ++r) acc[r] = 0.0;
  const double* colp = buf + min(lane, nc - 1);
#pragma unroll 4
  for (int j = 0; j < f; ++j) fma_row<KT>(colp[j * nc], ops + j * KT, acc);
  if (lane < nc) {
    double* xp = a.xperm + (int64_t)(tr.first + lane) * k;
    double* xo = a.X + (int64_t)idx[tr.nb + lane] * a.xrs;
#pragma unroll
    for (int r = 0; r < KT; ++r)
      if (r < k) { xp[r] = acc[r]; xo[(int64_t)r * a.xcs] = acc[r]; }
  }
}

constexpr int FRONT_DEPTH = 2;   // panel copies in flight per warp

// Every front of this CTA's slot that belongs to this warp (front te = T0(level) + warp + 16 j), level by level
// with a CTA barrier between levels.  The PANEL copies run ahead of the computation by up to FRONT_DEPTH fronts
// and across level boundaries (panels do not depend on computed data): a FIFO of variable-size allocations in the
// warp's ring buffer, one mbarrier per FIFO position.  The OPERANDS (right-hand side, child updates, D^-1, row
// positions; backward: row indices) are requested one front ahead, for the warp's next front of the SAME level only
// (the next level's depend on this level's results): into registers for k = 1 (FrontOps), into the front's ring
// allocation behind its panel in the backward sweep of k >= 2 and the forward sweep of k = 2 (FWD_STAGE).
template <int KT>
__device__ __forceinline__ void fronts_phase(const SolveArgs& a, int dir, bool use_perm, int nl, const int* s_tab, int tb,
                                             int nrec, const int4* s_rec, int lane, int warp, double* stage, char* ring,
                                             int ring_w, unsigned long long* bars, int* s_q) {
  constexpr bool K1 = KT == 1;
  const double* panels = dir == 0 ? a.sfwd : a.sbwd;
  auto record = [&](int te) {
    const int q = te - tb;
    return q < nrec ? unpack_tile(s_rec[3 * q], s_rec[3 * q + 1], s_rec[3 * q + 2]) : load_tile(a.tiles + te);
  };
  auto panel_bytes = [](const TileRec& t) { return (int)solve_panel_doubles(t.nc + t.nb, t.nc) * 8; };
  auto fits = [&](const TileRec& t, int b) {
    return t.nc <= 32 && b <= min(ring_w, FRONT_PANEL_MAX) && t.nc + t.nb <= (K1 ? FRONT_RT : FRONT_TILES_MAX) * SOLVE_TILE;
  };
  auto level_of = [&](int ll) { return dir == 0 ? ll : nl - 1 - ll; };
  // producer cursor (pl, pte): next front whose panel copy has not been requested yet
  int pl = 0, pte = s_tab[level_of(0)] + warp;
  auto p_skip = [&]() {           // move the producer cursor to a valid front or to the end (pl == nl)
    while (pl < nl && pte >= s_tab[level_of(pl) + 1]) {
      ++pl;
      if (pl < nl) pte = s_tab[level_of(pl)] + warp;
    }
  };
  p_skip();
  // FIFO head position and occupancy; entry e: s_q[2e] = offset (-1: tile path), s_q[2e+1] = bytes allocated (more than
  // the panel: the operand block follows it)
  int qh = 0, qn = 0;
  unsigned par = 0;               // parity bit per FIFO position
  int last_end = 0;               // end of the newest allocation
  auto produce = [&]() {
    while (qn < FRONT_DEPTH && pl < nl) {
      const TileRec t = record(pte);
      const int b = panel_bytes(t);
      const int e = (qh + qn) % FRONT_DEPTH;
      int off = -1, len = b;
      if (fits(t, b)) {
        if (!K1 && (dir == 1 || FWD_STAGE<KT>)) {
          // staged operands.  A forward front whose operands do not fit loads them directly, a backward one takes the
          // tile path (both paths of the backward sweep sum in the same order).
          const int ob = b + front_ops_doubles(t, dir, a.k, KT) * 8;
          if (ob <= ring_w) len = ob;
          else if (dir) len = -1;
        }
      } else {
        len = -1;
      }
      if (len >= 0) {
        off = (last_end + 127) & ~127;
        if (off + len > ring_w) off = 0;
        bool clash = false;
        for (int i = 0; i < qn; ++i) {
          const int ei = (qh + i) % FRONT_DEPTH;
          const int o = s_q[2 * ei], l = s_q[2 * ei + 1];
          if (o >= 0 && off < o + l && o < off + len) clash = true;
        }
        if (clash) return;         // no room yet: try again after the next front has been consumed
        if (lane == 0) bulk_load(ring + off, panels + t.soff, (unsigned)b, &bars[e]);
        last_end = off + len;
      }
      __syncwarp();
      if (lane == 0) { s_q[2 * e] = off; s_q[2 * e + 1] = len; }
      __syncwarp();
      ++qn;
      pte += SOLVE_WARPS;
      p_skip();
    }
  };
  // operand block of FIFO entry e holding front t, or NULL
  auto ops_of = [&](int e, const TileRec& t) -> double* {
    const int o = s_q[2 * e], b = panel_bytes(t);
    return (o >= 0 && s_q[2 * e + 1] > b) ? reinterpret_cast<double*>(ring + o + b) : nullptr;
  };
  produce();
  FrontOps ops, nops;
  bool ops_ready = false;
  for (int ll = 0; ll < nl; ++ll) {
    const int l = level_of(ll);
    const int t0 = s_tab[l], t1 = s_tab[l + 1];
    for (int te = t0 + warp; te < t1; te += SOLVE_WARPS) {
      TileRec tr = record(te);
      const int off = s_q[2 * qh];
      const unsigned parity = (par >> qh) & 1u;
      double* cur = nullptr;      // k >= 2: this front's staged operands
      bool nops_ready = false;
      if constexpr (K1) {
        if (off >= 0 && !ops_ready) front_request(a, dir, use_perm, tr, lane, ops);
        // operands of this warp's next front of the SAME level (the next level's depend on this level's results)
        if (te + SOLVE_WARPS < t1) {
          const TileRec nt = record(te + SOLVE_WARPS);
          if (fits(nt, panel_bytes(nt))) {
            front_request(a, dir, use_perm, nt, lane, nops);
            nops_ready = true;
          }
        }
      } else {
        cur = ops_of(qh, tr);
        if (cur && !ops_ready) front_ops_late<KT>(a, dir, use_perm, tr, lane, cur, front_ops_early<KT>(a, dir, use_perm, tr, lane, cur));
      }
      // k >= 2: the next front of the same level, if its FIFO entry already holds an operand block
      double* nxt = nullptr;
      int npo = 0;
      if (!K1 && te + SOLVE_WARPS < t1 && qn >= 2) {
        const TileRec nt = record(te + SOLVE_WARPS);
        nxt = ops_of((qh + 1) % FRONT_DEPTH, nt);
        if (nxt) npo = front_ops_early<KT>(a, dir, use_perm, nt, lane, nxt);
      }
      auto next_late = [&]() {      // (the record is read again: it would hold 12 registers across the front)
        if (nxt) front_ops_late<KT>(a, dir, use_perm, record(te + SOLVE_WARPS), lane, nxt, npo);
        else cp_async_commit();   // an empty group: front_backward waits for all but the newest
      };
      if (off < 0) {
        // ---- tile path (global loads), every 32-output tile of the front.  Panel loads in flight per lane: 8, 16 at
        // KT = 4, what the register budget left by the staged front paths allows.  Spill stores (ptxas, sm_100a) at
        // KT = 4 / 6 / 8 / 10: 20 / 0 / 24 / 20 bytes with 8, 8 / 16 / 20 / 92 with 16
        const int nc = tr.nc, f = tr.nc + tr.nb;
        const int ntile = ((dir == 0 ? f : nc) + SOLVE_TILE - 1) / SOLVE_TILE;
        for (int t = 0; t < ntile; ++t) {
          tr.tile = t;
          double acc[KT];
#pragma unroll
          for (int r = 0; r < KT; ++r) acc[r] = 0.0;
          NoWait nw;
          tile_compute<KT, (KT == 4 ? DefaultMC<KT>::value : 8)>(a, dir, use_perm, tr, lane, 0, 1, stage, acc, nw);
          tile_store<KT>(a, dir, tr, lane, acc);
        }
        if constexpr (!K1) next_late();
      } else {
        const double* buf = reinterpret_cast<const double*>(ring + off);
        if constexpr (K1) front_compute_k1(a, dir, tr, buf, &bars[qh], parity, ops, lane, stage);
        else if (dir == 0) front_forward<KT>(a, use_perm, tr, buf, &bars[qh], parity, FWD_STAGE<KT> ? cur : nullptr, lane, stage,
                                             next_late);
        else front_backward<KT>(a, tr, buf, &bars[qh], parity, cur, lane, next_late);
        par ^= 1u << qh;
      }
      __syncwarp();               // every lane is done with the allocation before it can be reused
      qh = (qh + 1) % FRONT_DEPTH;
      --qn;
      produce();
      if constexpr (K1) {
        ops = nops;
        ops_ready = nops_ready;
      } else {
        ops_ready = nxt != nullptr;
      }
    }
    ops_ready = false;
    __syncthreads();              // CTA-scope ordering: the level's results are visible to the whole slot
  }
}

// A subtree phase in FRONT MODE as its own (ordinary, non-cooperative) launch: one CTA per slot.  The forward one
// is the first thing a solve does, the backward one the last, so stream order replaces the grid barrier; the kernel
// gets its own register / shared-memory budget (panel ring) and the level kernel keeps its L1.  The operands of the next
// front are prefetched into registers for k = 1 and into the panel ring (cp.async) for k >= 2 (forward sweep: k = 2
// only): wider operands do not fit the 128-register budget of a 16-warp CTA.
template <int KT>
__global__ void __launch_bounds__(SOLVE_WARPS * 32, 1) subtree_kernel(SolveArgs a, int p) {
  extern __shared__ __align__(16) double smem[];
  __shared__ int s_tab[MAX_SUB_LEVELS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* stage = smem + warp * (32 * KT);                 // [KT][32] (tile path) or [32][KT] (front mode) per warp
  char* ring_all = reinterpret_cast<char*>(smem + SOLVE_WARPS * 32 * KT);
  unsigned long long* mbar_all = reinterpret_cast<unsigned long long*>(ring_all + (size_t)SOLVE_WARPS * a.ring_w);
  int* s_q = reinterpret_cast<int*>(mbar_all + FRONT_DEPTH * SOLVE_WARPS) + 2 * FRONT_DEPTH * warp;
  int4* s_rec = reinterpret_cast<int4*>(mbar_all + 2 * FRONT_DEPTH * SOLVE_WARPS);
  unsigned long long* bars = mbar_all + FRONT_DEPTH * warp;
  if (lane < FRONT_DEPTH) mbar_init(&bars[lane], 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  const PhaseRec ph = a.phases[p];
  const int dir = ph.dir, nl = ph.ntiles, nslots = ph.level;
  const bool use_perm = (p == 0);
  if (a.times && blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    a.times[p] = t;
  }
  for (int slot = blockIdx.x; slot < nslots; slot += gridDim.x) {
    const int* tab = a.sub_ptr + ph.tile_off + (int64_t)slot * (nl + 1);
    const int tb = __ldg(&tab[0]);
    const int nrec = min(__ldg(&tab[nl]) - tb, a.rec_cap);
    __syncthreads();
    if (threadIdx.x <= nl && threadIdx.x < MAX_SUB_LEVELS) s_tab[threadIdx.x] = __ldg(&tab[threadIdx.x]);
    {
      const int4* src = reinterpret_cast<const int4*>(a.tiles + tb);
      for (int e = threadIdx.x; e < 3 * nrec; e += blockDim.x) s_rec[e] = __ldg(src + e);
    }
    __syncthreads();
    fronts_phase<KT>(a, dir, use_perm, nl, s_tab, tb, nrec, s_rec, lane, warp, stage,
                     ring_all + (size_t)warp * a.ring_w, a.ring_w, bars, s_q);
  }
  if (use_perm) permute_rhs(a, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x);
  if (a.times && blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    a.times[p + 1] = t;
  }
}

// The partial sums of the ws warps that share a tile meet in shared memory (cta_sync: the CTA barrier of the warps that
// share tiles); the slice-0 warp (lead) adds them in a FIXED order (bitwise reproducible), for KT <= 2 in four
// independent chains at a time so that the shared-memory latencies overlap
template <int KT, class SyncFn>
__device__ __forceinline__ void reduce_slices(double* acc, double* part, int warp, int lane, int ws, bool lead,
                                              SyncFn cta_sync) {
#pragma unroll
  for (int r = 0; r < KT; ++r) part[(warp * KT + r) * 32 + lane] = acc[r];
  cta_sync();
  if (lead && KT > 2) {
    for (int s = 1; s < ws; ++s)
#pragma unroll
      for (int r = 0; r < KT; ++r) acc[r] += part[((warp + s) * KT + r) * 32 + lane];
  }
  if (lead && KT <= 2) {
#pragma unroll
    for (int r = 0; r < KT; ++r) {
      double p0 = 0.0, p1 = 0.0, p2 = 0.0, p3 = 0.0;
      for (int s = 1; s < ws; s += 4) {
        p0 += part[((warp + s) * KT + r) * 32 + lane];
        if (s + 1 < ws) p1 += part[((warp + s + 1) * KT + r) * 32 + lane];
        if (s + 2 < ws) p2 += part[((warp + s + 2) * KT + r) * 32 + lane];
        if (s + 3 < ws) p3 += part[((warp + s + 3) * KT + r) * 32 + lane];
      }
      acc[r] += (p0 + p1) + (p2 + p3);
    }
  }
}

// One level phase of the 16-warp level kernel (KT > 2): the tiles (height TH) of one level of the tree in one direction,
// CTA-strided; ws warps share a tile and split its reduction dimension.  Every tile reads its slice of the tile-major
// panel straight from global memory.  A tile waits for the completion counters of the fronts it reads from and
// increments its own front's counter when its outputs are stored (no grid barrier).
template <int KT, int TH>
__device__ __forceinline__ void level_phase(const SolveArgs& a, const PhaseRec& ph, int p, bool use_perm, int lane, int warp,
                                            double* stage, double* part, bool have_next, int4 (*s_next)[5]) {
  const int64_t tile_off = ph.tile_off;
  const int dir = ph.dir, ws = ph.ws, ntiles = ph.ntiles;
  const int tpc = SOLVE_WARPS / ws;
  const int sub = warp / ws, slice = warp - sub * ws;
  const int nct = (ntiles + tpc - 1) / tpc;
  for (int ct = blockIdx.x; ct < nct; ct += gridDim.x) {
    const int te = ct * tpc + sub;
    const bool have = te < ntiles;
    double acc[KT];
#pragma unroll
    for (int r = 0; r < KT; ++r) acc[r] = 0.0;
    TileRec tr{};
    DepWait dw{a.cnt, a.dep_ovf, a.epoch, TileDep{}, false};
    if (have) {
      int4 d0, d1;
      if (have_next && ct == (int)blockIdx.x) {
        tr = unpack_tile(s_next[warp][0], s_next[warp][1], s_next[warp][2]);
        d0 = s_next[warp][3];
        d1 = s_next[warp][4];
      } else {
        tr = load_tile(a.tiles + tile_off + te);
        const int4* q = reinterpret_cast<const int4*>(a.deps + tile_off + te);
        d0 = __ldg(q);
        d1 = __ldg(q + 1);
      }
      dw.arm(d0, d1);
      const bool tr_on = a.trace && blockIdx.x == 0 && ct == 0 && threadIdx.x == 0;
      if (tr_on) a.trace[16 * p + 0] = clock64();
      if (a.trace) {              // trace build of the chain: wait first so that the segments separate
        dw(lane);
        if (tr_on) a.trace[16 * p + 1] = clock64();
      }
      tile_compute<KT, DefaultMC<KT>::value, TH, true>(a, dir, use_perm, tr, lane, slice, ws, stage, acc, dw);
      if (tr_on) a.trace[16 * p + 2] = clock64();
    }
    if (ws > 1) reduce_slices<KT>(acc, part, warp, lane, ws, have && slice == 0, [] { __syncthreads(); });
    const bool tr_on2 = a.trace && blockIdx.x == 0 && ct == 0 && threadIdx.x == 0;
    if (tr_on2) a.trace[16 * p + 3] = clock64();
    if (have && slice == 0) {
      tile_store<KT, TH>(a, dir, tr, lane, acc);
      if (tr_on2) a.trace[16 * p + 4] = clock64();
      signal_done(a.cnt + dw.td.self);
      if (tr_on2) a.trace[16 * p + 5] = clock64();
    }
    if (ws > 1) __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------------
// ASYNCHRONOUS PANEL PIPELINE of the level phases: a warp-specialised producer / consumer kernel.
//
// Measured on the form in which every tile read its panel entries itself (profiles/r2_solve_pipeline.txt): a hop of
// the dependency chain took ~10 000 cycles, of which only ~2 000 are the hand-off through L2 -- the rest was a burst of
// 8-byte-per-lane panel loads through the SM's load path, requested only once the CTA had finished its tile of the
// previous phase, plus several thousand cycles of scalar bookkeeping (tile records, index arithmetic) executed by the
// same warp between two tiles.  Neither depends on computed data: the schedule is static (phase by phase, CTA-strided,
// warp = tile / slice) and the panels are constant during a solve.  So the level kernel has a 17th warp, the PRODUCER:
// lane w of it walks the tile sequence of consumer warp w ahead of time, fetches each tile's record and dependencies,
// works out the slice of the panel the warp will multiply -- ONE contiguous run in the tile-major panel storage
// (solve_plan.hpp) -- and requests it into the warp's shared-memory ring with one bulk copy (cp.async.bulk, completion
// on the slot's "full" mbarrier), up to PIPE_DEPTH tiles ahead, across phase boundaries.  A consumer warp waits for
// the slot (record + slice already there), for its dependencies' completion counters, gathers its operands, runs the
// FMAs out of shared memory, hands the slot back through its "empty" mbarrier and stores / signals.  Nothing but the
// hand-off, the operand gather and the arithmetic is left on the chain.
constexpr int PIPE_DEPTH = 3;      // slots (record + panel slice) per consumer warp
constexpr int PIPE_REC_INT4 = 6;   // TileRec (3 x 16 bytes) + TileDep (2 x 16 bytes) + slice descriptor (16 bytes)
constexpr int PIPE_THREADS = (SOLVE_WARPS + 1) * 32;

struct PipeSmem {              // per consumer warp
  char* ring;                  // lring_w bytes
  unsigned long long* full;    // PIPE_DEPTH mbarriers: record written and slice landed
  unsigned long long* empty;   // PIPE_DEPTH mbarriers: the consumer is done with the slot
  int4* rec;                   // PIPE_DEPTH x PIPE_REC_INT4
};
__device__ __forceinline__ PipeSmem pipe_smem(char* base, int lring_w, int w) {
  PipeSmem sm;
  sm.ring = base + (size_t)w * lring_w;
  char* q = base + (size_t)SOLVE_WARPS * lring_w;
  sm.full = reinterpret_cast<unsigned long long*>(q) + 2 * PIPE_DEPTH * w;
  sm.empty = sm.full + PIPE_DEPTH;
  q += SOLVE_WARPS * 2 * PIPE_DEPTH * 8;
  sm.rec = reinterpret_cast<int4*>(q) + PIPE_DEPTH * PIPE_REC_INT4 * w;
  return sm;
}
constexpr size_t pipe_smem_misc() { return (size_t)SOLVE_WARPS * (2 * PIPE_DEPTH * 8 + PIPE_DEPTH * PIPE_REC_INT4 * 16); }

__device__ __forceinline__ void consumer_sync() {      // CTA barrier of the 16 consumer warps (the producer is not part of it)
  asm volatile("bar.sync 1, %0;" ::"n"(SOLVE_WARPS * 32) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_test(unsigned long long* bar, unsigned parity) {
  unsigned ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok)
               : "r"(smem_u32(bar)), "r"(parity)
               : "memory");
  return ok != 0;
}

// the part of tile (tr, height th_) that warp `slice` of `ws` multiplies: first reduction index, count, leading dimension
// (rows of a forward row tile / pivot columns of a backward column tile) and the offset of the run in sfwd / sbwd;
// bm = SolveArgs::blk_mask (the reduction ranges of tile_compute)
struct SliceDesc {
  int64_t off;
  int r0, len, ld;
};
__device__ __forceinline__ SliceDesc slice_of(const TileRec& tr, int dir, int th_, int slice, int ws, int bm) {
  const int nc = tr.nc, f = tr.nc + tr.nb, o0 = tr.tile * th_;
  SliceDesc s;
  if (dir == 0) {
    const int cend = min(nc, (o0 + th_ + bm) & ~bm);
    const int per = solve_slice_len(cend, ws);
    s.r0 = min(cend, slice * per);
    s.len = min(cend, s.r0 + per) - s.r0;
    s.ld = min(th_, f - o0);
    s.off = tr.soff + (int64_t)o0 * nc + (int64_t)s.r0 * s.ld;
  } else {
    const int ob = o0 & ~bm;
    const int per = solve_slice_len(f - ob, ws);
    s.r0 = min(f, ob + slice * per);
    s.len = min(f, s.r0 + per) - s.r0;
    s.ld = min(th_, nc - o0);
    s.off = tr.soff + (int64_t)o0 * f + (int64_t)s.r0 * s.ld;
  }
  return s;
}

// tile of consumer warp w in (level phase ph, CTA-tile index ct), or -1
__device__ __forceinline__ int pipe_tile_of(const PhaseRec& ph, int ct, int w) {
  const int tpc = SOLVE_WARPS / ph.ws;
  const int te = ct * tpc + w / ph.ws;
  return te < ph.ntiles ? te : -1;
}

// The producer warp.  Lane w < SOLVE_WARPS serves consumer warp w; all lanes run the same non-blocking loop (a lane
// that cannot advance -- all its slots in use, or no room in the ring yet -- simply tries again), so lanes never wait
// for each other's consumers.
template <class PhaseFn>
__device__ __forceinline__ void pipe_producer(const SolveArgs& a, char* pipe_base, int lane, PhaseFn phase) {
  const int w = lane;
  const bool active = w < SOLVE_WARPS;
  const PipeSmem sm = pipe_smem(pipe_base, a.lring_w, active ? w : 0);
  // cursor over this consumer warp's tiles: (phase, CTA-tile index); lp >= p_end: exhausted
  int lp = a.p_begin, lct = blockIdx.x;
  auto skip = [&]() {
    while (lp < a.p_end) {
      if (pipe_tile_of(phase(lp), lct, w) >= 0) return;   // (te grows with ct: no later ct of this phase has a tile either)
      ++lp;
      lct = blockIdx.x;
    }
  };
  if (!active) lp = a.p_end;
  skip();
  int islot = 0, rslot = 0;            // slot of the next tile to produce / of the oldest tile not known to be released
  unsigned ipar = 0, rpar = 0;         // phase parity of those slots' barriers
  int live = 0;                        // tiles produced and not known to be released
  int last_end = 0;                    // end of the newest ring allocation
  int qoff[PIPE_DEPTH], qlen[PIPE_DEPTH];
#pragma unroll
  for (int d = 0; d < PIPE_DEPTH; ++d) { qoff[d] = -1; qlen[d] = 0; }
  bool loaded = false;
  int4 r0 = make_int4(0, 0, 0, 0), r1 = r0, r2 = r0, r3 = r0, r4 = r0;
  SliceDesc sd;
  sd.off = 0; sd.r0 = sd.len = sd.ld = 0;
  int bytes = 0, dir = 0;
  while (__any_sync(0xffffffffu, lp < a.p_end)) {
    // one release per round is enough: the consumers take thousands of cycles per tile
    if (live > 0 && mbar_test(&sm.empty[rslot], rpar)) {
#pragma unroll
      for (int d = 0; d < PIPE_DEPTH; ++d)
        if (d == rslot) qoff[d] = -1;
      --live;
      if (++rslot == PIPE_DEPTH) { rslot = 0; rpar ^= 1u; }
    }
    if (lp < a.p_end && live < PIPE_DEPTH) {
      if (!loaded) {
        const PhaseRec ph = phase(lp);
        const int te = pipe_tile_of(ph, lct, w);
        const int4* tp = reinterpret_cast<const int4*>(a.tiles + ph.tile_off + te);
        const int4* dp = reinterpret_cast<const int4*>(a.deps + ph.tile_off + te);
        r0 = __ldg(tp); r1 = __ldg(tp + 1); r2 = __ldg(tp + 2);
        r3 = __ldg(dp); r4 = __ldg(dp + 1);
        dir = ph.dir;
        sd = slice_of(unpack_tile(r0, r1, r2), dir, (int)ph.pad, w % ph.ws, ph.ws, a.blk_mask);
        bytes = (sd.len * sd.ld * 8 + 15) & ~15;
        loaded = true;
      }
      int off;
      bool clash = false;
      if (bytes == 0) off = -2;                                 // empty slice: nothing to copy
      else if (bytes > a.lring_w) off = -1;      // larger than the ring: the tile reads it from global memory
      else {
        off = (last_end + 127) & ~127;
        if (off + bytes > a.lring_w) off = 0;
#pragma unroll
        for (int d = 0; d < PIPE_DEPTH; ++d)
          if (qoff[d] >= 0 && off < qoff[d] + qlen[d] && qoff[d] < off + bytes) clash = true;
      }
      if (!clash) {
        int4* rec = sm.rec + islot * PIPE_REC_INT4;
        rec[0] = r0; rec[1] = r1; rec[2] = r2; rec[3] = r3; rec[4] = r4;
        rec[5] = make_int4(sd.r0, sd.len, sd.ld, off);
        if (off >= 0) {
          bulk_load(sm.ring + off, (dir == 0 ? a.sfwd : a.sbwd) + sd.off, (unsigned)bytes, &sm.full[islot]);
          last_end = off + bytes;
        } else {
          mbar_arrive(&sm.full[islot]);
        }
#pragma unroll
        for (int d = 0; d < PIPE_DEPTH; ++d)
          if (d == islot) { qoff[d] = off; qlen[d] = bytes; }
        ++live;
        if (++islot == PIPE_DEPTH) { islot = 0; ipar ^= 1u; }
        loaded = false;
        lct += gridDim.x;
        skip();
      }
    }
  }
  (void)ipar;
}

// the products of one warp tile with its panel slice in shared memory (sbuf: the slice, leading dimension ld)
template <int KT, int TH, class WaitFn>
__device__ __forceinline__ void tile_compute_smem(const SolveArgs& a, int dir, bool use_perm, const TileRec& tr, int lane,
                                                  int slice, int sr0, int slen, int sld, const double* sbuf, double* stage,
                                                  double* acc, WaitFn& wait) {
  constexpr int nks = 32 / TH;
  const int nc = tr.nc, f = tr.nc + tr.nb;
  const int o0 = tr.tile * TH;
  const int g = lane / TH;
  const int out = o0 + (lane % TH);
  const double* mp = sbuf + min(lane % TH, sld - 1) + g * sld;
  const int step = nks * sld;
  for (int cc = 0; cc < slen; cc += 32) {
    const int ncol = min(32, slen - cc);
    double v[KT];
#pragma unroll
    for (int r = 0; r < KT; ++r) v[r] = 0.0;
    wait(lane);
    if (lane < ncol) {
      const int c = sr0 + cc + lane;
      if (dir == 0) fwd_operand<KT>(a, use_perm, tr, c, v);
      else bwd_operand<KT>(a, tr, c, v);
    }
    // forward: the children's updates of this output row go straight into the sum (requested together with the operands;
    // slice 0 always has a first chunk: its range starts at column 0)
    if (dir == 0 && cc == 0 && slice == 0 && lane < TH && out >= nc && out < f) child_add<KT>(a, tr.w_off + out, tr.link, acc);
#pragma unroll
    for (int r = 0; r < KT; ++r) stage[r * 32 + lane] = v[r];
    __syncwarp();
    const double* mc = mp + (int64_t)cc * sld;
    const int nj = (ncol + nks - 1) / nks;
#pragma unroll 8
    for (int j = 0; j < nj; ++j) {
      const int col = g + j * nks;
      const double m = col < ncol ? mc[j * step] : 0.0;
#pragma unroll
      for (int r = 0; r < KT; ++r) acc[r] = fma(m, stage[r * 32 + (col & 31)], acc[r]);
    }
    __syncwarp();
  }
  wait(lane);
  group_reduce<KT, TH>(acc);
}

struct ConsumerState {
  int slot;          // slot of this warp's next tile
  unsigned par;      // parity of that slot's barriers
};

// One level phase on the consumer side of the panel pipeline (KT <= 2): as level_phase, but the tile's record,
// dependencies and slice descriptor come from the warp's current slot and the panel slice from its shared-memory ring.
template <int KT, int TH>
__device__ __forceinline__ void level_phase_pipe(const SolveArgs& a, const PhaseRec& ph, int p, bool use_perm, int lane, int warp,
                                                 double* stage, double* part, ConsumerState& cs, const PipeSmem& sm) {
  const int dir = ph.dir, ws = ph.ws, ntiles = ph.ntiles;
  const int lws = __ffs(ws) - 1;                            // ws is a power of two <= SOLVE_WARPS (pick_ws): no divisions here
  const int ltpc = 4 - lws, tpc = 1 << ltpc;
  static_assert(SOLVE_WARPS == 16, "level_phase_pipe: log2(SOLVE_WARPS) == 4");
  const int sub = warp >> lws, slice = warp & (ws - 1);
  const int nct = (ntiles + tpc - 1) >> ltpc;
  for (int ct = blockIdx.x; ct < nct; ct += gridDim.x) {
    const int te = (ct << ltpc) + sub;
    const bool have = te < ntiles;
    double acc[KT];
#pragma unroll
    for (int r = 0; r < KT; ++r) acc[r] = 0.0;
    TileRec tr{};
    DepWait dw{a.cnt, a.dep_ovf, a.epoch, TileDep{}, false};
    StoreOps sto{};
    const bool tr_on = a.trace && blockIdx.x == 0 && ct == (int)blockIdx.x && threadIdx.x == 0;
    const bool sk_on = a.skew && threadIdx.x == 0 && ct == (int)blockIdx.x && have;
    unsigned long long* sk = a.skew + ((size_t)p * gridDim.x + blockIdx.x) * 4;
    auto gtime = [] { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; };
    if (have) {
      if (tr_on) a.trace[16 * p + 0] = clock64();
      if (sk_on) sk[0] = gtime();
      mbar_wait(&sm.full[cs.slot], cs.par);                 // record written, panel slice landed
      const int4* r = sm.rec + cs.slot * PIPE_REC_INT4;
      tr = unpack_tile(r[0], r[1], r[2]);
      const int4 sl = r[5];
      dw.arm(r[3], r[4]);
      if (slice == 0) sto = tile_store_request<TH>(a, dir, tr, lane);
      if (a.trace || a.skew) {      // trace builds of the chain: wait first so that the segments separate
        if (tr_on) a.trace[16 * p + 6] = clock64();
        if (sk_on) sk[1] = gtime();
        dw(lane);
        if (tr_on) a.trace[16 * p + 1] = clock64();
        if (sk_on) sk[2] = gtime();
      }
      // the slice: in the warp's ring, or (larger than the ring, rare) where it lies in global memory -- same code,
      // generic loads
      const double* sbuf = reinterpret_cast<const double*>(sm.ring + max(sl.w, 0));
      if (sl.w == -1) sbuf = (dir == 0 ? a.sfwd : a.sbwd) + slice_of(tr, dir, TH, slice, ws, a.blk_mask).off;
      tile_compute_smem<KT, TH>(a, dir, use_perm, tr, lane, slice, sl.x, sl.y, sl.z, sbuf, stage, acc, dw);
      __syncwarp();                 // every lane is done with the slot
      if (lane == 0) mbar_arrive(&sm.empty[cs.slot]);
      if (++cs.slot == PIPE_DEPTH) { cs.slot = 0; cs.par ^= 1u; }
      if (tr_on) a.trace[16 * p + 2] = clock64();
    }
    if (ws > 1) reduce_slices<KT>(acc, part, warp, lane, ws, have && slice == 0, [] { consumer_sync(); });
    if (tr_on) a.trace[16 * p + 3] = clock64();
    if (have && slice == 0) {
      tile_store_with<KT, TH>(a, dir, tr, lane, acc, sto);
      if (tr_on) a.trace[16 * p + 4] = clock64();
      signal_done(a.cnt + dw.td.self);
      if (tr_on) a.trace[16 * p + 5] = clock64();
      if (sk_on) sk[3] = gtime();
    }
    if (ws > 1) consumer_sync();
    if (tr_on) a.trace[16 * p + 7] = clock64();
  }
}

// The phases [a.p_begin, a.p_end) as one persistent cooperative kernel.  Level phases follow each other WITHOUT a
// grid barrier: tiles are handed out in a fixed global order (phase by phase, CTA-strided inside a phase), every CTA
// walks its share in that order, and a tile spins only on the completion counters of the fronts it reads from
// (TileDep).  A dependency always lies earlier in the global order and all CTAs are co-resident (cooperative
// launch), so the earliest unfinished tile can always run: no deadlock.
// The one- and two-column solves of the eigensolver run the producer / consumer form (17 warps at 96 registers: the
// tiles keep no panel entries in registers; measured 228 -> 218 us and 296 -> 285 us at C2); that is too few
// registers for wider tiles (k = 4: 306 -> 330 us), which run 16 warps that read the tile-major panels themselves.
template <int KT>
__global__ void __launch_bounds__(KT <= 2 ? PIPE_THREADS : SOLVE_WARPS * 32, 1) solve_kernel(SolveArgs a) {
  constexpr bool pipe = KT <= 2;      // panel pipeline (producer warp + shared-memory rings)
  extern __shared__ double smem[];
  __shared__ PhaseRec s_phase[MAX_PHASES_SMEM];
  __shared__ int4 s_next[pipe ? 1 : SOLVE_WARPS][5];       // first tile record + dependencies of the next phase, per warp
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int NT = SOLVE_WARPS * 32;                      // consumer threads (the whole CTA without the pipeline)
  double* stage = smem + (warp % SOLVE_WARPS) * (32 * KT);  // [KT][32] per warp
  double* part = smem + SOLVE_WARPS * 32 * KT;              // [SOLVE_WARPS][KT][32] partial sums
  // panel pipeline: per-warp rings | full / empty mbarriers | slot records, behind the partial sums
  char* pipe_base = reinterpret_cast<char*>(smem + 2 * SOLVE_WARPS * 32 * KT);
  PipeSmem sm;
  sm.ring = nullptr; sm.full = sm.empty = nullptr; sm.rec = nullptr;
  if constexpr (pipe) {
    sm = pipe_smem(pipe_base, a.lring_w, warp % SOLVE_WARPS);
    if (warp < SOLVE_WARPS && lane < 2 * PIPE_DEPTH) mbar_init(&sm.full[lane], 1);   // full[0..D) and empty[0..D) are adjacent
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  unsigned long long target = a.bar_base;
  if (a.times && blockIdx.x == 0 && threadIdx.x == 0 && a.p_begin == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    a.times[0] = t;
  }
  {
    const int4* src = reinterpret_cast<const int4*>(a.phases);
    int4* dst = reinterpret_cast<int4*>(s_phase);
    for (int e = threadIdx.x; e < 2 * min(a.nphases, MAX_PHASES_SMEM); e += blockDim.x) dst[e] = __ldg(src + e);
  }
  __syncthreads();
  auto phase_of = [&](int p) { return p < MAX_PHASES_SMEM ? s_phase[p] : a.phases[p]; };
  if constexpr (pipe) {
    if (warp == SOLVE_WARPS) {          // the producer warp: streams records and panel slices, then leaves
      pipe_producer(a, pipe_base, lane, phase_of);
      return;
    }
  }
  auto cta_sync = [&]() {
    if constexpr (pipe) consumer_sync();
    else __syncthreads();
  };
  ConsumerState cs;
  cs.slot = 0;
  cs.par = 0u;
  bool have_next = false;                                  // s_next[warp] holds this warp's first tile of phase p
  for (int p = a.p_begin; p < a.p_end; ++p) {
    if (a.trace && blockIdx.x == 0 && threadIdx.x == 0) a.trace[16 * p + 8] = clock64();
    const PhaseRec ph = p < MAX_PHASES_SMEM ? s_phase[p] : a.phases[p];
    const bool use_perm = (p == 0);
    // request this warp's first tile record of the NEXT phase now (static schedule): the load completes
    // behind this phase's work instead of in front of the next phase's
    bool nxt_have = false;
    int4 nxt = make_int4(0, 0, 0, 0);
    if (!pipe && p + 1 < a.p_end) {
      const PhaseRec nx = (p + 1) < MAX_PHASES_SMEM ? s_phase[p + 1] : a.phases[p + 1];
      const int te = (int)blockIdx.x * (SOLVE_WARPS / nx.ws) + warp / nx.ws;
      if (te < nx.ntiles) {
        nxt_have = true;
        if (lane < 3) nxt = __ldg(reinterpret_cast<const int4*>(a.tiles + nx.tile_off + te) + lane);
        else if (lane < 5) nxt = __ldg(reinterpret_cast<const int4*>(a.deps + nx.tile_off + te) + (lane - 3));
      }
    }
    // without subtree phases, phase 0 gathers B through perm itself and writes the permuted copy that the later phases
    // read; the grid barrier behind it makes the copy complete for them
    const bool bar_after = p == 0 && a.p_end > 1;
    if (bar_after) permute_rhs(a, (int64_t)blockIdx.x * NT + threadIdx.x, (int64_t)gridDim.x * NT);
    const int th_ = (int)ph.pad;
    if constexpr (pipe) {
      if (a.trace && blockIdx.x == 0 && threadIdx.x == 0) a.trace[16 * p + 9] = clock64();
      if (th_ == 8) level_phase_pipe<KT, 8>(a, ph, p, use_perm, lane, warp, stage, part, cs, sm);
      else if (th_ == 16) level_phase_pipe<KT, 16>(a, ph, p, use_perm, lane, warp, stage, part, cs, sm);
      else level_phase_pipe<KT, SOLVE_TILE>(a, ph, p, use_perm, lane, warp, stage, part, cs, sm);
    } else {
      if (th_ == 8) level_phase<KT, 8>(a, ph, p, use_perm, lane, warp, stage, part, have_next, s_next);
      else if (th_ == 16) level_phase<KT, 16>(a, ph, p, use_perm, lane, warp, stage, part, have_next, s_next);
      else level_phase<KT, SOLVE_TILE>(a, ph, p, use_perm, lane, warp, stage, part, have_next, s_next);
    }
    if constexpr (!pipe) {
      // ---- hand the prefetched first tile record of the next phase to the whole warp
      have_next = nxt_have;
      if (nxt_have && lane < 5) s_next[warp][lane] = nxt;
      __syncwarp();
    }
    if (bar_after) {
      target += gridDim.x;
      cta_sync();
      grid_barrier_arrive_wait(a.barrier, target);
      cta_sync();
    }
    if (a.times && blockIdx.x == 0 && threadIdx.x == 0) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
      a.times[p + 1] = t;
    }
  }
}

template <class T>
int upload_vec(SymDevHolder* h, const std::vector<T>& v, T** out) {
  void* p = nullptr;
  size_t bytes = std::max<size_t>(v.size(), 1) * sizeof(T);
  EIGD_CUDA(cudaMalloc(&p, bytes));
  h->allocs.push_back(p);
  if (!v.empty()) EIGD_CUDA(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  *out = (T*)p;
  return 0;
}

struct KernelCfg {
  bool ready = false;
  int grid = 0;
  size_t smem = 0;      // cooperative level kernel: staging + partial sums (+ for KT <= 2 the panel rings, mbarriers
                        // and record slots of the panel pipeline)
  int lring_w = 0;      // panel ring bytes per warp in the level kernel (KT <= 2)
  size_t smem_sub = 0;  // subtree kernel: staging + panel ring + mbarriers + front records
  int ring_w = 0;       // panel ring bytes per warp
  int rec_cap = 0;      // front records staged in shared memory
};
KernelCfg g_cfg[8];
int g_num_sms = 0;

template <int KT>
int configure(int slot) {
  KernelCfg& c = g_cfg[slot];
  if (c.ready) return 0;
  const size_t stage_b = (size_t)SOLVE_WARPS * 32 * KT * 8;
  c.smem = 2 * stage_b;
  if (KT <= 2) {
    // panel pipeline of the level kernel: what is left of the 227 KB per CTA after the staging / partial-sum arrays,
    // the kernel's static shared memory (phase records, first-tile records) and the pipeline's own bookkeeping
    cudaFuncAttributes fa;
    EIGD_CUDA(cudaFuncGetAttributes(&fa, solve_kernel<KT>));
    const size_t misc = pipe_smem_misc();
    const size_t budget = 227 * 1024 - fa.sharedSizeBytes - 1024;
    size_t ring = budget > c.smem + misc ? (budget - c.smem - misc) / SOLVE_WARPS : 0;
    ring = std::min<size_t>(ring, 16384) / 256 * 256;
    if (ring < 2048) { eigd_set_error("solve: the panel rings of the level kernel do not fit in shared memory"); return 5; }
    c.lring_w = (int)ring;
    c.smem += (size_t)SOLVE_WARPS * c.lring_w + misc;
  }
  EIGD_CUDA(cudaFuncSetAttribute(solve_kernel<KT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c.smem));
  int occ = 0;
  EIGD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, solve_kernel<KT>, KT <= 2 ? PIPE_THREADS : SOLVE_WARPS * 32,
                                                          c.smem));
  if (occ < 1) { eigd_set_error("solve: kernel does not fit on an SM"); return 5; }
  // subtree kernel: staging [NW][KT][32] | panel ring | mbarriers + copy queue | front records; 227 KB per CTA on sm_100a
  constexpr int NW = SOLVE_WARPS;
  const size_t stage_s = (size_t)NW * 32 * KT * 8;
  const size_t budget = 227 * 1024 - 1024;
  c.rec_cap = KT <= 4 ? 512 : 256;
  size_t ring = (budget - stage_s - 2 * FRONT_DEPTH * NW * 8 - (size_t)c.rec_cap * 48) / NW;
  ring = std::min<size_t>(ring, 16384) / 256 * 256;   // the launches that stage no operands use FRONT_PANEL_MAX of it
  c.ring_w = (int)ring;
  c.smem_sub = stage_s + ring * NW + 2 * FRONT_DEPTH * NW * 8 + (size_t)c.rec_cap * 48;
  EIGD_CUDA(cudaFuncSetAttribute(subtree_kernel<KT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c.smem_sub));
  c.grid = g_num_sms;
  c.ready = true;
  return 0;
}

template <int KT>
int launch_solve(int slot, eigd_factor* f, SolveArgs& a) {
  int rc = configure<KT>(slot);
  if (rc) return rc;
  const KernelCfg& c = g_cfg[slot];
  const std::vector<PhaseRec>& hp = f->h->solve.host_phases;
  const int np = a.nphases;
  a.barrier = f->barrier;
  a.cnt = f->cnt;
  a.deps = f->h->solve.deps;
  a.dep_ovf = f->h->solve.dep_ovf;
  a.lring_w = c.lring_w;
  a.rec_cap = c.rec_cap;
  // the subtree phases (a plan with a cut: the first and the last phase) run as their own launches in front of / behind
  // the cooperative level kernel
  const bool sub = np >= 2 && hp[0].ws == 0;
  a.p_begin = sub ? 1 : 0;
  a.p_end = sub ? np - 1 : np;
  a.bar_base = f->bar_base;
  a.epoch = 0;
  // a subtree launch that stages operands in its ring (the backward one for KT >= 2, the forward one for KT = 2) gets the
  // whole ring; the others only hold panels, which FRONT_PANEL_MAX bounds, and leave the rest of the SM's shared memory
  // to L1
  auto subtree_launch = [&](int p, bool staged) -> int {
    a.ring_w = staged ? c.ring_w : std::min(c.ring_w, FRONT_PANEL_MAX);
    const size_t smem = c.smem_sub - (size_t)SOLVE_WARPS * (c.ring_w - a.ring_w);
    subtree_kernel<KT><<<hp[p].level, SOLVE_WARPS * 32, smem, g_eigd_stream>>>(a, p);
    EIGD_CUDA(cudaGetLastError());
    ++g_eigd_launches;
    return 0;
  };
  if (sub && (rc = subtree_launch(0, FWD_STAGE<KT>))) return rc;
  if (a.p_end > a.p_begin) {
    a.epoch = ++f->epoch;            // one epoch per cooperative launch: the completion counters never reset
    // the one grid barrier: behind phase 0 of a plan without subtree phases (solve_kernel)
    const int nbar = a.p_begin == 0 && a.p_end > 1 ? 1 : 0;
    void* params[] = {(void*)&a};
    EIGD_CUDA(cudaLaunchCooperativeKernel((void*)solve_kernel<KT>, dim3(c.grid), dim3(KT <= 2 ? PIPE_THREADS : SOLVE_WARPS * 32),
                                          params, c.smem, g_eigd_stream));
    ++g_eigd_launches;
    f->bar_base += (unsigned long long)nbar * (unsigned long long)c.grid;
  }
  if (sub && (rc = subtree_launch(np - 1, KT >= 2))) return rc;
  return 0;
}

// Y = X + s Y on n x k strided operands, s = -1 (residual b - r) or +1 (update dx + x): one rounding per element, so the
// results are fl(b - r) and fl(x + dx)
__global__ void refine_xpsy_kernel(int64_t n, int k, const double* __restrict__ X, int64_t xrs, int64_t xcs, double s,
                                   double* __restrict__ Y, int64_t yrs, int64_t ycs) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n * k; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t i; int c;
    if (ycs == 1) { i = e / k; c = (int)(e - i * k); } else { c = (int)(e / n); i = e - (int64_t)c * n; }
    Y[i * yrs + c * ycs] = X[i * xrs + c * xcs] + s * Y[i * yrs + c * ycs];
  }
}

}  // namespace

int build_solve_plan_dev(eigd_symbolic* S, SymDevHolder* h) {
  if (!g_num_sms) {
    int dev = 0;
    EIGD_CUDA(cudaGetDevice(&dev));
    EIGD_CUDA(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  SolvePlanHost P;
  build_solve_plan_host(S, g_num_sms * SOLVE_WARPS, g_num_sms, -2, P);
  SolvePlanDev& d = h->solve;
  int rc = 0;
  rc |= upload_vec(h, P.tiles, &d.tiles);
  rc |= upload_vec(h, P.deps, &d.deps);
  rc |= upload_vec(h, P.dep_ovf, &d.dep_ovf);
  rc |= upload_vec(h, P.phases, &d.phases);
  rc |= upload_vec(h, P.ovf_row, &d.ovf_row);
  rc |= upload_vec(h, P.ovf, &d.ovf);
  rc |= upload_vec(h, P.sub_ptr, &d.sub_ptr);
  rc |= upload_vec(h, P.th_fwd, &h->d.th_f);     // storage form of every front's solve panels (panel_build_kernel)
  rc |= upload_vec(h, P.th_bwd, &h->d.th_b);
  d.nphases = (int)P.phases.size();
  d.host_phases = P.phases;
  return rc;
}

void free_solve_plan_dev(SymDevHolder*) {}   // the arrays are owned by SymDevHolder::allocs

// ---- live timing of every solve launch (bench.py roofline): CUDA events on the launching stream ----------
struct SolveTiming {
  cudaEvent_t e0, e1;
  int k;
};
static bool g_timing_on = false;
static std::vector<SolveTiming> g_timings;

extern "C" int eigd_solve_timing_begin(void) {
  for (auto& t : g_timings) { cudaEventDestroy(t.e0); cudaEventDestroy(t.e1); }
  g_timings.clear();
  g_timing_on = true;
  return 0;
}

// calls_by_k / ms_by_k: 33 entries each (index = number of right-hand sides of the launch, 1 .. 32)
extern "C" int eigd_solve_timing_end(int64_t* calls_by_k, double* ms_by_k) {
  g_timing_on = false;
  for (int i = 0; i < 33; ++i) { calls_by_k[i] = 0; ms_by_k[i] = 0.0; }
  for (auto& t : g_timings) {
    EIGD_CUDA(cudaEventSynchronize(t.e1));
    float ms = 0.f;
    EIGD_CUDA(cudaEventElapsedTime(&ms, t.e0, t.e1));
    int k = t.k < 32 ? t.k : 32;
    calls_by_k[k] += 1;
    ms_by_k[k] += ms;
    cudaEventDestroy(t.e0);
    cudaEventDestroy(t.e1);
  }
  g_timings.clear();
  return 0;
}

// developer profiling hook: device buffer of (nphases + 1) u64 receiving per-phase timestamps of the next solves
static unsigned long long* g_phase_times = nullptr;
static long long* g_trace = nullptr;
static unsigned long long* g_skew = nullptr;
extern "C" int eigd_solve_set_phase_times(void* d_buf) { g_phase_times = (unsigned long long*)d_buf; return 0; }
// developer profiling: device buffer of 16 * nphases i64 (see SolveArgs::trace)
extern "C" int eigd_solve_set_trace(void* d_buf) { g_trace = (long long*)d_buf; return 0; }
// developer profiling: device buffer of 4 * nphases * (number of SMs) u64 (see SolveArgs::skew)
extern "C" int eigd_solve_set_skew(void* d_buf) { g_skew = (unsigned long long*)d_buf; return 0; }
extern "C" int eigd_solve_num_phases(const eigd_factor* f) { return f->h->solve.nphases; }

extern "C" int eigd_factor_solve(eigd_factor* f, const double* B, int64_t brs, int64_t bcs, double* X, int64_t xrs,
                                 int64_t xcs, int k) {
  if (k < 1) return 0;
  SymDevHolder* h = f->h;
  const int kmax = std::min(f->max_rhs, 16);
  // balanced chunks of at most kmax columns (20 columns -> 10 + 10, not 16 + 4)
  const int nchunks = (k + kmax - 1) / kmax;
  const int per = (k + nchunks - 1) / nchunks;
  for (int c0 = 0; c0 < k; c0 += per) {
    const int kc = std::min(per, k - c0);
    SolveArgs a;
    a.tiles = h->solve.tiles;
    a.phases = h->solve.phases;
    a.nphases = h->solve.nphases;
    a.ovf_row = h->solve.ovf_row;
    a.ovf = h->solve.ovf;
    a.sub_ptr = h->solve.sub_ptr;
    a.perm = h->d.perm;
    a.sn_rows = h->d.sn_rows;
    a.rel = h->d.rel;
    a.sumf = f->sym->w_off[f->sym->nsuper];
    a.slab_stride = a.sumf * kmax;
    a.bperm = f->bperm;
    a.n = f->sym->n;
    a.sfwd = f->sfwd;
    a.sbwd = f->sbwd;
    a.dinv = f->dinv;
    a.wbuf = f->wbuf;
    a.ybuf = f->ybuf;
    a.xperm = f->xperm;
    a.B = B + (int64_t)c0 * bcs;
    a.brs = brs;
    a.bcs = bcs;
    a.X = X + (int64_t)c0 * xcs;
    a.xrs = xrs;
    a.xcs = xcs;
    a.k = kc;
    a.blk_mask = f->pivoting ? 31 : 0;
    a.times = g_phase_times;
    a.trace = g_trace;
    a.skew = g_skew;
    int rc;
    SolveTiming tm;
    if (g_timing_on) {
      tm.k = kc;
      EIGD_CUDA(cudaEventCreate(&tm.e0));
      EIGD_CUDA(cudaEventCreate(&tm.e1));
      EIGD_CUDA(cudaEventRecord(tm.e0, g_eigd_stream));
    }
    if (kc == 1) rc = launch_solve<1>(0, f, a);
    else if (kc == 2) rc = launch_solve<2>(1, f, a);
    else if (kc <= 4) rc = launch_solve<4>(2, f, a);
    else if (kc <= 6) rc = launch_solve<6>(3, f, a);
    else if (kc <= 8) rc = launch_solve<8>(4, f, a);
    else if (kc <= 10) rc = launch_solve<10>(5, f, a);
    else if (kc <= 12) rc = launch_solve<12>(6, f, a);
    else rc = launch_solve<16>(7, f, a);
    if (rc) return rc;
    if (g_timing_on) {
      EIGD_CUDA(cudaEventRecord(tm.e1, g_eigd_stream));
      g_timings.push_back(tm);
    }
  }
  return 0;
}

// ---- iterative refinement x += F (b - A x) against the matrix registered with eigd_factor_set_refinement ----------
extern "C" int eigd_factor_set_refinement(eigd_factor* f, int steps, const int* d_indptr, const int* d_indices,
                                          const double* d_vals, double* d_work, int work_cols) {
  if (steps < 0 || work_cols < 0 || (steps > 0 && (!d_indptr || !d_indices || !d_vals)) || (work_cols > 0 && !d_work)) {
    eigd_set_error("factor_set_refinement: a refinement depth needs the matrix, a scratch width needs the scratch");
    return 7;
  }
  f->refine = {steps, work_cols, d_indptr, d_indices, d_vals, d_work};
  return 0;
}

extern "C" int eigd_factor_apply(eigd_factor* f, const double* B, int64_t brs, int64_t bcs, double* X, int64_t xrs,
                                 int64_t xcs, int k) {
  const auto& r = f->refine;
  if (r.steps == 0 || k < 1) return eigd_factor_solve(f, B, brs, bcs, X, xrs, xcs, k);
  if (k > r.cols) { eigd_set_error("factor_apply: %d right-hand sides, but the refinement scratch holds %d", k, r.cols); return 7; }
  const int n = f->sym->n;
  // the residual R (and the copy of B) are laid out like X, so that every element-wise pass is coalesced on both sides
  const int64_t rrs = xcs == 1 ? k : 1, rcs = xcs == 1 ? 1 : n;
  double* R = r.work;
  const int g = (int)std::min<int64_t>(((int64_t)n * k + 255) / 256, 148 * 8);     // grid of the element-wise passes
  int rc;
  if (X == B) {                                           // the solve overwrites B, which every residual needs
    if ((rc = eigd_copy2d(n, k, B, brs, bcs, R + (int64_t)n * k, rrs, rcs))) return rc;
    B = R + (int64_t)n * k, brs = rrs, bcs = rcs;
  }
  if ((rc = eigd_factor_solve(f, B, brs, bcs, X, xrs, xcs, k))) return rc;
  for (int it = 0; it < r.steps; ++it) {
    // k == 1 stays a one-column product (spmv_kernel): its summation order differs from the multi-column kernel's
    if ((rc = eigd_csr_spmm(n, r.indptr, r.indices, r.vals, X, xrs, xcs, R, rrs, rcs, k, 1.0, 0.0))) return rc;
    EIGD_LAUNCH(refine_xpsy_kernel, g, 256, 0, (int64_t)n, k, B, brs, bcs, -1.0, R, rrs, rcs);     // R = B - A X
    EIGD_CHECK_LAUNCH();
    if ((rc = eigd_factor_solve(f, R, rrs, rcs, R, rrs, rcs, k))) return rc;                    // dX = F R, in place
    EIGD_LAUNCH(refine_xpsy_kernel, g, 256, 0, (int64_t)n, k, R, rrs, rcs, 1.0, X, xrs, xcs);      // X = dX + X
    EIGD_CHECK_LAUNCH();
  }
  return 0;
}
