// Host-built execution plan of the persistent triangular-solve kernel (solve.cu).
// No reference counterpart: the reference calls SuperLU.solve once per right-hand side
// (eigd/eigenvector_derivatives.py:18-23).  See DESIGN.md "Triangular solves".
#pragma once
#include <cstdint>
#include <vector>

#include "symbolic.hpp"

constexpr int SOLVE_WARPS = 16;   // warps per CTA of the solve kernel
constexpr int SOLVE_TILE = 32;    // outputs (front rows / pivot columns) per warp tile

// link word of a tile record: where the front's update rows go in the forward sweep
//   bits  0..47  w-row offset of the PARENT front (prefix sum of front sizes)
//   bits 48..55  slab: 0 / 1 = rank of the front among its siblings (the parent adds slab 0 + slab 1,
//                no index look-up), 2 = third or later child (own rows in slab 2, the parent
//                gathers them through the overflow lists), 255 = root (nothing to pass up)
//   bit  56      the front has children of slab 2 (its rows consult ovf_row)
//   bit  57      the front has children at all (leaves skip the slab reads)
constexpr int LINK_SLAB_SHIFT = 48;
constexpr int64_t LINK_WOFF_MASK = ((int64_t)1 << 48) - 1;
constexpr int64_t LINK_HAS_OVF = (int64_t)1 << 56;
constexpr int64_t LINK_HAS_CHILDREN = (int64_t)1 << 57;

// doubles reserved for the f x nc solve panel of a front: an even count, so that every panel starts on a
// 16-byte boundary and spans a multiple of 16 bytes (the unit of a bulk copy into shared memory)
#ifdef __CUDACC__
#define EIGD_HD __host__ __device__
#else
#define EIGD_HD
#endif
EIGD_HD inline int64_t solve_panel_doubles(int f, int nc) { return ((int64_t)f * nc + 1) & ~(int64_t)1; }

// Reduction entries per warp when ws warps split a reduction of length len: an EVEN count, so that every warp's slice
// of a tile-major panel (below) starts on a 16-byte boundary -- the unit of a bulk copy into shared memory.
EIGD_HD inline int solve_slice_len(int len, int ws) { return (((len + ws - 1) / ws) + 1) & ~1; }

// TILE-MAJOR solve panels of the fronts ABOVE the cut (level phases; PhaseRec::pad is the tile height).  With tile
// height TH (outputs per warp tile: 32, 16 or 8, chosen per level and direction) the f x nc panel S of a front is
// stored tile by tile: row tile t (rows t TH ... , th = min(TH, f - t TH) of them) occupies th * nc doubles from
// offset t TH nc, element (row r, column c) at c * th + (r - t TH).  S^T (nc x f) likewise by column tiles: tile t
// (tw = min(TH, nc - t TH) pivot columns) from offset t TH f, element (column c, front row i) at i * tw + (c - t TH).
// The part of a tile that one warp multiplies -- a contiguous range of the reduction dimension -- is then ONE
// contiguous run of doubles, which the level kernel brings into shared memory with one bulk copy, ahead of time.
// Fronts below the cut keep plain column-major panels (the subtree kernels copy whole fronts).

// One warp tile: 32 consecutive outputs of one front.  Everything the warp needs about the front
// travels in this one 48-byte record; the forward sweep needs no further index look-up before it
// can read its operands (permuted right-hand side and the two child slabs are addressed by the
// front's own offsets).
struct TileRec {
  int first, nc, nb, tile;        // first pivot column (permuted), #pivot columns, #rows below, tile index
  int64_t soff;                   // offset of the front's f x nc solve panel (same in S and S^T storage)
  int64_t w_off;                  // offset of the front in the w-row space (prefix sum of front sizes)
  int64_t row_off;                // offset of the front's below-row list in sn_rows / rel
  int64_t link;                   // see LINK_*
};
static_assert(sizeof(TileRec) == 48, "TileRec is read as three 16-byte words");

// Dependencies of one LEVEL-phase tile (same index as its TileRec).  The level phases are not separated by grid
// barriers: every front above the cut owns two completion counters (forward: 2 * sn, backward: 2 * sn + 1) that
// each finished tile of the front increments once per solve; a tile starts when the counters of the fronts it
// reads from have reached (solve epoch) x (their tile count):
//   forward  tile of front P : the forward counters of P's children above the cut (children below the cut were
//                              finished by the subtree launch that precedes the level kernel in stream order);
//   backward tile of front F : the backward counter of F's parent (which transitively covers every ancestor and
//                              the whole forward sweep); a root waits for its own forward counter.
// Two dependencies travel inline, further ones (fronts with three or more children above the cut) in dep_ovf as
// (counter, tile count) pairs starting at `ovf`.
struct TileDep {
  int self;       // counter this tile increments when its outputs are stored
  int ndep;       // number of dependencies
  int d0, n0;     // counter index / tiles per solve of dependency 0
  int d1, n1;     // ... of dependency 1
  int ovf;        // offset of dependencies 2 .. ndep-1 in SolvePlanHost::dep_ovf (pairs)
  int pad;
};
static_assert(sizeof(TileDep) == 32, "TileDep is read as two 16-byte words");

// One phase = the tiles of one level of the assembly tree in one direction.  Level phases are ordered (every CTA
// walks them in sequence) but synchronised tile by tile through TileDep, not by a grid-wide barrier.  ws warps share a tile (they split its reduction dimension).
// ws == 0 marks a SUBTREE phase: the bottom levels 0..cut of the tree are partitioned into complete
// subtrees, every subtree is owned by one CTA slot, and the slot walks its levels with CTA-local
// barriers only (no grid barrier below the cut).  For such a phase ntiles = cut + 1 (local levels),
// level = number of slots and tile_off = offset into SolvePlanHost::sub_ptr of the slot x level table.
struct PhaseRec {
  int dir, ws, ntiles, level;     // dir 0 forward, 1 backward
  int64_t tile_off;
  int64_t pad;                    // level phase: tile height (32, 16 or 8); subtree phase: 0 (one record per front,
                                  // tile field 0)
};
static_assert(sizeof(PhaseRec) == 32, "PhaseRec layout");

struct SolvePlanHost {
  std::vector<int64_t> soff;      // nsuper + 1, prefix sum of solve_panel_doubles(f, nc)
  // overflow form of the extend-add of the forward sweep (fronts with more than two children):
  // ovf_row[t] = -1, or the offset o of a list ovf[o] = count, ovf[o+1 ..] = source rows in slab 2
  std::vector<int> ovf_row;       // sum_front
  std::vector<int> ovf;
  std::vector<int> slab;          // per supernode: 0, 1, 2 or 255 (root)
  std::vector<TileRec> tiles;
  std::vector<TileDep> deps;      // parallel to tiles (all-zero for the tiles of the subtree phases)
  std::vector<int> dep_ovf;       // (counter, tile count) pairs of the third and later dependencies
  std::vector<PhaseRec> phases;   // forward phases (leaves -> root) then backward phases (root -> leaves)
  int nfwd = 0;
  int cut_level = -1;             // levels <= cut_level are executed by the subtree phases (-1: none)
  int nslots = 0;
  std::vector<int> sub_ptr;       // two tables (forward, backward) of nslots * (cut_level + 2) tile indices
  std::vector<int> sub_slot;      // owning slot of every supernode below the cut (-1 above it)
  std::vector<int> th_fwd, th_bwd;  // per supernode: tile height of its tile-major S / S^T panel, 0 = column-major
};

// target_warps: resident warps the level phases are balanced for; nslots: CTA slots of the subtree
// phases (0 disables them); cut: -2 = choose automatically, -1 = no subtree phases, >= 0 = forced
void build_solve_plan_host(const eigd_symbolic* S, int target_warps, int nslots, int cut, SolvePlanHost& P);
