// Host side of the triangular-solve plan: tile records, per-level phases, gather lists.
// Pure C++ (no CUDA) so that the plan can be checked on a machine without a GPU
// (tests/test_solve_plan.py emulates the kernel on these arrays).
#include "solve_plan.hpp"

#include <algorithm>
#include <functional>
#include <queue>

namespace {

int pick_ws(int ntiles, int redmax, int target_warps) {
  // split the reduction dimension of a tile over ws warps while (i) the level would otherwise leave
  // most resident warps idle and (ii) every warp still gets >= 8 terms
  int ws = 1;
  while (ws < SOLVE_WARPS && (int64_t)ntiles * ws * 2 <= target_warps && redmax / (2 * ws) >= 4) ws *= 2;
  return ws;
}

// Partition the levels 0..cut into complete subtrees and spread them over nslots CTA slots
// (longest-processing-time greedy on the panel sizes).  Returns max load / mean load.
double assign_subtrees(const eigd_symbolic* S, int cut, int nslots, std::vector<int>& slot_of) {
  const int ns = S->nsuper;
  std::vector<double> wsub(ns, 0.0);
  std::vector<int> roots;
  for (int k = 0; k < ns; ++k) {                       // postorder: children come before their parent
    if (S->sn_level[k] > cut) continue;
    wsub[k] += (double)sn_fsize(S, k) * sn_ncols(S, k) + 4096.0;   // panel entries + a latency charge per front
    int p = S->sn_parent[k];
    if (p >= 0 && S->sn_level[p] <= cut) wsub[p] += wsub[k];
    else roots.push_back(k);
  }
  std::sort(roots.begin(), roots.end(), [&](int a, int b) { return wsub[a] != wsub[b] ? wsub[a] > wsub[b] : a < b; });
  typedef std::pair<double, int> Load;
  std::priority_queue<Load, std::vector<Load>, std::greater<Load>> pq;
  for (int s = 0; s < nslots; ++s) pq.push(Load(0.0, s));
  slot_of.assign(ns, -1);
  double total = 0.0, maxload = 0.0;
  for (int r : roots) {
    Load l = pq.top();
    pq.pop();
    slot_of[r] = l.second;
    l.first += wsub[r];
    total += wsub[r];
    maxload = std::max(maxload, l.first);
    pq.push(l);
  }
  for (int k = ns - 1; k >= 0; --k) {                  // parents have larger indices: inherit the root's slot
    if (S->sn_level[k] > cut || slot_of[k] >= 0) continue;
    slot_of[k] = slot_of[S->sn_parent[k]];
  }
  return total > 0.0 ? maxload / (total / nslots) : 1e30;
}

}  // namespace

void build_solve_plan_host(const eigd_symbolic* S, int target_warps, int nslots, int cut_req, SolvePlanHost& P) {
  const int ns = S->nsuper;
  P.soff.assign(ns + 1, 0);
  for (int k = 0; k < ns; ++k) P.soff[k + 1] = P.soff[k] + solve_panel_doubles(sn_fsize(S, k), sn_ncols(S, k));

  // ---- child slabs and overflow lists ---------------------------------------------------------
  // children 0 and 1 of a front (ascending order) write their update rows straight into the parent's
  // rows of slab 0 / slab 1; later children keep theirs in slab 2 and the parent gathers them
  const int64_t sumf = S->w_off[ns];
  P.slab.assign(ns, 255);
  std::vector<char> has_ovf(ns, 0);
  std::vector<std::vector<int>> extra;          // per overflow row: sources in slab 2
  std::vector<int64_t> extra_of(sumf, -1);
  for (int p = 0; p < ns; ++p)
    for (int q = S->child_ptr[p]; q < S->child_ptr[p + 1]; ++q) {   // children in ascending order: fixed sum order
      int c = S->child_idx[q];
      int rank = q - S->child_ptr[p];
      P.slab[c] = rank < 2 ? rank : 2;
      if (rank < 2) continue;
      has_ovf[p] = 1;
      int ncc = sn_ncols(S, c), nbc = sn_nbelow(S, c);
      for (int i = 0; i < nbc; ++i) {
        int64_t t = S->w_off[p] + S->rel[S->sn_rowptr[c] + i];
        if (extra_of[t] < 0) { extra_of[t] = (int64_t)extra.size(); extra.emplace_back(); }
        extra[extra_of[t]].push_back((int)(S->w_off[c] + ncc + i));
      }
    }
  P.ovf_row.assign(sumf, -1);
  P.ovf.clear();
  for (int64_t t = 0; t < sumf; ++t)
    if (extra_of[t] >= 0) {
      const std::vector<int>& e = extra[extra_of[t]];
      P.ovf_row[t] = (int)P.ovf.size();
      P.ovf.push_back((int)e.size());
      P.ovf.insert(P.ovf.end(), e.begin(), e.end());
    }

  // ---- tiles and phases ---------------------------------------------------------------------
  P.tiles.clear();
  P.deps.clear();
  P.dep_ovf.clear();
  P.phases.clear();
  auto rec = [&](int k, int tile) {
    TileRec r;
    r.first = S->sn_first[k];
    r.nc = sn_ncols(S, k);
    r.nb = sn_nbelow(S, k);
    r.tile = tile;
    r.soff = P.soff[k];
    r.w_off = S->w_off[k];
    r.row_off = S->sn_rowptr[k];
    int p = S->sn_parent[k];
    r.link = (p >= 0 ? S->w_off[p] : 0) | ((int64_t)P.slab[k] << LINK_SLAB_SHIFT);
    if (has_ovf[k]) r.link |= LINK_HAS_OVF;
    if (S->child_ptr[k + 1] > S->child_ptr[k]) r.link |= LINK_HAS_CHILDREN;
    return r;
  };
  // ---- subtree phases: the largest cut whose subtrees still balance over the slots -----------
  P.cut_level = -1;
  P.nslots = nslots;
  P.sub_ptr.clear();
  P.sub_slot.assign(ns, -1);
  if (cut_req >= S->nlevels - 1) cut_req = S->nlevels - 2;
  if (cut_req >= 0 && nslots > 0) {
    assign_subtrees(S, cut_req, nslots, P.sub_slot);
    P.cut_level = cut_req;
  } else if (cut_req == -2 && nslots > 0 && S->nlevels > 2) {
    // largest cut that still leaves every slot several subtrees (>= 4 on average: the slot's warps then have
    // enough independent fronts per local level to hide latency) and balances within 25 %
    for (int cut = S->nlevels - 2; cut >= 1; --cut) {
      std::vector<int> slot_of;
      int nroots = 0;
      for (int k = 0; k < ns; ++k)
        if (S->sn_level[k] <= cut && (S->sn_parent[k] < 0 || S->sn_level[S->sn_parent[k]] > cut)) ++nroots;
      if (nroots < 4 * nslots) continue;
      if (assign_subtrees(S, cut, nslots, slot_of) <= 1.25) {
        P.cut_level = cut;
        P.sub_slot = slot_of;
        break;
      }
    }
  }
  const int cut = P.cut_level, nl = cut + 1;
  // ONE record per front in the subtree phases (front mode): a warp brings the front's whole panel into shared memory
  // with one bulk copy and runs all its row tiles from there
  auto subtree_phase = [&](int dir) {
    // tiles ordered by (slot, level); table entry [slot * (nl + 1) + l] = first tile of local level l
    std::vector<std::vector<int>> bucket((size_t)nslots * nl);
    for (int k = 0; k < ns; ++k)
      if (S->sn_level[k] <= cut) bucket[(size_t)P.sub_slot[k] * nl + S->sn_level[k]].push_back(k);
    PhaseRec ph{dir, 0, nl, nslots, (int64_t)P.sub_ptr.size(), 0};
    for (int s = 0; s < nslots; ++s) {
      for (int l = 0; l < nl; ++l) {
        P.sub_ptr.push_back((int)P.tiles.size());
        for (int k : bucket[(size_t)s * nl + l]) {
          P.tiles.push_back(rec(k, 0));
          P.deps.push_back(TileDep{0, 0, 0, 0, 0, 0, 0, 0});
        }
      }
      P.sub_ptr.push_back((int)P.tiles.size());
    }
    P.phases.push_back(ph);
  };
  if (cut >= 0) subtree_phase(0);
  // Tile height of a level phase: 32 outputs per warp tile, or 16 / 8 where a level has so few 32-output tiles that most
  // SMs would idle while a few of them stream 64 - 128 KB panel slices each (the upper levels: one to a few dozen wide
  // fronts).  With per-front completion counters instead of grid barriers a finer tiling costs no extra synchronisation.
  // (Round 1 measured a variable tile height as slower -- with a grid barrier per level and the tile-serial overheads of
  // that kernel.)
  auto count_tiles = [&](int dir, int l, int to) {
    int64_t nt = 0;
    for (int q = S->level_ptr[l]; q < S->level_ptr[l + 1]; ++q) {
      int k = S->level_sn[q];
      nt += ((dir == 0 ? sn_fsize(S, k) : sn_ncols(S, k)) + to - 1) / to;
    }
    return nt;
  };
  const int ncta = std::max(1, target_warps / SOLVE_WARPS);
  std::vector<int> height(2 * (size_t)S->nlevels, SOLVE_TILE);      // [dir * nlevels + level]
  for (int dir = 0; dir < 2; ++dir)
    for (int l = cut + 1; l < S->nlevels; ++l) {
      int to = SOLVE_TILE;
      while (to > 8 && count_tiles(dir, l, to / 2) <= ncta) to /= 2;
      height[(size_t)dir * S->nlevels + l] = to;
    }
  // the panels of the fronts above the cut are stored tile-major in their level's tile height (solve_plan.hpp)
  P.th_fwd.assign(ns, 0);
  P.th_bwd.assign(ns, 0);
  for (int k = 0; k < ns; ++k)
    if (S->sn_level[k] > cut) {
      P.th_fwd[k] = height[(size_t)0 * S->nlevels + S->sn_level[k]];
      P.th_bwd[k] = height[(size_t)1 * S->nlevels + S->sn_level[k]];
    }
  auto level_phase = [&](int dir, int l) {
    int redmax = 1;
    const int to = height[(size_t)dir * S->nlevels + l];
    for (int q = S->level_ptr[l]; q < S->level_ptr[l + 1]; ++q) {
      int k = S->level_sn[q];
      redmax = std::max(redmax, dir == 0 ? sn_ncols(S, k) : sn_fsize(S, k));
    }
    const int64_t nt = count_tiles(dir, l, to);
    const int ws = pick_ws((int)nt, redmax, target_warps);
    PhaseRec ph{dir, ws, 0, l, (int64_t)P.tiles.size(), to};
    // tiles of front k in direction d, in the tile height of ITS level's phase (completion-counter targets)
    auto ntile = [&](int k, int d) {
      const int tk = S->sn_level[k] > cut ? height[(size_t)d * S->nlevels + S->sn_level[k]] : SOLVE_TILE;
      return ((d == 0 ? sn_fsize(S, k) : sn_ncols(S, k)) + tk - 1) / tk;
    };
    for (int q = S->level_ptr[l]; q < S->level_ptr[l + 1]; ++q) {
      int k = S->level_sn[q];
      int outs = dir == 0 ? sn_fsize(S, k) : sn_ncols(S, k);
      // completion-counter dependencies of the front's tiles (see TileDep)
      std::vector<std::pair<int, int>> dl;
      if (dir == 0) {
        for (int c = S->child_ptr[k]; c < S->child_ptr[k + 1]; ++c) {
          int ch = S->child_idx[c];
          if (S->sn_level[ch] > cut) dl.emplace_back(2 * ch, ntile(ch, 0));
        }
      } else {
        int p = S->sn_parent[k];
        if (p >= 0) dl.emplace_back(2 * p + 1, ntile(p, 1));
        else dl.emplace_back(2 * k, ntile(k, 0));
      }
      TileDep td{2 * k + dir, (int)dl.size(), 0, 0, 0, 0, 0, 0};
      if (dl.size() > 0) { td.d0 = dl[0].first; td.n0 = dl[0].second; }
      if (dl.size() > 1) { td.d1 = dl[1].first; td.n1 = dl[1].second; }
      if (dl.size() > 2) {
        td.ovf = (int)P.dep_ovf.size();
        for (size_t i = 2; i < dl.size(); ++i) { P.dep_ovf.push_back(dl[i].first); P.dep_ovf.push_back(dl[i].second); }
      }
      for (int t = 0; t * to < outs; ++t) { P.tiles.push_back(rec(k, t)); P.deps.push_back(td); }
    }
    ph.ntiles = (int)((int64_t)P.tiles.size() - ph.tile_off);
    P.phases.push_back(ph);
  };
  for (int l = cut + 1; l < S->nlevels; ++l) level_phase(0, l);     // forward: outputs are the f rows of each front
  P.nfwd = (int)P.phases.size();
  for (int l = S->nlevels - 1; l > cut; --l) level_phase(1, l);     // backward: outputs are the nc pivot columns
  if (cut >= 0) subtree_phase(1);
}

// ---- inspection entry point (tests; not used by the product path) ----------------------------
template <class T>
static int64_t copy_out64(const std::vector<T>& v, int64_t* out, int64_t cap) {
  int64_t m = std::min<int64_t>((int64_t)v.size(), cap);
  if (out) for (int64_t i = 0; i < m; ++i) out[i] = (int64_t)v[i];
  return (int64_t)v.size();
}

extern "C" int64_t eigd_solve_plan_get(const eigd_symbolic* s, int target_warps, int nslots, int cut, int which,
                                       int64_t* out, int64_t cap) {
  SolvePlanHost P;
  build_solve_plan_host(s, target_warps, nslots, cut, P);
  switch (which) {
    case 0: return copy_out64(P.soff, out, cap);
    case 1: return copy_out64(P.ovf_row, out, cap);
    case 2: return copy_out64(P.ovf, out, cap);
    case 3: {
      std::vector<int64_t> flat;
      flat.reserve(P.tiles.size() * 8);
      for (const TileRec& r : P.tiles) {
        int64_t a[8] = {r.first, r.nc, r.nb, r.tile, r.soff, r.w_off, r.row_off, r.link};
        flat.insert(flat.end(), a, a + 8);
      }
      return copy_out64(flat, out, cap);
    }
    case 4: {
      std::vector<int64_t> flat;
      for (const PhaseRec& p : P.phases) {
        int64_t a[6] = {p.dir, p.ws, p.ntiles, p.level, p.tile_off, p.pad};
        flat.insert(flat.end(), a, a + 6);
      }
      return copy_out64(flat, out, cap);
    }
    case 5: return copy_out64(P.sub_ptr, out, cap);
    case 6: return copy_out64(P.sub_slot, out, cap);
    case 8: return copy_out64(P.slab, out, cap);
    case 11: return copy_out64(P.th_fwd, out, cap);
    case 12: return copy_out64(P.th_bwd, out, cap);
    case 9: {
      std::vector<int64_t> flat;
      flat.reserve(P.deps.size() * 8);
      for (const TileDep& d : P.deps) {
        int64_t a[8] = {d.self, d.ndep, d.d0, d.n0, d.d1, d.n1, d.ovf, d.pad};
        flat.insert(flat.end(), a, a + 8);
      }
      return copy_out64(flat, out, cap);
    }
    case 10: return copy_out64(P.dep_ovf, out, cap);
    case 7: {
      std::vector<int64_t> v{P.cut_level, P.nslots, P.nfwd};
      return copy_out64(v, out, cap);
    }
    default: return -1;
  }
}
