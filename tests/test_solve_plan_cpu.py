"""CPU emulation of the persistent triangular-solve kernel on the host-built plan (csrc/solve_plan.cpp).

The plan is pure integer data (tile records, phases, subtree tables, child slabs, overflow lists); this
test walks it exactly as solve.cu does -- phase by phase, slot by slot, tile by tile, with the same
index arithmetic -- on panels built by the numpy multifrontal oracle, and compares the solution with
scipy.  It needs no GPU: it pins the schedule and the index-free forward data flow."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from eigd_b200 import _lib, fe
from eigd_b200.device import Symbolic
import multifrontal_oracle as mo
import factor_cases as fc

MASK48 = (1 << 48) - 1


def plan_arrays(sym, target_warps, nslots, cut):
    lib = _lib.load()

    def get(which):
        cnt = lib.eigd_solve_plan_get(sym.handle, target_warps, nslots, cut, which, None, 0)
        out = np.zeros(max(cnt, 1), dtype=np.int64)
        lib.eigd_solve_plan_get(sym.handle, target_warps, nslots, cut, which, out.ctypes.data_as(ctypes.c_void_p), cnt)
        return out[:cnt]

    return {"ovf_row": get(1), "ovf": get(2), "tiles": get(3).reshape(-1, 8), "phases": get(4).reshape(-1, 6),
            "sub_ptr": get(5), "sub_slot": get(6), "meta": get(7), "slab": get(8), "deps": get(9).reshape(-1, 8),
            "dep_ovf": get(10)}


def tile_deps(plan, te):
    """[(counter, tiles per solve), ...] of tile te (TileDep, solve_plan.hpp)."""
    selfc, ndep, d0, n0, d1, n1, ovf, _ = (int(v) for v in plan["deps"][te])
    out = [(d0, n0), (d1, n1)][:min(ndep, 2)]
    for q in range(2, ndep):
        out.append((int(plan["dep_ovf"][ovf + 2 * (q - 2)]), int(plan["dep_ovf"][ovf + 2 * (q - 2) + 1])))
    return selfc, out


def emulate(plan, S, sym_arr, dinv, b, shuffle=None):
    """shuffle: a numpy Generator -> the level-phase tiles run in a RANDOM order constrained only by their
    completion-counter dependencies (what the barrier-free kernel guarantees), instead of the plan order."""
    perm, sn_rows, rel = sym_arr["perm"], sym_arr["sn_rows"], sym_arr["rel"]
    n = len(perm)
    sumf = len(plan["ovf_row"])
    wbuf = np.zeros((3, sumf))
    bperm = b[perm]
    y, xp = np.zeros(n), np.zeros(n)
    done = set()

    def child(t, link):
        if not (link >> 57) & 1:
            return 0.0
        v = wbuf[0, t] + wbuf[1, t]
        if (link >> 56) & 1:
            o = plan["ovf_row"][t]
            if o >= 0:
                cnt = plan["ovf"][o]
                v += sum(wbuf[2, plan["ovf"][o + 1 + q]] for q in range(cnt))
        return v

    def do_tile(direction, rec, th=32):
        first, nc, nb, tile, soff, w_off, row_off, link = (int(v) for v in rec)
        f = nc + nb
        o0 = tile * th
        Sk = S[first]
        assert Sk.shape == (f, nc)
        key = (direction, first, tile)
        assert key not in done, "tile scheduled twice"
        done.add(key)
        if direction == 0:
            cend = min(nc, o0 + th)
            w1 = np.array([bperm[first + c] + child(w_off + c, link) for c in range(cend)])
            for out in range(o0, min(o0 + th, f)):
                acc = Sk[out, :cend] @ w1
                if out >= nc:
                    acc += child(w_off + out, link)
                if out < nc:
                    y[first + out] = dinv[first + out] * acc
                else:
                    slab = (link >> 48) & 0xff
                    assert slab in (0, 1, 2), "a root front has no rows below its pivots"
                    if slab < 2:
                        wbuf[slab, (link & MASK48) + rel[row_off + out - nc]] = acc
                    else:
                        wbuf[2, w_off + out] = acc
        else:
            vec = np.concatenate([y[first:first + nc], xp[sn_rows[row_off:row_off + nb]]])
            for out in range(o0, min(o0 + th, nc)):
                xp[first + out] = Sk[o0:, out] @ vec[o0:]

    tiles = plan["tiles"]
    cnt = {}
    pending = []                       # level-phase tiles not yet run: (te, direction)

    height = {}                        # tile index -> tile height of its level phase (PhaseRec.pad)
    for d, ws, ntiles, level, tile_off, _to in plan["phases"]:
        if ws > 0:
            assert int(_to) in (8, 16, 32)
            for te in range(tile_off, tile_off + ntiles):
                height[int(te)] = int(_to)

    def run_level_tile(te, d):
        selfc, deps = tile_deps(plan, te)
        assert all(cnt.get(c, 0) >= need for c, need in deps), "dependency not complete in plan order"
        do_tile(d, tiles[te], height[int(te)])
        cnt[selfc] = cnt.get(selfc, 0) + 1

    def drain():
        # random topological execution: any tile whose counters are complete may run next
        while pending:
            ready = [i for i, (te, d) in enumerate(pending)
                     if all(cnt.get(c, 0) >= need for c, need in tile_deps(plan, te)[1])]
            assert ready, "deadlock: no runnable tile"
            i = ready[int(shuffle.integers(len(ready)))]
            te, d = pending.pop(i)
            run_level_tile(te, d)

    for d, ws, ntiles, level, tile_off, _to in plan["phases"]:
        if ws == 0 and pending:
            drain()                    # the backward subtree launch follows the level kernel in stream order
        if ws == 0:
            assert _to == 0
            nl, nslots = int(ntiles), int(level)
            for slot in range(nslots):
                tab = plan["sub_ptr"][tile_off + slot * (nl + 1): tile_off + (slot + 1) * (nl + 1)]
                for ll in range(nl):
                    l = ll if d == 0 else nl - 1 - ll
                    for te in range(tab[l], tab[l + 1]):
                        # one record per front, the subtree kernel runs all its tiles
                        first, nc, nb, tile = (int(v) for v in tiles[te][:4])
                        assert tile == 0
                        outs = nc + nb if d == 0 else nc
                        for t in range((outs + 31) // 32):
                            rec = tiles[te].copy()
                            rec[3] = t
                            do_tile(int(d), rec)
        else:
            for te in range(tile_off, tile_off + ntiles):
                if shuffle is None:
                    run_level_tile(te, int(d))
                else:
                    pending.append((te, int(d)))
    if pending:
        drain()
    x = np.empty(n)
    x[perm] = xp
    return x, done


def build_case(nx, ny, dof, use_coords):
    conn, X = fe.grid_mesh(nx, ny, 1.0, 0.7)
    var = fe.element_dofs(conn, dof)
    ndof = dof * X.shape[0]
    indptr, indices, _, _ = fe.assembly_structure(var, ndof)
    rng = np.random.default_rng(nx * 100 + ny + dof)
    A = sp.csr_matrix((rng.uniform(-1.0, 1.0, len(indices)), indices, indptr), shape=(ndof, ndof))
    A = A + A.T + sp.diags(np.full(ndof, 40.0))            # symmetric positive definite on the same pattern
    A = sp.csr_matrix(A)
    A.sort_indices()
    sym = Symbolic(A.indptr, A.indices, ndof, coords=X if use_coords else None, dof_per_node=dof)
    arr = sym.arrays()
    arr["amap"] = sym.assembly_map_host()
    orc = mo.MultifrontalOracle(arr).factor(A.data)
    S = {}
    for k in range(len(arr["sn_first"]) - 1):
        Fk, nc, nb = orc._front_view(orc.F, k)
        L11 = np.tril(Fk[:nc, :nc], -1) + np.eye(nc)
        Xi = np.linalg.inv(L11)
        S[int(arr["sn_first"][k])] = np.vstack([Xi, -Fk[nc:, :nc] @ Xi])
    return A, sym, arr, orc, S


# the plan arguments of the device solve on a B200: 148 SMs x 16 warps, 148 CTA slots, automatic cut
PRODUCTION = (148 * 16, 148, -2)


@pytest.mark.parametrize("nx,ny,dof,use_coords", [(22, 17, 1, True), (14, 11, 2, True), (19, 13, 1, False)])
def test_plan_emulation_matches_scipy(nx, ny, dof, use_coords):
    A, sym, arr, orc, S = build_case(nx, ny, dof, use_coords)
    n = A.shape[0]
    b = np.random.default_rng(7).normal(size=n)
    x_ref = spla.spsolve(A.tocsc(), b)
    ntiles_f = sum(-(-(S[f].shape[0]) // 32) for f in S)
    ntiles_b = sum(-(-(S[f].shape[1]) // 32) for f in S)
    nlevels = len(arr["level_ptr"]) - 1
    seen_cut = set()
    for target_warps, nslots, cut in [(64, 4, -1), (64, 4, -2), PRODUCTION, (32, 3, 1), (32, 5, 2), (16, 2, nlevels)]:
        plan = plan_arrays(sym, target_warps, nslots, cut)
        x, done = emulate(plan, S, arr, orc.dinv, b)
        assert np.abs(x - x_ref).max() <= 1e-10 * np.abs(x_ref).max(), (target_warps, nslots, cut)
        # the completion counters alone order the level phases correctly: random dependency-respecting schedules
        xs, _ = emulate(plan, S, arr, orc.dinv, b, shuffle=np.random.default_rng(target_warps + nslots))
        assert np.array_equal(xs, x), (target_warps, nslots, cut)
        # every tile of every front is scheduled exactly once per direction (32-output tiles below the cut and wherever
        # the level keeps the full height; thinner tiles only add to the count)
        assert len([1 for k in done if k[0] == 0]) >= ntiles_f
        assert len([1 for k in done if k[0] == 1]) >= ntiles_b
        if int(plan["phases"][:, 5][plan["phases"][:, 1] > 0].min(initial=32)) == 32:
            assert len([1 for k in done if k[0] == 0]) == ntiles_f and len([1 for k in done if k[0] == 1]) == ntiles_b
        if (target_warps, nslots, cut) == PRODUCTION:
            ph = plan["phases"]
            assert (ph[ph[:, 1] == 0, 5] == 0).all()                        # subtree phases: one record per front
            assert np.isin(ph[ph[:, 1] > 0, 5], (8, 16, 32)).all()          # level phases: the tile height
        cutl = int(plan["meta"][0])
        seen_cut.add(cutl)
        if cutl >= 0:
            # subtrees are complete: a front below the cut lives in the slot of its parent (if that is below the cut too)
            slot, lvl, par = plan["sub_slot"], arr["sn_level"], arr["sn_parent"]
            for k in range(len(slot)):
                assert (slot[k] >= 0) == (lvl[k] <= cutl)
                if slot[k] >= 0 and par[k] >= 0 and lvl[par[k]] <= cutl:
                    assert slot[k] == slot[par[k]]
    assert -1 in seen_cut and max(seen_cut) >= 1


def test_child_slabs_are_consistent():
    A, sym, arr, orc, S = build_case(19, 13, 1, False)
    plan = plan_arrays(sym, 64, 4, -1)
    par = arr["sn_parent"]
    slab = plan["slab"]
    ns = len(par)
    for p in range(ns):
        kids = [c for c in range(ns) if par[c] == p]
        assert [int(slab[c]) for c in kids] == [min(i, 2) for i in range(len(kids))]
    assert all(int(slab[k]) == 255 for k in range(ns) if par[k] < 0)


RING_CAP = 16384        # the largest panel ring per warp of the pipelined level kernel (solve.cu, configure)


def slice_bytes(rec, d, th, ws, bm=0):
    """Bytes of the tile-major panel slice each of the ws warps of level-phase tile rec multiplies (slice_of, solve.cu)."""
    first, nc, nb, tile = (int(v) for v in rec[:4])
    f, o0 = nc + nb, tile * th
    if d == 0:
        lo, hi, ld = 0, min(nc, (o0 + th + bm) & ~bm), min(th, f - o0)
    else:
        lo, hi, ld = o0 & ~bm, f, min(th, nc - o0)
    per = ((-(-(hi - lo) // ws)) + 1) & ~1                            # solve_slice_len
    out = []
    for s in range(ws):
        r0 = min(hi, lo + s * per)
        out.append((min(hi, r0 + per) - r0) * ld * 8)
    return out


def test_block_diagonal_slices_exceed_the_ring():
    """The block-diagonal case of the device tests is there to make level-phase tiles read a panel slice larger than
    the pipelined kernel's ring from global memory, in both sweeps; no grid case does."""
    c = fc.block_diagonal_case()
    sym = Symbolic(c.A.indptr, c.A.indices, c.n, coords=c.coords, dof_per_node=c.dof, opts=c.opts)
    plan = plan_arrays(sym, *PRODUCTION)
    big = {0: 0, 1: 0}
    for d, ws, ntiles, level, tile_off, th in plan["phases"]:
        if ws == 0:
            continue
        for te in range(tile_off, tile_off + ntiles):
            big[int(d)] += sum(b > RING_CAP for b in slice_bytes(plan["tiles"][te], int(d), int(th), int(ws)))
    assert big[0] > 0 and big[1] > 0, big
