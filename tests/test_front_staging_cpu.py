"""Which fronts below the cut take which path of the subtree kernel (solve.cu, fronts_phase), restated on the host.

A front takes FRONT MODE when it has at most 32 pivot columns, at most 256 rows and a panel of at most 10 KB
(FRONT_PANEL_MAX).  In the backward sweep of every k >= 2, and in the forward sweep of k = 2, its operands are staged
in the warp's panel ring right behind the panel when panel and operand block fit in the ring together.  Otherwise a
forward front loads them directly and a backward front takes the tile path.  The GPU test in test_front_staging_gpu.py relies on its case having fronts on every side of this rule."""
import ctypes

import numpy as np

from eigd_b200 import _lib, fe
from eigd_b200.device import Symbolic

PRODUCTION = (148 * 16, 148, -2)   # plan arguments of the device solve on a B200
CASE = (100, 80, 6)                # nx, ny, dof of the GPU test


def ring_w(kt):
    """Panel ring bytes per warp of subtree_kernel<kt> (solve.cu, configure)."""
    rec_cap = 512 if kt <= 4 else 256
    ring = (227 * 1024 - 1024 - 16 * 32 * kt * 8 - 2 * 2 * 16 * 8 - rec_cap * 48) // 16
    return min(ring, 16384) // 256 * 256


def ops_doubles(nc, nb, kids, d, k, kt):
    """front_ops_doubles (solve.cu)."""
    f = nc + nb
    if d == 0:
        return k * nc + (2 * k * f if kids else 0) + nc + (nb + 1) // 2
    return f * kt + (nb + nc + 1) // 2


def front_path(rec, d, k, kt):
    first, nc, nb, tile, soff, w_off, row_off, link = (int(v) for v in rec)
    f = nc + nb
    b = ((f * nc + 1) & ~1) * 8
    if not (nc <= 32 and b <= min(ring_w(kt), 10240) and f <= 256):
        return "tile"
    if (d == 1 or kt == 2) and b + 8 * ops_doubles(nc, nb, (link >> 57) & 1, d, k, kt) <= ring_w(kt):
        return "staged"
    return "direct" if d == 0 else "tile"


def subtree_paths(nx, ny, dof, k, kt):
    conn, X = fe.grid_mesh(nx, ny, 1.0, ny / nx)
    n = X.shape[0] * dof
    indptr, indices, _, _ = fe.assembly_structure(fe.element_dofs(conn, dof), n)
    sym = Symbolic(indptr, indices, n, coords=X, dof_per_node=dof)
    lib = _lib.load()

    def get(which):
        cnt = lib.eigd_solve_plan_get(sym.handle, *PRODUCTION, which, None, 0)
        out = np.zeros(max(cnt, 1), dtype=np.int64)
        lib.eigd_solve_plan_get(sym.handle, *PRODUCTION, which, out.ctypes.data_as(ctypes.c_void_p), cnt)
        return out[:cnt]

    tiles, phases, sub_ptr = get(3).reshape(-1, 8), get(4).reshape(-1, 6), get(5)
    out = {}
    for d, ws, nl, nslots, off, _ in phases:
        if ws:
            continue
        for slot in range(nslots):
            tab = sub_ptr[off + slot * (nl + 1): off + (slot + 1) * (nl + 1)]
            for te in range(tab[0], tab[nl]):
                key = (int(d), front_path(tiles[te], int(d), k, kt))
                out[key] = out.get(key, 0) + 1
    return out


def test_ring_sizes():
    assert [ring_w(kt) for kt in (1, 2, 4, 6, 8, 10, 12, 16)] == [12544, 12288, 11776, 12032, 11520, 11008, 10496, 9472]


def test_case_has_fronts_on_every_side():
    for k, kt in ((2, 2), (10, 10)):
        paths = subtree_paths(*CASE, k, kt)
        for key in ((0, "direct"), (0, "tile"), (1, "staged"), (1, "tile")) + (((0, "staged"),) if kt == 2 else ()):
            assert paths.get(key, 0) > 0, (k, key, paths)
