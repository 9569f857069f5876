"""What the matrices of tests/factor_cases.py cover in the symbolic analysis and the solve plan (no GPU needed): the
device tests in test_factor_dense_ref_gpu.py rely on these shapes, so a change of symbolic.cpp or solve_plan.cpp that
silently removes one of them fails here.

  * every dense case is ONE supernode of exactly its width (1 .. 512, either side of the 32-column edges);
  * every bordered case has one supernode per diagonal block with exactly `border` rows below, and the border on top;
  * a grid case has a supernode wider than 256 columns (the hb = 256 stage of the recursive-doubling inverse runs),
    the grid cases cover 1, 2, 3 and 6 DOF per node, and the caps they are built with hold;
  * the front-mode grid cases and the Kronecker cases have subtree phases and thin (16- or 8-row) tiles, the
    90 x 70 case of the right-hand-side sweep has none;
  * the Kronecker spectra are the closed form (eigvalsh on small instances, eigenvectors on the full ones) and every
    shift sits in a gap of at least 1e-6 relative."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp

from eigd_b200 import _lib
from eigd_b200.device import Symbolic
import factor_cases as fc


def symbolic(c):
    return Symbolic(c.A.indptr, c.A.indices, c.n, coords=c.coords, dof_per_node=c.dof, opts=c.opts)


def plan_meta(sym):
    """(subtree phase meta of the solve plan, set of tile heights above the cut), for the B200 plan (148 SMs)."""
    lib = _lib.load()
    meta = np.zeros(3, dtype=np.int64)
    lib.eigd_solve_plan_get(sym.handle, 148 * 16, 148, -2, 7, meta.ctypes.data_as(ctypes.c_void_p), 3)
    heights = set()
    for which in (11, 12):
        cnt = lib.eigd_solve_plan_get(sym.handle, 148 * 16, 148, -2, which, None, 0)
        th = np.zeros(cnt, dtype=np.int64)
        lib.eigd_solve_plan_get(sym.handle, 148 * 16, 148, -2, which, th.ctypes.data_as(ctypes.c_void_p), cnt)
        heights |= set(th.tolist())
    return meta, heights


@pytest.mark.parametrize("kind", ["spd", "indefinite", "saddle"])
def test_dense_cases_are_one_supernode_of_their_width(kind):
    for w in fc.DENSE_WIDTHS:
        if kind == "saddle" and w < 2:
            continue
        c = fc.dense_case(w, kind)
        assert c.A.nnz == w * w                          # zeros of the saddle stay in the pattern
        sym = symbolic(c)
        assert np.diff(sym.get("sn_first")).tolist() == [w], (kind, w)
        assert sym.query("max_cols") == w
        if kind == "saddle":
            assert (c.A.diagonal() == 0).sum() == c.nneg
        if w <= 64:
            assert (np.linalg.eigvalsh(c.A.toarray()) < 0).sum() == c.nneg


def test_dense_widths_straddle_the_block_edges():
    ws = set(fc.DENSE_WIDTHS)
    for edge in (32, 64, 128, 256):
        assert {edge - 1, edge, edge + 1} <= ws
    assert 1 in ws and 512 in ws and 511 in ws


@pytest.mark.parametrize("blocks,border", fc.BORDERED)
def test_bordered_cases_widths_and_rows_below(blocks, border):
    c = fc.bordered_case(blocks, border)
    sym = symbolic(c)
    widths = np.diff(sym.get("sn_first"))
    below = np.diff(sym.get("sn_rowptr"))
    got = sorted(zip(widths.tolist(), below.tolist()))
    assert got == sorted([(b, border) for b in blocks] + [(border, 0)]), got
    parent = sym.get("sn_parent")
    top = int(np.nonzero(parent < 0)[0][0])
    assert (parent < 0).sum() == 1 and widths[top] == border and (parent[np.arange(len(parent)) != top] == top).all()


@pytest.mark.parametrize("case", fc.GRID_CASES, ids=lambda g: "x".join(map(str, g)))
def test_grid_case_caps(case):
    sym = symbolic(fc.grid_case(*case))
    assert sym.query("max_cols") <= (case[3] or 256)


def test_grid_cases_cover_wide_supernodes_and_dofs():
    assert {g[0] for g in fc.GRID_CASES} == {1, 2, 3, 6}
    sym = symbolic(fc.grid_case(*fc.WIDE_6DOF))
    # the recursive-doubling inverse of the pivot blocks runs its hb = 256 stage only for supernodes wider than 256
    assert sym.query("max_cols") > 256
    # relaxation changes the partition (both settings are exercised, not one twice)
    for d, nx, ny in fc.GRID_SIZES:
        parts = [np.diff(symbolic(fc.grid_case(d, nx, ny, 256, r)).get("sn_first")).tolist() for r in (0, 1)]
        assert parts[0] != parts[1]


@pytest.mark.parametrize("case", fc.FRONT_MODE + [None], ids=["250x200x1", "160x120x2", "kron"])
def test_large_cases_have_subtree_phases_and_thin_tiles(case):
    cases = [fc.grid_case(*case)] if case else [fc.kron_case(*k) for k in fc.KRON]
    for c in cases:
        meta, heights = plan_meta(symbolic(c))
        assert meta[0] >= 0, (c.name, "expected subtree phases")
        assert heights & {16, 8}, (c.name, "expected thin tiles (height 16 or 8)", heights)


def test_rhs_sweep_level_only_case_has_no_subtree_phase():
    meta, _ = plan_meta(symbolic(fc.grid_case(*fc.RHS_LEVEL_ONLY)))
    assert meta[0] < 0


@pytest.mark.parametrize("nx,ny,dof", [(13, 11, 1), (9, 7, 2), (12, 12, 1)])
def test_kron_spectrum_closed_form_small(nx, ny, dof):
    L = sp.kron(fc.second_difference(nx), sp.identity(ny)) + sp.kron(sp.identity(nx), fc.second_difference(ny))
    if dof == 2:
        L = sp.kron(L, sp.csr_matrix(fc.KRON_C))
    assert np.abs(np.linalg.eigvalsh(L.toarray()) - fc.kron_spectrum(nx, ny, dof)).max() < 1e-12


@pytest.mark.parametrize("nx,ny,dof,target", fc.KRON)
def test_kron_cases_shift_in_a_gap(nx, ny, dof, target):
    c = fc.kron_case(nx, ny, dof, target)
    assert np.gcd(nx, ny) == 1
    ev = c.spectrum                                  # eigenvalues of the shifted matrix, ascending
    assert len(ev) == c.n
    assert (ev < 0).sum() == c.nneg and abs(c.nneg - target) <= 10
    assert c.gap >= fc.GAP_REL and np.abs(ev).min() >= fc.GAP_REL * c.sigma
    # the two eigenpairs either side of the shift, from the closed-form eigenvectors sin(i a pi/(nx+1)) sin(j b pi/(ny+1))
    # (times an eigenvector of C): A v = (lam - sigma) v on the full matrix
    ti = fc.dirichlet_eigenvalues(nx)
    tj = fc.dirichlet_eigenvalues(ny)
    mu, W = np.linalg.eigh(fc.KRON_C) if dof == 2 else (np.ones(1), np.ones((1, 1)))
    lam = (ti[:, None, None] + tj[None, :, None]) * mu[None, None, :]
    for shifted in (ev[c.nneg - 1], ev[c.nneg]):
        i, j, q = np.unravel_index(np.argmin(np.abs(lam - c.sigma - shifted)), lam.shape)
        v = np.kron(np.kron(np.sin((i + 1) * np.pi * np.arange(1, nx + 1) / (nx + 1)),
                            np.sin((j + 1) * np.pi * np.arange(1, ny + 1) / (ny + 1))), W[:, q])
        assert np.abs(c.A @ v - shifted * v).max() <= 1e-12 * np.abs(v).max()
