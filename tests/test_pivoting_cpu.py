"""Restricted Bunch-Kaufman pivoting of the multifrontal LDL^T, CPU reference (tests/bunch_kaufman_oracle.py).

The matrices here are the ones the GPU tests (test_pivoting_gpu.py) factor: a 2-DOF-per-node operator whose node
blocks are [[0, c], [c, 0]] (zero diagonal, stored explicitly) plus a weaker (or, "mixed", an equally strong) grid
coupling, and grid matrices shifted between two close eigenvalues.  Pivoted, the oracle must give the exact inertia
and a plain (unrefined) solve at rounding level; the static path must meet perturbed pivots on the zero-diagonal
operator."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from eigd_b200.device import Symbolic
import fe_oracle as fo
from bunch_kaufman_oracle import BunchKaufmanOracle


def zero_diagonal_matrix(nx, ny, seed, coupling=0.2):
    """2 DOF per node: node block [[0, c], [c, 0]] (c in [1, 2]), every other entry of the Q4 pattern uniform in
    [-coupling, coupling]; the zero diagonal is stored.  Returns (A, node coordinates)."""
    rng = np.random.default_rng(seed)
    conn, X = fo.grid_mesh(nx, ny, 1.0, ny / nx)
    i, j = fo.coo_index(fo.element_dofs(conn, 2))
    P = sp.coo_matrix((np.ones(len(i)), (i, j))).tocsr()
    P.sum_duplicates()
    A = P.copy()
    A.data = rng.uniform(-coupling, coupling, A.nnz)
    A = ((A + A.T) * 0.5).tocsr()
    A.sort_indices()
    rows = np.repeat(np.arange(A.shape[0]), np.diff(A.indptr))
    cnode = rng.uniform(1.0, 2.0, A.shape[0] // 2)
    same = rows // 2 == A.indices // 2
    A.data[same & (rows == A.indices)] = 0.0
    A.data[same & (rows != A.indices)] = cnode[rows[same & (rows != A.indices)] // 2]
    assert A.nnz == P.nnz and (A.indices == P.indices).all()       # the zeros stay in the pattern
    return A, X


def shifted_grid_matrix(nx, ny, seed, between=4):
    """SPD grid matrix (1 DOF per node) minus a shift half-way between its between-th and (between+1)-th smallest
    eigenvalues: exactly `between` negative eigenvalues."""
    rng = np.random.default_rng(seed)
    conn, X = fo.grid_mesh(nx, ny, 1.0, ny / nx)
    i, j = fo.coo_index(fo.element_dofs(conn, 1))
    A = sp.coo_matrix((rng.uniform(-1, 1, len(i)), (i, j))).tocsr()
    A = (A + A.T) * 0.5
    A = A + sp.diags(np.abs(A).sum(axis=1).A1 + 0.1)
    lo = np.sort(spla.eigsh(A.tocsc(), k=between + 2, sigma=0.0, which="LM", return_eigenvectors=False))
    As = (A - 0.5 * (lo[between - 1] + lo[between]) * sp.identity(A.shape[0])).tocsr()
    As.sort_indices()
    return As, X


def oracle_for(A, X, dof):
    sym = Symbolic(A.indptr, A.indices, A.shape[0], coords=X, dof_per_node=dof)
    d = sym.arrays()
    d["amap"] = sym.assembly_map_host()
    return BunchKaufmanOracle(d)


def negative_eigenvalues(A):
    return int((np.linalg.eigvalsh(A.toarray()) < 0).sum())


def residual(A, x, b):
    return np.abs(A @ x - b).max() / np.abs(b).max()


# "mixed": the zero-diagonal operator with a coupling as strong as the node blocks, where the pivot search also picks
# interchanged 1x1 pivots and interchanges before 2x2 pivots
CASES = [("zero_diagonal", 12, 10, 0), ("zero_diagonal", 20, 15, 1), ("mixed", 12, 10, 1), ("shifted", 40, 30, 7),
         ("shifted", 60, 45, 3)]


def case_matrix(kind, nx, ny, seed):
    if kind in ("zero_diagonal", "mixed"):
        A, X = zero_diagonal_matrix(nx, ny, seed, coupling=1.0 if kind == "mixed" else 0.2)
        return A, X, 2
    A, X = shifted_grid_matrix(nx, ny, seed)
    return A, X, 1


@pytest.mark.parametrize("kind,nx,ny,seed", CASES)
def test_oracle_bunch_kaufman_inertia_and_residual(kind, nx, ny, seed):
    A, X, dof = case_matrix(kind, nx, ny, seed)
    ref = oracle_for(A, X, dof).factor(A.data, pivoting="bunch-kaufman")
    nneg, npert = ref.info
    assert npert == 0
    assert nneg == negative_eigenvalues(A)
    assert ref.counts["negative_pivots"] == nneg
    b = np.random.default_rng(seed + 100).normal(size=(A.shape[0], 3))
    r = residual(A, ref.solve(b), b)
    assert r <= 1e-12, r
    if kind != "shifted":
        assert ref.counts["two_by_two_pivots"] > 0
    if kind != "zero_diagonal":
        assert ref.counts["interchanges"] > 0


def test_oracle_static_path_perturbs_the_zero_diagonal():
    A, X, dof = case_matrix(*CASES[0])
    ref = oracle_for(A, X, dof).factor(A.data)
    assert ref.info[1] > 0


def test_oracle_bunch_kaufman_on_spd_takes_no_pivot_action():
    """On a strongly diagonally dominant SPD matrix every pivot test keeps the diagonal entry: no 2x2 pivot, no
    interchange, and the pivoted factor solves like the static one."""
    rng = np.random.default_rng(5)
    conn, X = fo.grid_mesh(14, 11, 1.0, 11 / 14)
    i, j = fo.coo_index(fo.element_dofs(conn, 1))
    A = sp.coo_matrix((rng.uniform(-1, 1, len(i)), (i, j))).tocsr()
    A = ((A + A.T) * 0.5 + sp.diags(np.abs(A).sum(axis=1).A1 * 2.0 + 1.0)).tocsr()
    A.sort_indices()
    o = oracle_for(A, X, 1)
    bk = o.factor(A.data, pivoting="bunch-kaufman")
    assert bk.counts["two_by_two_pivots"] == 0 and bk.counts["interchanges"] == 0
    b = rng.normal(size=A.shape[0])
    x_bk = bk.solve(b)
    x_st = oracle_for(A, X, 1).factor(A.data).solve(b)
    assert np.abs(x_bk - x_st).max() / np.abs(x_st).max() < 1e-13


def test_oracle_rejects_unknown_pivoting():
    A, X, dof = case_matrix(*CASES[0])
    with pytest.raises(ValueError):
        oracle_for(A, X, dof).factor(A.data, pivoting="partial")
