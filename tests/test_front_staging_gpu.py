"""Subtree phases whose fronts take every path of the subtree kernel at k >= 2: operands staged in shared memory,
operands loaded directly (forward), and the tile path (test_front_staging_cpu.py asserts that the case has all three)."""
import numpy as np
import pytest

from test_front_staging_cpu import CASE
from test_kernels_gpu import grid_matrix

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def test_front_staging_paths():
    from eigd_b200 import device as D
    D.init()
    nx, ny, dof = CASE
    rng = np.random.default_rng(nx + ny + dof)
    A, X = grid_matrix(nx, ny, dof, rng)
    n = A.shape[0]
    sym = D.Symbolic(A.indptr, A.indices, n, coords=X, dof_per_node=dof)
    Ad = D.CsrDevice.from_scipy(A)
    fac = D.Factor(sym, max_rhs=16).numeric(Ad.data, sym.assembly_map_device(Ad.indptr, Ad.indices))
    for k in (1, 2, 3, 10, 16):
        B = rng.normal(size=(n, k))
        Bd = D.to_device(B)
        X1 = fac.solve(Bd).cpu().numpy()
        r = np.abs(A @ X1 - B).max() / np.abs(B).max()
        assert r < 1e-11, (k, r)
        X2 = fac.solve(Bd).cpu().numpy()
        assert np.array_equal(X1, X2), "solve is not bitwise reproducible"
