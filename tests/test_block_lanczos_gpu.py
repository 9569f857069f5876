"""Block Lanczos (csrc/block_krylov.cu: one cooperative launch per block step) on thermal Q4 pencils built on the host.

For block sizes 2, 3, 4, with and without refinement steps of the solve, and at a size whose 1024-element chunks
outnumber the co-resident CTAs (several chunks per CTA): the returned basis is B-orthonormal, the returned projected
matrix is V^T B OP V, and two runs with the same seed are bitwise identical."""
import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def E():
    import eigd_b200
    from eigd_b200 import device
    device.init()
    return eigd_b200


def q4_thermal(nx, ny):
    """Bilinear Q4 conductivity K and capacity M on an (nx - 1) x (ny - 1) grid of the unit square, no boundary
    conditions (K is singular, M is positive definite)."""
    def line(k):
        h = 1.0 / (k - 1)
        d = np.full(k, 2.0)
        d[[0, -1]] = 1.0
        K1 = sp.diags([-np.ones(k - 1), d, -np.ones(k - 1)], [-1, 0, 1]) / h
        M1 = sp.diags([np.ones(k - 1), 2.0 * d, np.ones(k - 1)], [-1, 0, 1]) * (h / 6.0)
        return K1, M1
    Kx, Mx = line(nx)
    Ky, My = line(ny)
    K = (sp.kron(Ky, Mx) + sp.kron(My, Kx)).tocsr()
    M = sp.kron(My, Mx).tocsr()
    return K, M


def run(E, K, M, sigma, k, ncv, P, refine):
    f = E.SpLuOperator((K - sigma * M).tocsc(), refine=refine)
    from eigd_b200.arpack import eigsh_mod
    d, z, Tm, v = eigsh_mod(K, k=k, M=M, sigma=sigma, OPinv=f, ncv=ncv, tol=1e-8, seed=3, block=P)
    return f, d, Tm, v[:, :ncv]


def check_basis(E, K, M, sigma, k, ncv, P, refine):
    f, d, Tm, V = run(E, K, M, sigma, k, ncv, P, refine)
    assert (f.refine > 0) == (refine > 0)
    BV = M @ V
    G = V.T @ BV
    assert np.abs(G - np.eye(ncv)).max() < 1e-12
    OPV = np.column_stack([f(BV[:, c]) for c in range(ncv)])     # OP = (K - sigma M)^-1 M through the factor
    T = BV.T @ OPV
    assert np.abs(Tm - T).max() < 1e-10 * np.abs(T).max()
    _, d2, Tm2, V2 = run(E, K, M, sigma, k, ncv, P, refine)
    assert np.array_equal(d, d2) and np.array_equal(Tm, Tm2) and np.array_equal(V, V2)


@pytest.mark.parametrize("P", [2, 3, 4])
def test_block_sizes(E, P):
    K, M = q4_thermal(73, 61)                     # n = 4453: the last 1024-element chunk is partial
    check_basis(E, K, M, -1.0, 4, 24, P, 0)


def test_refinement_indefinite_shift(E):
    K, M = q4_thermal(73, 61)
    sigma = 60.0                                  # between 5 pi^2 and 8 pi^2: LDL^T with negative pivots
    check_basis(E, K, M, sigma, 4, 24, 2, 1)


def test_more_chunks_than_resident_ctas(E):
    K, M = q4_thermal(700, 521)                   # n = 364 700: 357 chunks, more than 2 CTAs x 148 SMs
    check_basis(E, K, M, -1.0, 2, 8, 2, 0)
