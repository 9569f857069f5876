"""The H8 solid without a GPU: mesh numbering and orientation of fe.hex_mesh, known answers of the element restated in
tests/h8_oracle.py, and the symbolic structures of a 3-D pattern (3 coordinates, 3 dofs per node) bit for bit against
the numpy restatement of oracle/multifrontal_oracle.py."""
import numpy as np
import pytest
import scipy.sparse as sp

import h8_oracle as ho
import multifrontal_oracle as mo
from eigd_b200 import fe
from eigd_b200.device import Symbolic


def test_hex_mesh_numbering():
    nx, ny, nz = 3, 2, 4
    conn, X = fe.hex_mesh(nx, ny, nz, 3.0, 1.0, 2.0)
    assert conn.shape == (nx * ny * nz, 8) and X.shape == ((nx + 1) * (ny + 1) * (nz + 1), 3)
    node = lambda i, j, k: (i * (ny + 1) + j) * (nz + 1) + k           # noqa: E731
    for i in range(nx + 1):
        for j in range(ny + 1):
            for k in range(nz + 1):
                assert np.allclose(X[node(i, j, k)], [i * 3.0 / nx, j * 1.0 / ny, k * 2.0 / nz])
    for i in range(nx):
        for j in range(ny):
            for k in range(nz):
                e = i + nx * (j + ny * k)
                assert list(conn[e]) == [node(i, j, k), node(i + 1, j, k), node(i + 1, j + 1, k), node(i, j + 1, k),
                                         node(i, j, k + 1), node(i + 1, j, k + 1), node(i + 1, j + 1, k + 1),
                                         node(i, j + 1, k + 1)]
    assert sorted(np.unique(conn)) == list(range(X.shape[0]))


@pytest.mark.parametrize("perturb", [False, True])
def test_hex_mesh_positive_jacobian(perturb):
    conn, X = fe.hex_mesh(4, 3, 3, 2.0, 1.0, 1.0)
    if perturb:
        X = ho.perturbed_box(4, 3, 3, (2.0, 1.0, 1.0), amp=0.3, seed=1)
    dets = np.array([ho.detj(X[c]) for c in conn])
    assert np.all(dets > 0.0)


def _distorted_element():
    xe = ho.SIGNS * 0.5 + 0.5
    return xe * np.array([1.3, 0.8, 1.1]) + np.random.default_rng(2).uniform(-0.12, 0.12, (8, 3))


@pytest.mark.parametrize("which", ["cube", "distorted"])
def test_element_null_space_is_rigid_motion(which):
    xe = ho.SIGNS * 0.5 + 0.5 if which == "cube" else _distorted_element()
    K, _ = ho.element_matrices(xe, E=2.0, nu=0.3)
    assert np.allclose(K, K.T, rtol=0, atol=1e-14 * np.abs(K).max())
    w = np.linalg.eigvalsh(K)
    assert np.all(np.abs(w[:6]) <= 1e-12 * w[-1])
    assert np.all(w[6:] > 1e-6 * w[-1])
    R = ho.rigid_modes(xe)
    assert np.linalg.norm(K @ R) <= 1e-12 * np.linalg.norm(K) * np.linalg.norm(R)
    assert np.linalg.matrix_rank(R) == 6


@pytest.mark.parametrize("which", ["cube", "distorted"])
def test_element_uniform_strain_energy_and_mass(which):
    xe = ho.SIGNS * 0.5 + 0.5 if which == "cube" else _distorted_element()
    E, nu, density = 3.0, 0.25, 2.5
    K, M = ho.element_matrices(xe, E, nu, density)
    vol = ho.detj(xe).sum()                                  # exact for the trilinear map on the 2x2x2 rule
    eps = np.array([1e-3, -2e-3, 5e-4, 7e-4, -3e-4, 1.1e-3])
    G = np.array([[eps[0], eps[5] / 2, eps[4] / 2], [eps[5] / 2, eps[1], eps[3] / 2], [eps[4] / 2, eps[3] / 2, eps[2]]])
    u = (xe @ G.T).ravel()                                   # u(x) = G x: uniform strain eps
    C = ho.elasticity(E, nu)
    energy = 0.5 * eps @ C @ eps * vol
    assert abs(0.5 * u @ K @ u - energy) <= 1e-12 * energy
    for d in range(3):
        assert abs(M[d::3, d::3].sum() - density * vol) <= 1e-13 * density * vol
        others = [c for c in range(3) if c != d]
        assert np.all(M[d::3][:, others[0]::3] == 0.0)


@pytest.mark.parametrize("use_coords", [True, False])
def test_symbolic_structures_of_3d_pattern_bit_exact(use_coords):
    conn, X = fe.hex_mesh(5, 4, 3, 1.0, 0.8, 0.6)
    ndof = 3 * X.shape[0]
    indptr, indices, _, _ = fe.assembly_structure(fe.element_dofs(conn, 3), ndof)
    A = sp.csr_matrix((np.ones(len(indices)), indices, indptr), shape=(ndof, ndof))
    sym = Symbolic(indptr, indices, ndof, coords=X if use_coords else None, dof_per_node=3)
    arr = sym.arrays()
    perm, snf = arr["perm"], arr["sn_first"]
    assert np.array_equal(np.sort(perm), np.arange(ndof))
    assert snf[0] == 0 and snf[-1] == ndof and np.all(np.diff(snf) > 0)
    ns = len(snf) - 1
    parent_o, count_o = mo.etree_and_counts(A, perm)
    assert np.array_equal(arr["parent"], parent_o)
    assert np.array_equal(arr["colcount"], count_o)
    rows_o, snpar_o = mo.front_structures(A, perm, snf, parent_o)
    assert np.array_equal(arr["sn_parent"], snpar_o)
    rp, rel = arr["sn_rowptr"], arr["rel"]
    for k in range(ns):
        assert np.array_equal(arr["sn_rows"][rp[k]:rp[k + 1]], rows_o[k]), k
        p = arr["sn_parent"][k]
        if p >= 0:
            prow = np.concatenate([np.arange(snf[p], snf[p + 1]), rows_o[p]])
            assert np.array_equal(prow[rel[rp[k]:rp[k + 1]]], rows_o[k]), k
    assert np.array_equal(np.sort(arr["level_sn"]), np.arange(ns))
    kids = arr["sn_parent"] >= 0
    assert np.all(arr["sn_level"][arr["sn_parent"][kids]] > arr["sn_level"][kids])
    f = np.array([snf[k + 1] - snf[k] + len(rows_o[k]) for k in range(ns)])
    nc = np.diff(snf)
    assert sym.query("exact_nnzL") == int(count_o.sum())
    assert sym.query("nnzL") == int(sum(nc[k] * f[k] - nc[k] * (nc[k] + 1) // 2 for k in range(ns)))
    assert sym.query("max_front") == int(f.max())
