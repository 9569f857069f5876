"""Linearised buckling of the H8 solid without a GPU: boundary conditions and loads of the 3-D compressed column, the
reduced pattern and its source lists against scipy, the nested-dissection ordering of the reduced column, and
self-checks of the numpy restatement tests/h8_buckling_oracle.py (symmetry, rigid translations, dG/du)."""
import numpy as np
import pytest
import scipy.sparse as sp

import h8_buckling_oracle as hbo
import h8_oracle as ho
from eigd_b200 import fe, topo
from eigd_b200.device import Symbolic


def _reduced(bcs, ndof):
    fixed = np.zeros(ndof, dtype=bool)
    for node, comps in bcs.items():
        fixed[3 * node + np.asarray(comps)] = True
    return np.nonzero(~fixed)[0]


@pytest.mark.parametrize("dims", [(4, 3, 10), (32, 24, 128), (31, 17, 5)])
def test_column_bcs_and_loads(dims):
    nx, ny, nz = dims
    conn, X, bcs, forces = topo.domain_compressed_column_3d(nx, ny, nz, 1.0, 0.75, 4.0)
    base = np.nonzero(X[:, 2] == 0.0)[0]
    assert sorted(bcs) == list(base) and len(base) == (nx + 1) * (ny + 1)
    assert all(list(c) == [0, 1, 2] for c in bcs.values())
    F = np.array(list(forces.values()))
    nodes = np.array(list(forces))
    assert np.all(F[:, :2] == 0.0) and np.all(F[:, 2] < 0.0)
    assert abs(F[:, 2].sum() + 3e-4) < 1e-18
    assert np.all(X[nodes, 2] == 4.0)                                              # top face
    ox, oy = int(np.ceil(nx / 30)), int(np.ceil(ny / 30))
    assert len(nodes) == (2 * ox + 1) * (2 * oy + 1)
    assert np.allclose(X[nodes, :2].mean(axis=0), [1.0 * (nx // 2) / nx, 0.75 * (ny // 2) / ny])     # central patch


def test_reduced_pattern_matches_scipy_fancy_indexing():
    nx, ny, nz = 4, 3, 5
    conn, X, bcs, _ = topo.domain_compressed_column_3d(nx, ny, nz, 1.0, 0.75, 2.0)
    ndof = 3 * X.shape[0]
    var = fe.element_dofs(conn, 3)
    indptr, indices, src_ptr, src = fe.assembly_structure(var, ndof)
    reduced = _reduced(bcs, ndof)
    r_indptr, r_indices, r_src_ptr, r_src = fe.reduced_structure(indptr, indices, src_ptr, src, reduced, ndof)
    Ke = np.random.default_rng(0).normal(size=(len(conn), 24, 24))
    i = np.repeat(var, 24, axis=1).ravel()
    j = np.tile(var, (1, 24)).ravel()
    K = sp.coo_matrix((Ke.ravel(), (i, j)), shape=(ndof, ndof)).tocsr()
    Kr = K[reduced, :][:, reduced]
    assert np.array_equal(r_indptr, Kr.indptr) and np.array_equal(r_indices, Kr.indices)
    vals = np.add.reduceat(Ke.ravel()[r_src], r_src_ptr[:-1])          # every non-zero has at least one source
    assert np.allclose(vals, Kr.data, rtol=1e-13, atol=1e-13)


def test_reduced_column_ordering_equals_node_ordering():
    """BucklingH8Problem.dof_coords gives one coordinate per reduced dof; the symbolic analysis merges the three
    indistinguishable dofs of a node, so on the clamped column it orders the reduced system as node coordinates with 3
    dofs per node do."""
    nx, ny, nz = 6, 4, 12
    conn, X, bcs, _ = topo.domain_compressed_column_3d(nx, ny, nz, 1.0, 0.75, 2.0)
    ndof = 3 * X.shape[0]
    indptr, indices, src_ptr, src = fe.assembly_structure(fe.element_dofs(conn, 3), ndof)
    reduced = _reduced(bcs, ndof)
    r_indptr, r_indices, _, _ = fe.reduced_structure(indptr, indices, src_ptr, src, reduced, ndof)
    per_dof = Symbolic(r_indptr, r_indices, len(reduced), coords=X[reduced // 3], dof_per_node=1)
    per_node = Symbolic(r_indptr, r_indices, len(reduced), coords=X[reduced[::3] // 3], dof_per_node=3)
    assert np.array_equal(per_dof.get("perm"), per_node.get("perm"))
    assert per_dof.stats() == per_node.stats()


@pytest.fixture(scope="module")
def small():
    nx, ny, nz = 2, 2, 2
    conn, _ = fe.hex_mesh(nx, ny, nz)
    X = ho.perturbed_box(nx, ny, nz, (1.2, 0.9, 1.1), amp=0.25, seed=1)
    X[13] += [0.05, -0.04, 0.03]                            # the one interior node is perturbed as well
    return hbo.H8BucklingOracle(conn, X, E=1.7, nu=0.27)


def test_oracle_G_symmetric_and_translation_free(small):
    rng = np.random.default_rng(2)
    u = rng.normal(size=small.ndof)
    G0 = small.G0(u)
    assert np.abs(G0 - G0.transpose(0, 2, 1)).max() <= 1e-14 * np.abs(G0).max()
    t = np.tile(rng.normal(size=3), small.ndof // 3)                    # rigid translation: no strain, no stress
    assert np.abs(small.G0(t)).max() <= 1e-14 * np.abs(G0).max()
    assert np.abs(small.stresses(t, np.ones(len(small.conn)))).max() <= 1e-14 * np.abs(small.stresses(u, np.ones(8))).max()


def test_oracle_dGdu_matches_central_difference(small):
    rng = np.random.default_rng(3)
    kg = rng.uniform(0.2, 1.0, len(small.conn))
    W, V = rng.normal(size=(small.ndof, 3)), rng.normal(size=(small.ndof, 3))
    u, du = rng.normal(size=small.ndof), rng.normal(size=small.ndof)

    def form(x):
        return float(np.sum(kg * small.quadform(small.G0(x), np.ones(len(kg)), W, V)))
    h = 1e-3
    fd = (form(u + h * du) - form(u - h * du)) / (2 * h)
    d = float(small.dG_du(kg, W, V) @ du)
    assert abs(fd - d) <= 1e-11 * abs(d)
    assert abs(form(u) - float(small.dG_du(kg, W, V) @ u)) <= 1e-11 * abs(form(u))       # linear in u
