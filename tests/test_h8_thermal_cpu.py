"""The scalar (heat conduction) H8 model without a GPU: known answers of the element restated in
tests/h8_thermal_oracle.py, the symbolic structures and front-pool offsets of the scalar 3-D pattern, the arguments
``make_thermal_3d_model`` builds its mesh and filter with, and the shapes the model and the Helmholtz filter refuse."""
import inspect

import numpy as np
import pytest
import scipy.sparse as sp

import h8_oracle as ho
import h8_thermal_oracle as hto
import multifrontal_oracle as mo
from eigd_b200 import fe, topo as T
from eigd_b200.device import Symbolic
from test_front_pool_cpu import check_pool


def _perturbed_element():
    """The central element of a perturbed 3 x 3 x 3 box: all eight of its nodes are interior, so all of them move."""
    conn, _ = fe.hex_mesh(3, 3, 3)
    X = ho.perturbed_box(3, 3, 3, (1.2, 0.9, 1.0), amp=0.3, seed=11)
    return X[conn[13]]


@pytest.fixture(scope="module")
def element():
    xe = _perturbed_element()
    K, M = hto.element_matrices(xe)
    return xe, K, M, ho.detj(xe).sum()          # the 2x2x2 rule integrates the trilinear volume exactly


def test_conductivity_annihilates_constants(element):
    _, K, _, _ = element
    assert np.abs(K @ np.ones(8)).max() <= 1e-14 * np.abs(K).max()


def test_conductivity_is_spsd_with_one_dimensional_null_space(element):
    _, K, _, _ = element
    assert np.allclose(K, K.T, rtol=0, atol=1e-15 * np.abs(K).max())
    w = np.linalg.eigvalsh(K)
    assert abs(w[0]) <= 1e-13 * w[-1]
    assert np.all(w[1:] > 1e-6 * w[-1])


def test_linear_field_energy(element):
    xe, K, _, vol = element
    g = np.array([0.7, -1.3, 0.4])
    T_ = xe @ g                                  # T(x) = g . x, reproduced exactly by the trilinear element
    assert abs(T_ @ K @ T_ - g @ g * vol) <= 1e-13 * (g @ g) * vol


def test_capacity_sums_to_volume_and_is_the_solid_mass_block(element):
    xe, _, M, vol = element
    assert abs(M.sum() - vol) <= 1e-14 * vol
    _, Ms = ho.element_matrices(xe, density=1.0)
    assert np.abs(Ms[::3, ::3] - M).max() <= 1e-15 * np.abs(M).max()


@pytest.mark.parametrize("use_coords", [True, False])
def test_symbolic_structures_of_scalar_3d_pattern_bit_exact(use_coords):
    conn, X = fe.hex_mesh(6, 5, 4, 1.0, 0.8, 0.6)
    ndof = X.shape[0]
    indptr, indices, _, _ = fe.assembly_structure(fe.element_dofs(conn, 1), ndof)
    A = sp.csr_matrix((np.ones(len(indices)), indices, indptr), shape=(ndof, ndof))
    assert np.all(np.diff(indptr) <= 27)
    sym = Symbolic(indptr, indices, ndof, coords=X if use_coords else None, dof_per_node=1)
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


@pytest.mark.parametrize("box", [(6, 5, 4), (24, 20, 16)])
def test_pool_offsets_of_scalar_hex_meshes(box):
    conn, X = fe.hex_mesh(*box, 1.0, 0.8, 0.6)
    indptr, indices, _, _ = fe.assembly_structure(fe.element_dofs(conn, 1), X.shape[0])
    pool, resident = check_pool(Symbolic(indptr, indices, X.shape[0], coords=X, dof_per_node=1))
    assert pool <= resident


def test_factory_defaults():
    sig = inspect.signature(T.make_thermal_3d_model).parameters
    nx, ny, nz = (sig[k].default for k in ("nx", "ny", "nz"))
    assert (nx, ny, nz) == (80, 64, 48) and (nx + 1) * (ny + 1) * (nz + 1) == 257985
    assert (sig["Lx"].default, sig["Ly"].default, sig["Lz"].default) == (1.0, 0.8, 0.6)
    assert sig["rfact"].default == 4.0 and sig["ftype"].default == "spatial"


@pytest.mark.parametrize("ftype", ["spatial", "helmholtz"])
def test_factory_builds_box_and_filter(monkeypatch, ftype):
    seen = {}

    def fake_filter(conn, X, r0=1.0, ftype="spatial", **kw):
        seen["filter"] = (conn, X, r0, ftype, kw)
        return "filter"

    def fake_analysis(fltr, conn, X, **kw):
        seen["analysis"] = (fltr, conn, X, kw)
        return "model"

    monkeypatch.setattr(fe, "NodeFilter", fake_filter)
    monkeypatch.setattr(T, "ThermalTopology3DAnalysis", fake_analysis)
    assert T.make_thermal_3d_model(5, 4, 3, Lx=2.0, Ly=1.2, Lz=0.9, rfact=2.5, ftype=ftype, N=7, fronts="pooled") == "model"
    conn, X, r0, ft, kw = seen["filter"]
    c_ref, X_ref = fe.hex_mesh(5, 4, 3, 2.0, 1.2, 0.9)
    assert np.array_equal(conn, c_ref) and np.array_equal(X, X_ref)
    assert r0 == pytest.approx(2.5 * 1.2 / 4) and ft == ftype and kw == {}
    fltr, conn2, X2, kw2 = seen["analysis"]
    assert fltr == "filter" and conn2 is conn and X2 is X
    assert kw2 == {"N": 7, "fronts": "pooled"}


def test_the_3d_driver_only_replaces_the_element_model():
    own = set(vars(T.ThermalTopology3DAnalysis)) - {"__module__", "__doc__", "__qualname__", "__firstlineno__",
                                                     "__static_attributes__"}
    assert own == {"_make_problem"}
    assert issubclass(T.ThermalTopology3DAnalysis, T.ThermalTopologyAnalysis)


@pytest.mark.parametrize("conn_shape,X_shape", [((4, 4), (20, 3)), ((4, 8), (20, 2)), ((32,), (20, 3)), ((4, 8), (60,))])
def test_model_refuses_bad_shapes(conn_shape, X_shape):
    with pytest.raises(ValueError, match=r"H8ThermalProblem needs conn \(nelems, 8\) and X \(nnodes, 3\)"):
        fe.H8ThermalProblem(np.zeros(conn_shape, dtype=np.int64), np.zeros(X_shape))


def test_helmholtz_filter_refuses_mismatched_mesh():
    conn, X = fe.grid_mesh(4, 3)
    X3 = np.concatenate([X, np.zeros((X.shape[0], 1))], axis=1)
    with pytest.raises(ValueError, match="3-D coordinates with 4-node conn"):
        fe.NodeFilter(conn, X3, r0=0.5, ftype="helmholtz")
    hconn, hX = fe.hex_mesh(2, 2, 2)
    with pytest.raises(ValueError, match="2-D coordinates with 8-node conn"):
        fe.NodeFilter(hconn, hX[:, :2], r0=0.5, ftype="helmholtz")
