"""The quadratic tetrahedron (T10) without a GPU: the quadrature table of csrc/t10_element.cuh, known answers of the
solid and scalar elements restated in tests/t10_oracle.py, the box mesh generator and the linear-to-quadratic
conversion, the symbolic structures and front-pool offsets of T10 patterns, the factory defaults, the shapes the models
and the Helmholtz filter refuse, and the convergence of the insulated box's eigenvalues against the continuous ones and
the H8 values on the same nodes."""
import inspect
from math import factorial

import numpy as np
import pytest
import scipy.sparse as sp

import h8_oracle as ho
import h8_thermal_oracle as hto
import multifrontal_oracle as mo
import t10_oracle as to
from eigd_b200 import fe, topo as T
from eigd_b200.device import Symbolic
from test_front_pool_cpu import check_pool


def _perturbed_element():
    """An element of the central cube of a perturbed 3 x 3 x 3 box: all ten of its nodes are interior, so all of
    them move and its edges are curved."""
    conn, _ = fe.tet10_mesh(3, 3, 3)
    X = to.perturbed_tet_box(3, 3, 3, (1.2, 0.9, 1.0), amp=0.15, seed=11)
    return X[conn[6 * 13 + 4]]


@pytest.fixture(scope="module")
def element():
    xe = _perturbed_element()
    K, M = to.element_matrices(xe, E=2.0, nu=0.28, density=1.7)
    Kt, Mt = to.thermal_element_matrices(xe)
    vol = sum(w * np.linalg.det(xe.T @ dN) for _, dN, w in to.points())     # exact: detJ is cubic, the rule degree 5
    return xe, K, M, Kt, Mt, vol


def test_rule_integrates_barycentric_monomials_of_degree_4():
    """sum_q w_q l^a = int l0^a0 l1^a1 l2^a2 l3^a3 = 6 V a0! a1! a2! a3! / (|a| + 3)! on the reference tetrahedron."""
    assert to.RULE.shape == (14, 4) and np.all(to.RULE[:, 3] > 0)
    lam = np.array([to.barycentric(q) for q in range(14)])
    assert np.all(lam > 0)
    for n in range(5):
        for a0 in range(n + 1):
            for a1 in range(n + 1 - a0):
                for a2 in range(n + 1 - a0 - a1):
                    e = (a0, a1, a2, n - a0 - a1 - a2)
                    got = np.sum(to.RULE[:, 3] * np.prod(lam ** np.array(e)[None, :], axis=1))
                    exact = np.prod([factorial(k) for k in e]) / factorial(n + 3)     # 6 V = 1
                    assert abs(got - exact) <= 2e-15 * exact, (e, got, exact)


def test_shape_functions_partition_unity_and_interpolate():
    for q in range(14):
        N, dN = to.shape(to.barycentric(q))
        assert abs(N.sum() - 1.0) < 1e-15 and np.abs(dN.sum(axis=0)).max() < 1e-14
    corners = np.eye(4)
    nodes = list(corners) + [0.5 * (corners[i] + corners[j]) for i, j in to.EDGES]
    assert np.allclose(np.array([to.shape(l)[0] for l in nodes]), np.eye(10), atol=1e-15)


def test_stiffness_annihilates_rigid_modes_and_has_six_dimensional_null_space(element):
    xe, K, _, _, _, _ = element
    assert np.allclose(K, K.T, rtol=0, atol=1e-14 * np.abs(K).max())
    assert np.abs(K @ to.rigid_modes(xe)).max() <= 1e-13 * np.abs(K).max()
    w = np.linalg.eigvalsh(K)
    assert np.all(np.abs(w[:6]) <= 1e-12 * w[-1])
    assert np.all(w[6:] > 1e-6 * w[-1])


def test_constant_strain_energy(element):
    xe, K, _, _, _, vol = element
    A = np.array([[0.3, -0.2, 0.5], [0.1, 0.7, -0.4], [-0.6, 0.2, 0.25]])
    u = (xe @ A.T).ravel()                          # u(x) = A x, reproduced exactly by the isoparametric element
    eps = np.array([A[0, 0], A[1, 1], A[2, 2], A[1, 2] + A[2, 1], A[0, 2] + A[2, 0], A[0, 1] + A[1, 0]])
    energy = eps @ ho.elasticity(2.0, 0.28) @ eps * vol
    assert abs(u @ K @ u - energy) <= 1e-13 * abs(energy)


def test_mass_sums_to_density_times_volume_per_component(element):
    xe, _, M, _, Mt, vol = element
    assert vol > 0 and abs(vol - to.volume(xe)) > 1e-6 * vol       # the curved element's volume is not the corners'
    for c in range(3):
        assert abs(M[c::3, c::3].sum() - 1.7 * vol) <= 1e-14 * vol
        for d in range(3):
            if d != c:
                assert not M[c::3, d::3].any()
    assert abs(Mt.sum() - vol) <= 1e-14 * vol
    assert np.abs(M[::3, ::3] / 1.7 - Mt).max() <= 1e-15 * np.abs(Mt).max()


def test_thermal_conductivity_null_space_and_linear_field_energy(element):
    xe, _, _, Kt, _, vol = element
    assert np.abs(Kt @ np.ones(10)).max() <= 1e-14 * np.abs(Kt).max()
    w = np.linalg.eigvalsh(Kt)
    assert abs(w[0]) <= 1e-13 * w[-1] and np.all(w[1:] > 1e-6 * w[-1])
    g = np.array([0.7, -1.3, 0.4])
    T_ = xe @ g
    assert abs(T_ @ Kt @ T_ - g @ g * vol) <= 1e-13 * (g @ g) * vol


@pytest.mark.parametrize("box", [(1, 1, 1), (3, 2, 2), (4, 3, 5)])
def test_box_mesh(box):
    nx, ny, nz = box
    L = (1.3, 0.9, 0.7)
    conn, X = fe.tet10_mesh(nx, ny, nz, *L)
    _, X8 = fe.hex_mesh(2 * nx, 2 * ny, 2 * nz, *L)
    assert conn.shape == (6 * nx * ny * nz, 10) and np.array_equal(X, X8)
    assert np.array_equal(np.unique(conn), np.arange(len(X)))      # every lattice node is used
    xe = X[conn]
    vols = np.array([to.volume(x) for x in xe])
    assert np.all(vols > 0) and abs(vols.sum() - np.prod(L)) <= 1e-13
    for m, (i, j) in enumerate(to.EDGES):
        assert np.allclose(xe[:, 4 + m], 0.5 * (xe[:, i] + xe[:, j]), rtol=0, atol=1e-15)
    # conformity: every face is shared by two elements, or lies on the boundary
    faces = np.sort(np.concatenate([conn[:, f] for f in ([0, 1, 2, 4, 5, 6], [0, 1, 3, 4, 8, 7], [1, 2, 3, 5, 9, 8],
                                                         [0, 2, 3, 6, 9, 7])]), axis=1)
    _, cnt = np.unique(faces, axis=0, return_counts=True)
    assert set(cnt) <= {1, 2}
    assert np.sum(cnt == 1) == 4 * (nx * ny + ny * nz + nx * nz)   # two triangles per boundary cube face


def test_tet10_from_tet4_round_trip_and_orientation():
    conn, X = fe.tet10_mesh(2, 3, 2, 1.0, 0.8, 0.6)
    corners = np.unique(conn[:, :4])
    renum = np.full(len(X), -1)
    renum[corners] = np.arange(len(corners))
    conn4 = renum[conn[:, :4]]
    X4 = X[corners]
    rng = np.random.default_rng(1)
    flip = rng.random(len(conn4)) < 0.5
    c4 = conn4.copy()
    c4[flip, 1], c4[flip, 2] = conn4[flip, 2], conn4[flip, 1]
    c10, X10 = fe.tet10_from_tet4(c4, X4)
    assert c10.shape == conn.shape and X10.shape == X.shape           # one midside node per edge
    assert np.array_equal(c10[:, :4], conn4)                          # flipped back to positive volume
    assert np.allclose(X10[c10], X[conn], rtol=0, atol=1e-15)        # same elements, node for node
    assert np.all(np.array([to.volume(x) for x in X10[c10]]) > 0)


def test_tet10_from_tet4_refuses_degenerate_and_bad_shapes():
    X = np.array([[0.0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 1, 0]])
    with pytest.raises(ValueError, match="degenerate"):
        fe.tet10_from_tet4([[0, 1, 2, 3], [0, 1, 4, 2]], X)
    with pytest.raises(ValueError, match=r"needs conn \(nelems, 4\)"):
        fe.tet10_from_tet4([[0, 1, 2]], X)


@pytest.mark.parametrize("dof", [1, 3])
def test_symbolic_structures_of_t10_pattern_bit_exact(dof):
    conn, X = fe.tet10_mesh(3, 2, 2, 1.0, 0.8, 0.6)
    ndof = dof * X.shape[0]
    indptr, indices, _, _ = fe.assembly_structure(fe.element_dofs(conn, dof), ndof)
    A = sp.csr_matrix((np.ones(len(indices)), indices, indptr), shape=(ndof, ndof))
    sym = Symbolic(indptr, indices, ndof, coords=X, dof_per_node=dof)
    arr = sym.arrays()
    perm, snf = arr["perm"], arr["sn_first"]
    assert np.array_equal(np.sort(perm), np.arange(ndof))
    ns = len(snf) - 1
    parent_o, count_o = mo.etree_and_counts(A, perm)
    assert np.array_equal(arr["parent"], parent_o)
    assert np.array_equal(arr["colcount"], count_o)
    rows_o, snpar_o = mo.front_structures(A, perm, snf, parent_o)
    assert np.array_equal(arr["sn_parent"], snpar_o)
    rp = arr["sn_rowptr"]
    for k in range(ns):
        assert np.array_equal(arr["sn_rows"][rp[k]:rp[k + 1]], rows_o[k]), k
    assert sym.query("exact_nnzL") == int(count_o.sum())


@pytest.mark.parametrize("box,dof", [((3, 2, 2), 3), ((12, 10, 8), 1), ((8, 4, 4), 3)])
def test_pool_offsets_of_t10_meshes(box, dof):
    conn, X = fe.tet10_mesh(*box, 1.0, 0.8, 0.6)
    indptr, indices, _, _ = fe.assembly_structure(fe.element_dofs(conn, dof), dof * X.shape[0])
    pool, resident = check_pool(Symbolic(indptr, indices, dof * X.shape[0], coords=X, dof_per_node=dof))
    assert pool <= resident


def test_factory_defaults():
    sig = inspect.signature(T.make_natural_frequency_tet_model).parameters
    nx, ny, nz = (sig[k].default for k in ("nx", "ny", "nz"))
    assert (nx, ny, nz) == (32, 16, 16) and 3 * (2 * nx + 1) * (2 * ny + 1) * (2 * nz + 1) == 212355
    assert (sig["Lx"].default, sig["Ly"].default, sig["Lz"].default, sig["rfact"].default) == (2.0, 1.0, 1.0, 4.0)
    sig = inspect.signature(T.make_thermal_tet_model).parameters
    nx, ny, nz = (sig[k].default for k in ("nx", "ny", "nz"))
    assert (nx, ny, nz) == (40, 32, 24) and (2 * nx + 1) * (2 * ny + 1) * (2 * nz + 1) == 257985
    assert (sig["Lx"].default, sig["Ly"].default, sig["Lz"].default) == (1.0, 0.8, 0.6)
    assert sig["rfact"].default == 4.0 and sig["ftype"].default == "spatial"


@pytest.mark.parametrize("which", ["thermal", "nf"])
def test_factories_build_the_h8_lattice_and_filter_radius(monkeypatch, which):
    seen = {}

    def fake_filter(conn, X, r0=1.0, ftype="spatial", **kw):
        seen["filter"] = (conn, X, r0, ftype, kw)
        return "filter"

    def fake_analysis(fltr, conn, X, **kw):
        seen["analysis"] = (fltr, conn, X, kw)
        return "model"

    monkeypatch.setattr(fe, "NodeFilter", fake_filter)
    if which == "thermal":
        monkeypatch.setattr(T, "ThermalTopologyTetAnalysis", fake_analysis)
        assert T.make_thermal_tet_model(5, 4, 3, Lx=2.0, Ly=1.2, Lz=0.9, rfact=2.5, ftype="helmholtz", N=7,
                                        fronts="pooled") == "model"
        r0_h8 = 2.5 * 1.2 / 8                                      # make_thermal_3d_model(10, 8, 6, ...)
    else:
        monkeypatch.setattr(T, "NaturalFrequencyTetAnalysis", fake_analysis)
        assert T.make_natural_frequency_tet_model(5, 4, 3, Lx=2.0, Ly=1.2, Lz=0.9, rfact=2.5, N=7, fronts="pooled") == "model"
        r0_h8 = 2.5 * 1.2 / 8                                      # make_natural_frequency_3d_model(10, 8, 6, ...)
    conn, X, r0, ft, kw = seen["filter"]
    c_ref, X_ref = fe.tet10_mesh(5, 4, 3, 2.0, 1.2, 0.9)
    assert np.array_equal(conn, c_ref) and np.array_equal(X, X_ref)
    assert np.array_equal(X, fe.hex_mesh(10, 8, 6, 2.0, 1.2, 0.9)[1])
    assert r0 == pytest.approx(r0_h8) and ft == ("helmholtz" if which == "thermal" else "spatial") and kw == {}
    fltr, conn2, X2, kw2 = seen["analysis"]
    assert fltr == "filter" and conn2 is conn and X2 is X
    assert kw2 == {"N": 7, "fronts": "pooled"}


def test_the_tet_drivers_only_replace_the_element_model():
    for cls, base in ((T.ThermalTopologyTetAnalysis, T.ThermalTopologyAnalysis),
                      (T.NaturalFrequencyTetAnalysis, T.NaturalFrequency3DAnalysis)):
        own = set(vars(cls)) - {"__module__", "__doc__", "__qualname__", "__firstlineno__", "__static_attributes__"}
        assert own == {"_make_problem"} and issubclass(cls, base)


@pytest.mark.parametrize("cls", [fe.T10Problem, fe.T10ThermalProblem])
@pytest.mark.parametrize("conn_shape,X_shape", [((4, 8), (20, 3)), ((4, 10), (20, 2)), ((40,), (20, 3)), ((4, 10), (60,))])
def test_models_refuse_bad_shapes(cls, conn_shape, X_shape):
    with pytest.raises(ValueError, match=r"%s needs conn \(nelems, 10\) and X \(nnodes, 3\)" % cls.__name__):
        cls(np.zeros(conn_shape, dtype=np.int64), np.zeros(X_shape))


def test_helmholtz_filter_refuses_mismatched_tet_mesh():
    conn, X = fe.tet10_mesh(1, 1, 1)
    with pytest.raises(ValueError, match="2-D coordinates with 10-node conn"):
        fe.NodeFilter(conn, X[:, :2], r0=0.5, ftype="helmholtz")
    with pytest.raises(ValueError, match="3-D coordinates with 4-node conn"):
        fe.NodeFilter(conn[:, :4], X, r0=0.5, ftype="helmholtz")


@pytest.fixture(scope="module")
def box_eigenvalues():
    """The first 9 eigenvalues of the insulated 1 x 0.8 x 0.6 box on the 13 x 11 x 9 node lattice: T10 (6 x 5 x 4
    cubes) and H8 (12 x 10 x 8), unit conductivity and capacity, and the continuous Neumann Laplacian's."""
    from scipy.linalg import eigh
    L = (1.0, 0.8, 0.6)
    conn, X = fe.tet10_mesh(6, 5, 4, *L)
    K0, M0 = to.all_thermal_element_matrices(conn, X)
    one = np.ones(len(conn))
    K, M = to.assemble(conn, K0, M0, one, one, len(X))
    lt = eigh(K.toarray(), M.toarray(), eigvals_only=True, subset_by_index=[0, 8])
    c8, X8 = fe.hex_mesh(12, 10, 8, *L)
    assert np.array_equal(X8, X)
    K0, M0 = hto.all_element_matrices(c8, X8)
    one = np.ones(len(c8))
    K, M = hto.assemble(c8, K0, M0, one, one, len(X8))
    lh = eigh(K.toarray(), M.toarray(), eigvals_only=True, subset_by_index=[0, 8])
    exact = sorted(np.pi ** 2 * (i * i / L[0] ** 2 + j * j / L[1] ** 2 + k * k / L[2] ** 2)
                   for i in range(4) for j in range(4) for k in range(4))[:9]
    return lt, lh, np.array(exact)


def test_t10_eigenvalues_converge_to_the_continuous_box(box_eigenvalues):
    lt, _, exact = box_eigenvalues
    assert abs(lt[0]) < 1e-10 * lt[1]
    err = np.abs(lt[1:] - exact[1:]) / exact[1:]
    # the oracle gives 9.3e-5 .. 3.4e-3 on this lattice (the upper bound of the conforming element: lt >= exact)
    assert np.all(lt[1:] >= exact[1:]) and err.max() < 5e-3, err


def test_t10_is_closer_than_h8_on_the_same_nodes(box_eigenvalues):
    lt, lh, exact = box_eigenvalues
    assert np.all(np.abs(lt[1:] - exact[1:]) < np.abs(lh[1:] - exact[1:]))
