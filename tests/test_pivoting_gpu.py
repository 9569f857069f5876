"""Restricted Bunch-Kaufman pivoting of the device LDL^T (Factor(pivoting="bunch-kaufman"), diag_factor_bk_kernel)
against the numpy restatement (tests/bunch_kaufman_oracle.py) on the matrices of test_pivoting_cpu.py: the same pivot
decisions (inertia, 2x2 pivots, interchanges, no perturbation) and the same solutions; the thin-tile and front-mode
solve paths on a pivoted factor; SpLuOperator and the buckling driver with the option."""
import ctypes
import warnings

import numpy as np
import pytest

from conftest import load_golden
from test_pivoting_cpu import CASES, case_matrix, negative_eigenvalues, oracle_for, residual, zero_diagonal_matrix

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def D():
    from eigd_b200 import device
    device.init()
    return device


def rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(b).max(), 1e-300)


def device_factor(D, A, X, dof, pivoting="bunch-kaufman"):
    sym = D.Symbolic(A.indptr, A.indices, A.shape[0], coords=X, dof_per_node=dof)
    Ad = D.CsrDevice.from_scipy(A)
    fac = D.Factor(sym, max_rhs=32, pivoting=pivoting).numeric(Ad.data, sym.assembly_map_device(Ad.indptr, Ad.indices))
    return sym, fac


@pytest.mark.parametrize("kind,nx,ny,seed", CASES)
def test_bunch_kaufman_matches_oracle(D, kind, nx, ny, seed):
    A, X, dof = case_matrix(kind, nx, ny, seed)
    sym, fac = device_factor(D, A, X, dof)
    ref = oracle_for(A, X, dof).factor(A.data, pivoting="bunch-kaufman")
    # pivot decisions are comparisons of computed entries: the seeds are chosen so that none lies within rounding of
    # its threshold (GPU and numpy round differently, FMA vs separate products)
    print("%s %dx%d seed %d: smallest relative margin of a pivot test %.2e, counts %s"
          % (kind, nx, ny, seed, ref.margin, ref.counts))
    assert ref.margin > 1e-8
    info = fac.info()
    assert info["non_finite"] == 0 and info["perturbed_pivots"] == 0 and ref.counts["perturbed_pivots"] == 0
    for key in ("negative_pivots", "two_by_two_pivots", "interchanges"):
        assert info[key] == ref.counts[key], (key, info[key], ref.counts[key])
    assert info["negative_pivots"] == negative_eigenvalues(A)          # Sylvester inertia
    B = np.random.default_rng(seed + 200).normal(size=(A.shape[0], 4))
    x = fac.solve(D.to_device(B)).cpu().numpy()
    assert rel(x, ref.solve(B)) < 1e-10
    assert residual(A, x, B) < 1e-11


def test_static_factor_reports_no_pivot_counts(D):
    A, X, dof = case_matrix(*CASES[0])
    _, fac = device_factor(D, A, X, dof, pivoting="static")
    info = fac.info()
    assert info["perturbed_pivots"] > 0
    assert info["two_by_two_pivots"] == 0 and info["interchanges"] == 0


@pytest.mark.parametrize("nx,ny", [(250, 200), (160, 120)])
def test_bunch_kaufman_thin_tiles_and_front_mode(D, nx, ny):
    """Zero-diagonal operator at the sizes of test_factor_solve_front_mode (2 DOF per node): the solve plan has subtree
    phases (front mode) and upper-level fronts with 16- or 8-row tiles, whose skip bounds must cover the dense 32 x 32
    diagonal blocks of a pivoted factor."""
    from eigd_b200 import _lib
    A, X = zero_diagonal_matrix(nx, ny, nx + ny)
    n = A.shape[0]
    sym, fac = device_factor(D, A, X, 2)
    lib = _lib.load()
    meta = np.zeros(3, dtype=np.int64)
    lib.eigd_solve_plan_get(sym.handle, 148 * 16, 148, -2, 7, meta.ctypes.data_as(ctypes.c_void_p), 3)
    assert meta[0] >= 0, "expected subtree phases at this size"
    ths = []
    for which in (11, 12):
        cnt = lib.eigd_solve_plan_get(sym.handle, 148 * 16, 148, -2, which, None, 0)
        th = np.zeros(cnt, dtype=np.int64)
        lib.eigd_solve_plan_get(sym.handle, 148 * 16, 148, -2, which, th.ctypes.data_as(ctypes.c_void_p), cnt)
        ths.append(th)
    assert any(((th == 16) | (th == 8)).any() for th in ths), "expected thin tiles (height 16 or 8)"
    info = fac.info()
    assert info["perturbed_pivots"] == 0 and info["two_by_two_pivots"] > 0
    rng = np.random.default_rng(nx * ny)
    for k in (1, 2, 5, 10, 16, 24):
        B = rng.normal(size=(n, k))
        Bd = D.to_device(B)
        X1 = fac.solve(Bd).cpu().numpy()
        r = residual(A, X1, B)
        assert r <= 1e-11, (k, r)
        X2 = fac.solve(Bd).cpu().numpy()
        assert np.array_equal(X1, X2), "solve is not bitwise reproducible"


def test_spluoperator_bunch_kaufman(D):
    import eigd_b200 as E
    A, X = zero_diagonal_matrix(40, 30, 3)
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        op = E.SpLuOperator(A.tocsc(), coords=X, dof_per_node=2, pivoting="bunch-kaufman")
        info = op.info
        b = np.random.default_rng(1).normal(size=A.shape[0])
        x = op(b)
    assert info["perturbed_pivots"] == 0 and info["non_finite"] == 0 and info["two_by_two_pivots"] > 0
    assert info["negative_pivots"] == negative_eigenvalues(A)
    assert residual(A, x, b) <= 1e-12
    with pytest.raises(ValueError):
        E.SpLuOperator(A.tocsc(), pivoting="partial")
    with pytest.raises(ValueError):
        D.Factor(op.symbolic, pivoting="rook")


def test_buckling_bunch_kaufman_vs_golden(D):
    from eigd_b200 import topo
    g = load_golden("buckling_basiclanczos")
    E_, nu, p, rho0_K, rho0_G = (float(v) for v in g["material"])
    model = topo.make_buckling_model(nx=int(g["nx"]), ny=int(g["ny"]), N=int(g["N"]), m=int(g["m_max"]),
                                     sigma=float(g["sigma"]), solver_type="IRAM", adjoint_method="sibk",
                                     adjoint_options={"lanczos_guess": True, "update_guess": False, "bs_target": 1},
                                     rtol=1e-12, deriv_type="tensor", E=E_, nu=nu, p=p, rho0_K=rho0_K, rho0_G=rho0_G,
                                     pivoting="bunch-kaufman")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.initialize()
    assert model.factor.lu.pivoting == "bunch-kaufman" and model.Kfact.lu.pivoting == "static"
    assert rel(model.BLF, g["BLF"]) < 1e-10
    model.initialize_adjoint()
    model.add_eigenvector_aggregate_derivative(1.0, 100.0, int(g["node"]), mode="tanh")
    model.finalize_adjoint()
    assert rel(model.xb.cpu().numpy(), g["xb_sibk"]) < 1e-8
