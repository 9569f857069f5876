"""Linearised buckling of the H8 solid on the device (fe.BucklingH8Problem, topo.BucklingTopology3DAnalysis) against
tests/h8_buckling_oracle.py and dense references, on a perturbed mesh with random density:

  * element stresses and G_r(u) (1e-12) and K_r (1e-13) against the oracle and scipy's fancy-indexed reduction;
  * the fundamental path against scipy.sparse.linalg.spsolve (1e-10);
  * the dGdu / dGdx / dKdx callbacks against the oracle's einsum (1e-11) for host and device operands, and the
    linearity identity sum_k w_k^T G_r(u) v_k = u^T dGdu(W, V);
  * load factors of a small column against dense eigh of the (G_r, K_r) pencil, with both pivot strategies of the
    indefinite shifted factor;
  * design gradients of the tanh eigenvector aggregate (IRAM + sibk, BasicLanczos) and of the KS buckling measure
    against central differences, with simple modes asserted first;
  * bitwise-reproducible load factors and modes."""
import warnings

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
P, RHO0_K, RHO0_G, E, NU = 3.0, 1e-6, 1e-9, 1.7, 0.27


def rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(b).max(), 1e-300)


@pytest.fixture(scope="module")
def column():
    import h8_buckling_oracle as hbo
    import h8_oracle as ho
    import scipy.sparse.linalg as sla
    from eigd_b200 import device as D, fe, topo
    D.init()
    nx, ny, nz, L = 4, 3, 6, (1.0, 0.75, 1.5)
    conn, _, bcs, forces = topo.domain_compressed_column_3d(nx, ny, nz, *L)
    X = ho.perturbed_box(nx, ny, nz, L, amp=0.25, seed=5)                 # base and top faces stay in place
    pr = fe.BucklingH8Problem(conn, X, bcs, forces, E=E, nu=NU, p=P, rho0_K=RHO0_K, rho0_G=RHO0_G)
    rhoE = np.random.default_rng(6).uniform(0.2, 1.0, pr.nelems)
    pr.set_density(rhoE=rhoE)
    o = hbo.H8BucklingOracle(conn, X, E=E, nu=NU)
    K0, _ = ho.all_element_matrices(conn, X, E, NU)
    ks, kg = rhoE**P + RHO0_K, rhoE**P + RHO0_G
    K, _ = ho.assemble(conn, K0, K0, ks, ks, pr.ndof)
    red = pr.reduced
    Kr = K[red, :][:, red]
    ur = sla.spsolve(Kr.tocsc(), pr.f[red])
    u = np.zeros(pr.ndof)
    u[red] = ur
    G0 = o.G0(u)
    G, _ = ho.assemble(conn, G0, G0, kg, kg, pr.ndof)
    ref = dict(o=o, K0=K0, G0=G0, Kr=Kr, Gr=G[red, :][:, red], u=u, ur=ur, rhoE=rhoE, kg=kg, dk=P * rhoE ** (P - 1.0),
               dkg=P * rhoE ** (P - 1.0))
    return pr, ref


def test_stiffness_stress_and_stress_stiffness_match_oracle(column):
    from eigd_b200 import device as D
    pr, ref = column
    Kr = pr.assemble_K().to_scipy()
    Kr_o = ref["Kr"]
    Kr_o.sort_indices()
    assert np.array_equal(pr.indptr, Kr_o.indptr) and np.array_equal(pr.indices, Kr_o.indices)
    assert rel(Kr.data, Kr_o.data) < 1e-13
    pr.set_displacement(D.to_device(ref["ur"]))
    Gr = pr.assemble_G().to_scipy()
    Gr_o = ref["Gr"]
    Gr_o.sort_indices()
    assert np.array_equal(Gr.indptr, Gr_o.indptr) and np.array_equal(Gr.indices, Gr_o.indices)
    assert rel(Gr.data, Gr_o.data) < 1e-12
    assert rel(pr.stress_d.cpu().numpy(), ref["o"].stresses(ref["u"], ref["kg"])) < 1e-12
    assert rel(pr.G0_d.cpu().numpy().reshape(ref["G0"].shape), ref["G0"]) < 1e-12


def test_fundamental_path_matches_spsolve(column):
    from eigd_b200.eigenvector_derivatives import SpLuOperator
    pr, ref = column
    Kr = pr.assemble_K()
    ur = SpLuOperator(Kr, max_rhs=1).solve_dev(pr.fr_d)
    assert rel(ur.cpu().numpy(), ref["ur"]) < 1e-10
    assert rel(pr.set_displacement(ur).cpu().numpy(), ref["u"]) < 1e-10


@pytest.mark.parametrize("N", [1, 3, 8, 13, 32])
@pytest.mark.parametrize("operands", ["host", "device"])
def test_callbacks_match_oracle_einsum(column, N, operands):
    from eigd_b200 import device as D
    pr, ref = column
    o = ref["o"]
    pr.set_displacement(D.to_device(ref["ur"]))
    Gr = pr.assemble_G().to_scipy()
    rng = np.random.default_rng(N)
    W, V = rng.normal(size=(pr.nred, N)), rng.normal(size=(pr.nred, N))
    Wf, Vf = np.zeros((pr.ndof, N)), np.zeros((pr.ndof, N))
    Wf[pr.reduced], Vf[pr.reduced] = W, V
    args = (W, V) if operands == "host" else (D.to_device(W), D.to_device(V))
    out = [pr.dGdu(*args), pr.dGdx(*args), pr.dKdx(*args)]
    if operands == "device":
        assert all(t.is_cuda for t in out)
        out = [t.cpu().numpy() for t in out]
    du, dx, dk = out
    assert du.shape == (pr.ndof,) and dx.shape == (pr.nelems,) and dk.shape == (pr.nelems,)
    assert rel(du, o.dG_du(ref["kg"], Wf, Vf)) < 1e-11
    assert rel(dx, o.quadform(ref["G0"], ref["dkg"], Wf, Vf)) < 1e-11
    assert rel(dk, o.quadform(ref["K0"], ref["dk"], Wf, Vf)) < 1e-11
    lhs = float(np.sum(W * (Gr @ V)))
    assert abs(lhs - float(ref["u"] @ du)) <= 1e-11 * abs(lhs)
    psi = rng.normal(size=pr.ndof)
    single = pr.dK_single(D.to_device(psi), D.to_device(ref["u"])).cpu().numpy()
    assert rel(single, o.quadform(ref["K0"], ref["dk"], psi[:, None], ref["u"][:, None])) < 1e-11


def _model(N=6, solver_type="IRAM", **kw):
    from eigd_b200 import topo
    return topo.make_buckling_3d_model(4, 3, 16, 1.0, 0.75, 4.0, rfact=1.5, N=N, m=40, solver_type=solver_type, seed=0,
                                       rtol=1e-12, adjoint_options={"lanczos_guess": True}, **kw)


def _initialize(model, x):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.initialize(x=x)


@pytest.mark.parametrize("pivoting", ["static", "bunch-kaufman"])
def test_load_factors_match_dense_eigh(pivoting):
    from scipy.linalg import eigh
    from eigd_b200 import device as D
    D.init()
    model = _model(pivoting=pivoting, tol=1e-14)
    _initialize(model, np.random.default_rng(7).uniform(0.3, 0.7, model.fltr.num_design_vars))
    Kr, Gr = model.Kr.to_scipy().toarray(), model.Gr.to_scipy().toarray()
    mu = eigh(-Gr, Kr, eigvals_only=True)                                     # K phi + BLF G phi = 0: mu = 1 / BLF
    blf_ref = np.sort(1.0 / mu[mu > 0])
    blf = np.asarray(model.BLF)
    nearest = blf_ref[np.argmin(np.abs(blf_ref[None, :] - blf[:, None]), axis=1)]
    assert rel(blf, nearest) < 1e-10
    assert len(np.unique(nearest)) == len(blf)
    below = int(np.count_nonzero(blf_ref < model.sigma))
    assert below > 0 and blf_ref[0] in nearest
    info = model.factor.info
    assert info["negative_pivots"] > 0 and info["non_finite"] == 0, info
    if pivoting == "static" and info["perturbed_pivots"] == 0:
        assert info["negative_pivots"] == below                              # inertia of K_r + sigma G_r


def _simple(model):
    blf = np.sort(np.asarray(model.BLF))
    assert np.min(np.diff(blf)) > 1e-3 * blf[-1], blf


@pytest.mark.parametrize("solver_type", ["IRAM", "BasicLanczos"])
def test_eigenvector_aggregate_gradient_matches_central_difference(solver_type):
    from eigd_b200 import device as D
    D.init()
    model = _model(solver_type=solver_type, tol=1e-14 if solver_type == "BasicLanczos" else 0.0)
    rng = np.random.default_rng(8)
    x0 = rng.uniform(0.3, 0.7, model.fltr.num_design_vars)
    p = rng.uniform(-1.0, 1.0, x0.shape)
    _initialize(model, x0)
    _simple(model)
    node = int(np.argmax(np.abs(model.prob.full_vector(model.Qr[:, 0].contiguous()).cpu().numpy())))
    model.initialize_adjoint()
    model.add_eigenvector_aggregate_derivative(1.0, 100.0, node, mode="tanh")
    model.finalize_adjoint()
    g = float(model.xb.cpu().numpy() @ p)
    h = 1e-5
    fs = []
    for s in (1.0, -1.0):
        _initialize(model, x0 + s * h * p)
        fs.append(model.get_eigenvector_aggregate(100.0, node, mode="tanh"))
    fd = (fs[0] - fs[1]) / (2 * h)
    assert abs(g - fd) <= 1e-6 * abs(fd), (g, fd)


def test_ks_buckling_gradient_matches_central_difference():
    from eigd_b200 import device as D
    D.init()
    model = _model()
    rng = np.random.default_rng(9)
    x0 = rng.uniform(0.3, 0.7, model.fltr.num_design_vars)
    p = rng.uniform(-1.0, 1.0, x0.shape)
    _initialize(model, x0)
    _simple(model)
    g = float(model.eval_ks_buckling_derivative(ks_rho=10.0) @ p)
    h = 1e-5
    fs = []
    for s in (1.0, -1.0):
        _initialize(model, x0 + s * h * p)
        fs.append(model.eval_ks_buckling(ks_rho=10.0))
    fd = (fs[0] - fs[1]) / (2 * h)
    assert abs(g - fd) <= 1e-6 * abs(fd), (g, fd)


def test_evaluations_are_bitwise_reproducible():
    from eigd_b200 import device as D
    D.init()
    x0 = np.random.default_rng(10).uniform(0.3, 0.7, _model().fltr.num_design_vars)
    a, b = _model(), _model()
    _initialize(a, x0)
    _initialize(b, x0)
    assert np.array_equal(a.BLF, b.BLF)
    assert torch.equal(a.Qr, b.Qr)
    _initialize(a, x0)                                   # second design on the same model: old factors dropped first
    assert np.array_equal(a.BLF, b.BLF)
    assert torch.equal(a.Qr, b.Qr)
