"""The quadratic tetrahedron (T10) on the device: T10Problem, T10ThermalProblem, their drivers
(NaturalFrequencyTetAnalysis, ThermalTopologyTetAnalysis) and the Helmholtz filter on T10 meshes, against
tests/t10_oracle.py and dense / scipy references:

  * unit element matrices of a perturbed (curved) mesh (1e-13), also with a partial last warp, and the thermal capacity
    against the scalar block of the solid's mass matrix (bit for bit);
  * assembled K and M against scipy's COO assembly, the fused sensitivities against the oracle's einsum, the tangent
    assembly against its definition and a central difference;
  * eigenpairs of a small free solid (six rigid modes dropped) and of an insulated box against scipy.linalg.eigh;
  * the design gradients of both drivers against a central difference and the dual-number (complex-step) directional
    derivative of BasicLanczos, with the conic and the Helmholtz filter;
  * the T10 Helmholtz filter against scipy's spsolve, its transpose and tangent;
  * pooled and resident fronts give bitwise equal eigenpairs and gradients;
  * with two GPUs, element-range-sharded sensitivities against the unsharded ones."""
import os
import socket
import sys
import warnings

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P, RHO0, BETA = 3.0, 1e-6, 1e-6
E_, NU, DENS = 2.0, 0.28, 1.7


def rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(b).max(), 1e-300)


@pytest.fixture(scope="module")
def meshes():
    import t10_oracle as to
    from eigd_b200 import device as D, fe
    D.init()
    nx, ny, nz = 3, 2, 2
    conn, _ = fe.tet10_mesh(nx, ny, nz)
    X = to.perturbed_tet_box(nx, ny, nz, (1.5, 1.0, 0.8), amp=0.15, seed=3)
    solid = fe.T10Problem(conn, X, E=E_, nu=NU, density=DENS, p=P, rho0_K=RHO0)
    thermal = fe.T10ThermalProblem(conn, X, kappa=1.3, density=1.7, heat_capacity=0.6, p=P, beta=BETA)
    return {"solid": (solid, *to.all_element_matrices(conn, X, E_, NU, DENS)),
            "thermal": (thermal, *to.all_thermal_element_matrices(conn, X))}


def _law(kind, rhoE):
    """ks, ms, dk, dm of the model's material law."""
    if kind == "solid":
        return rhoE ** P + RHO0, rhoE, P * rhoE ** (P - 1.0), np.ones_like(rhoE)
    import h8_thermal_oracle as hto
    return hto.thermal_law(rhoE, P, 1.3, 1.7 * 0.6, BETA)


def test_element_matrices_match_oracle(meshes):
    from eigd_b200 import fe
    for kind, (prob, K0, M0) in meshes.items():
        Kd = prob.K0_d.cpu().numpy().reshape(K0.shape)
        Md = prob.M0_d.cpu().numpy().reshape(M0.shape)
        assert rel(Kd, K0) < 1e-13, kind
        assert rel(Md, M0) < 1e-13, kind
    thermal = meshes["thermal"][0]
    unit = fe.T10Problem(thermal.conn, thermal.X, density=1.0)
    Ms = unit.M0_d.cpu().numpy().reshape(-1, 30, 30)
    Mt = thermal.M0_d.cpu().numpy().reshape(-1, 10, 10)
    assert np.array_equal(Mt, Ms[:, ::3, ::3])
    assert not Ms[:, ::3, 1::3].any()


def test_element_matrices_of_a_partial_last_warp():
    """Odd element counts leave the second 16-lane group of the thermal kernel's last warp without an element."""
    import t10_oracle as to
    from eigd_b200 import device as D, fe
    D.init()
    conn, X = fe.tet10_mesh(1, 1, 1, 0.5, 0.7, 0.9)
    for ne in (1, 3, 5, 6):
        c = conn[:ne]
        used = np.unique(c)
        renum = np.full(len(X), -1)
        renum[used] = np.arange(len(used))
        c, Xe = renum[c], X[used]
        s, t = fe.T10Problem(c, Xe), fe.T10ThermalProblem(c, Xe)
        K0, M0 = to.all_element_matrices(c, Xe, 1.0, 0.3, 1.0)
        Kt, Mt = to.all_thermal_element_matrices(c, Xe)
        assert rel(s.K0_d.cpu().numpy().reshape(K0.shape), K0) < 1e-13
        assert rel(s.M0_d.cpu().numpy().reshape(M0.shape), M0) < 1e-13
        assert rel(t.K0_d.cpu().numpy().reshape(Kt.shape), Kt) < 1e-13
        assert rel(t.M0_d.cpu().numpy().reshape(Mt.shape), Mt) < 1e-13


@pytest.mark.parametrize("kind", ["solid", "thermal"])
def test_assembly_matches_scipy_coo(meshes, kind):
    import t10_oracle as to
    prob, K0, M0 = meshes[kind]
    rhoE = np.random.default_rng(4).uniform(0.2, 1.0, prob.nelems)
    prob.set_density(rhoE=rhoE)
    K, M = prob.assemble()
    ks, ms, _, _ = _law(kind, rhoE)
    Ko, Mo = to.assemble(prob.var, K0, M0, ks, ms, prob.ndof)
    for A, B in ((K.to_scipy(), Ko), (M.to_scipy(), Mo)):
        assert np.array_equal(A.indptr, B.indptr) and np.array_equal(A.indices, B.indices)
        assert rel(A.data, B.data) < 1e-13


@pytest.mark.parametrize("kind", ["solid", "thermal"])
@pytest.mark.parametrize("N", [1, 7, 16])
def test_fused_sensitivities_match_einsum(meshes, kind, N):
    import t10_oracle as to
    from eigd_b200 import device as D
    prob, K0, M0 = meshes[kind]
    rng = np.random.default_rng(N)
    rhoE = rng.uniform(0.2, 1.0, prob.nelems)
    prob.set_density(rhoE=rhoE)
    WA, WB, V = (rng.normal(size=(prob.ndof, N)) for _ in range(3))
    _, _, dk, dm = _law(kind, rhoE)
    ref = to.fused_sensitivities(prob.var, K0, M0, dk, dm, WA, WB, V, 0.7, -1.3)
    out = prob.device_call_fused(D.to_device(WA), D.to_device(WB), D.to_device(V), 0.7, -1.3).cpu().numpy()
    assert rel(out, ref) < 1e-12
    assert rel(prob.dAdx(WA, V), to.fused_sensitivities(prob.var, K0, M0, dk, dm, WA, WB, V, 1.0, 0.0)) < 1e-12
    assert rel(prob.dBdx(WB, V), to.fused_sensitivities(prob.var, K0, M0, dk, dm, WA, WB, V, 0.0, 1.0)) < 1e-12


@pytest.mark.parametrize("kind", ["solid", "thermal"])
def test_tangent_assembly(meshes, kind):
    import t10_oracle as to
    from eigd_b200 import device as D
    prob, K0, M0 = meshes[kind]
    rng = np.random.default_rng(5)
    rho, rho_t = rng.uniform(0.3, 1.0, prob.nnodes), rng.normal(size=prob.nnodes)
    prob.set_density(rho=D.to_device(rho))
    assert rel(prob.rhoE_d.cpu().numpy(), rho[prob.conn].mean(axis=1)) < 1e-15
    Kt, Mt = prob.assemble_tangent(D.to_device(rho_t))
    rhoE, rhoEt = rho[prob.conn].mean(axis=1), rho_t[prob.conn].mean(axis=1)
    _, _, dk, dm = _law(kind, rhoE)
    Ko, Mo = to.assemble(prob.var, K0, M0, dk * rhoEt, dm * rhoEt, prob.ndof)
    assert rel(Kt.to_scipy().data, Ko.data) < 1e-12
    assert rel(Mt.to_scipy().data, Mo.data) < 1e-12
    h = 1e-5
    vals = []
    for s in (1.0, -1.0):
        prob.set_density(rho=D.to_device(rho + s * h * rho_t))
        K, M = prob.assemble()
        vals.append((K.to_scipy().data, M.to_scipy().data))
    assert rel((vals[0][0] - vals[1][0]) / (2 * h), Kt.to_scipy().data) < 1e-7
    assert rel((vals[0][1] - vals[1][1]) / (2 * h), Mt.to_scipy().data) < 1e-7


def test_scatter_to_nodes_is_the_transpose_of_the_element_mean(meshes):
    prob = meshes["solid"][0]
    ev = np.random.default_rng(8).normal(size=prob.nelems)
    ref = np.zeros(prob.nnodes)
    np.add.at(ref, prob.conn.ravel(), np.repeat(ev, 10) / 10.0)
    assert rel(prob.scatter_to_nodes(ev), ref) < 1e-14


def _nf_model(nx, ny, nz, L, N, solver_type="IRAM", ftype="spatial", **kw):
    from eigd_b200 import fe, topo as T
    opts = dict(rfact=1.5, N=N, solver_type=solver_type, seed=0, rtol=1e-12, adjoint_options={"lanczos_guess": True},
                tol=1e-14, **kw)
    if ftype == "spatial":
        return T.make_natural_frequency_tet_model(nx, ny, nz, *L, **opts)
    conn, X = fe.tet10_mesh(nx, ny, nz, *L)
    fltr = fe.NodeFilter(conn, X, r0=opts.pop("rfact") * L[1] / (2 * ny), ftype="helmholtz")
    return T.NaturalFrequencyTetAnalysis(fltr, conn, X, **opts)


def _thermal_model(nx, ny, nz, N, solver_type="IRAM", **kw):
    from eigd_b200 import topo as T
    return T.make_thermal_tet_model(nx, ny, nz, rfact=1.5, N=N, solver_type=solver_type, seed=0, rtol=1e-12, tol=1e-14,
                                    adjoint_options={"lanczos_guess": True}, **kw)


def test_free_solid_eigenpairs_match_dense():
    from scipy.linalg import eigh
    from eigd_b200 import device as D
    D.init()
    model = _nf_model(3, 2, 2, (2.0, 1.1, 0.9), N=8)
    assert model.nvars == 3 * 7 * 5 * 5 and model.nrigid == 6
    model.initialize(x=np.random.default_rng(6).uniform(0.4, 1.0, model.nnodes))
    K, M = model.K.to_scipy().toarray(), model.M.to_scipy().toarray()
    lam_ref = eigh(K, M, eigvals_only=True)
    lam0 = np.asarray(model.lam0)
    assert np.all(np.abs(lam0[:6]) < 1e-8 * lam_ref[6])
    assert rel(model.lam, lam_ref[6:6 + 8]) < 1e-10
    Phi = model.Q0.cpu().numpy()
    assert np.abs(Phi.T @ M @ Phi - np.eye(Phi.shape[1])).max() < 1e-10


def test_insulated_box_eigenpairs_match_dense():
    from scipy.linalg import eigh
    from eigd_b200 import device as D
    D.init()
    N = 8
    model = _thermal_model(3, 3, 2, N=N)
    assert model.nvars == 7 * 7 * 5
    model.initialize(x=np.random.default_rng(6).uniform(0.4, 1.0, model.nnodes))
    K, M = model.K.to_scipy().toarray(), model.M.to_scipy().toarray()
    lam_ref = eigh(K, M, eigvals_only=True)
    lam = np.asarray(model.lam)
    assert abs(lam_ref[0]) < 1e-10 * lam_ref[1] and abs(lam[0]) < 1e-10 * lam_ref[1]
    assert rel(lam[1:], lam_ref[1:N]) < 1e-10
    Phi = model.Q.cpu().numpy()
    assert np.abs(Phi.T @ M @ Phi - np.eye(N)).max() < 1e-10


def _nf_objective(model, w_d):
    from eigd_b200 import device as D
    c = D.col_dot(model.Q, w_d).cpu().numpy()
    return float(np.sum(model.get_frequencies()) + np.sum(c ** 2))


@pytest.mark.parametrize("ftype", ["spatial", "helmholtz"])
def test_natural_frequency_gradient_matches_central_difference_and_dual_numbers(ftype):
    from eigd_b200 import device as D
    D.init()
    N, L = 4, (2.0, 1.1, 0.7)
    model = _nf_model(3, 2, 1, L, N=N, ftype=ftype)
    rng = np.random.default_rng(7)
    x0 = rng.uniform(0.4, 1.0, model.nnodes)
    p = rng.uniform(-1.0, 1.0, model.nnodes)
    w = rng.normal(size=(model.nvars, N))
    w_d = D.to_device(w)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.initialize(x=x0)
    lam = np.array(model.lam)
    assert np.min(np.diff(lam)) > 1e-3 * lam[-1]                       # simple modes
    model.initialize_adjoint()
    model.add_frequency_derivatives(np.ones(N))
    model.add_modal_function_derivative(w_d)
    model.finalize_adjoint()
    g = float(model.xb.cpu().numpy() @ p)
    h = 1e-5
    fs = []
    for s in (1.0, -1.0):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model.initialize(x=x0 + s * h * p)
        fs.append(_nf_objective(model, w_d))
    fd = (fs[0] - fs[1]) / (2 * h)
    assert abs(g - fd) <= 1e-6 * abs(fd), (g, fd)
    dual = _nf_model(3, 2, 1, L, N=N, solver_type="BasicLanczos", ftype=ftype)
    dual.initialize(x=x0 + 1j * p)
    # single-vector Lanczos resolves the six-fold zero eigenvalue only in part: take the flexible modes by value
    lam0_c = np.asarray(dual.lam0)
    idx = [int(np.argmin(np.abs(lam0_c.real - v))) for v in lam]
    assert rel(lam0_c.real[idx], lam) < 1e-8, (lam0_c, lam)
    lam_c, Q_c = lam0_c[idx], np.asarray(dual.Q0)[:, idx]
    c_r, c_t = np.einsum("ij,ij->j", Q_c.real, w), np.einsum("ij,ij->j", Q_c.imag, w)
    d_dual = float(np.sum(0.5 * lam_c.imag / np.sqrt(lam_c.real)) + np.sum(2.0 * c_r * c_t))
    assert abs(g - d_dual) <= 1e-8 * abs(d_dual), (g, d_dual)


def _thermal_objective(model, vec):
    return model.get_thermal_compliance(vec) + np.sum(np.asarray(model.lam)[1:])


@pytest.mark.parametrize("ftype", ["spatial", "helmholtz"])
def test_thermal_gradient_matches_central_difference_and_dual_numbers(ftype):
    from eigd_b200 import device as D
    D.init()
    N = 5
    model = _thermal_model(3, 2, 2, N=N, ftype=ftype)
    rng = np.random.default_rng(7)
    x0 = rng.uniform(0.4, 1.0, model.nnodes)
    p = rng.uniform(-1.0, 1.0, model.nnodes)
    vec = rng.uniform(size=model.nnodes)
    vec_d = D.to_device(vec)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.initialize(x=x0)
    lam = np.asarray(model.lam)
    assert abs(lam[0]) < 1e-10 * lam[1]
    assert np.min(np.diff(lam[1:])) > 1e-3 * lam[-1]                   # simple modes
    model.initialize_adjoint()
    model.add_thermal_compliance_derivative(1.0, vec_d)
    model.lamb[1:] += 1.0
    model.finalize_adjoint()
    g = float(model.xb.cpu().numpy() @ p)
    h = 1e-5
    fs = []
    for s in (1.0, -1.0):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model.initialize(x=x0 + s * h * p)
        fs.append(_thermal_objective(model, vec_d))
    fd = (fs[0] - fs[1]) / (2 * h)
    assert abs(g - fd) <= 1e-6 * abs(fd), (g, fd)
    dual = _thermal_model(3, 2, 2, N=N, ftype=ftype, solver_type="BasicLanczos")
    dual.initialize(x=x0 + 1j * p)
    lam_c, Q_c = np.asarray(dual.lam), np.asarray(dual.Q)
    c_r, c_t = Q_c.real.T @ vec, Q_c.imag.T @ vec
    l_r, l_t = lam_c.real[1:], lam_c.imag[1:]
    d_dual = float(np.sum((2.0 * c_r[1:] * c_t[1:] * l_r - c_r[1:] ** 2 * l_t) / l_r ** 2) + np.sum(l_t))
    assert abs(g - d_dual) <= 1e-8 * abs(d_dual), (g, d_dual)


@pytest.mark.parametrize("projection", [False, True])
def test_helmholtz_filter_on_t10(projection):
    import scipy.sparse.linalg as spla
    import t10_oracle as to
    from eigd_b200 import device as D, fe
    D.init()
    nx, ny, nz = 3, 2, 2
    conn, _ = fe.tet10_mesh(nx, ny, nz)
    X = to.perturbed_tet_box(nx, ny, nz, (1.2, 0.8, 0.6), amp=0.15, seed=12)
    r0 = 0.35
    flt = fe.NodeFilter(conn, X, r0=r0, ftype="helmholtz", projection=projection, beta=8.0, eta=0.45)
    K0, M0 = to.all_thermal_element_matrices(conn, X)
    ones = np.ones(len(conn))
    Ko, Mo = to.assemble(conn, K0, M0, ones, ones, X.shape[0])
    rng = np.random.default_rng(13)
    x = rng.uniform(0.1, 1.0, flt.num_design_vars)
    rho_ref = spla.spsolve((r0 ** 2 * Ko + Mo).tocsc(), Mo @ x)
    if projection:
        t = np.tanh
        rho_ref = (t(8.0 * 0.45) + t(8.0 * (rho_ref - 0.45))) / (t(8.0 * 0.45) + t(8.0 * 0.55))
    assert rel(flt.apply(x), rho_ref) < 1e-12
    xt, g = rng.normal(size=x.shape), rng.normal(size=X.shape[0])
    Fxt = flt.apply_tangent(D.to_device(x), D.to_device(xt)).cpu().numpy()
    FTg = flt.apply_gradient(g, x)
    assert abs(Fxt @ g - xt @ FTg) <= 1e-12 * np.abs(Fxt).max() * np.abs(g).sum()
    h = 1e-6
    fd = (flt.apply(x + h * xt) - flt.apply(x - h * xt)) / (2 * h)
    assert rel(Fxt, fd) < 1e-7
    assert flt._hA.lu.fronts == "pooled" and isinstance(flt._hprob, fe.T10ThermalProblem)


@pytest.mark.parametrize("kind", ["solid", "thermal"])
def test_pooled_and_resident_fronts_are_bitwise_equal(kind):
    from eigd_b200 import device as D
    D.init()
    N = 5
    rng = np.random.default_rng(14)
    out = []
    for fronts in ("resident", "pooled"):
        model = _nf_model(4, 2, 2, (2.0, 1.1, 0.9), N=N, fronts=fronts) if kind == "solid" else \
            _thermal_model(4, 3, 2, N=N, fronts=fronts)
        if not out:
            x0 = rng.uniform(0.3, 1.0, model.nnodes)
            vec = D.to_device(rng.uniform(size=(model.nvars, N)))
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model.initialize(x=x0)
        model.initialize_adjoint()
        if kind == "solid":
            model.add_modal_function_derivative(vec)
        else:
            model.add_thermal_compliance_derivative(1.0, vec[:, 0].contiguous())
        model.finalize_adjoint()
        assert model.factor.lu.fronts == fronts
        out.append((np.asarray(model.lam).copy(), model.Q.cpu().numpy(), model.xb.cpu().numpy()))
    for a, b in zip(out[0], out[1]):
        assert np.array_equal(a, b)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _sharded_worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    try:
        from eigd_b200 import device as D, fe
        from eigd_b200.dist import ModeSharding
        D.init("cuda:%d" % rank)
        conn, X = fe.tet10_mesh(4, 3, 2, 1.4, 1.0, 0.8)
        errs = []
        for prob in (fe.T10Problem(conn, X), fe.T10ThermalProblem(conn, X)):
            rng = np.random.default_rng(10)
            prob.set_density(rhoE=rng.uniform(0.2, 1.0, prob.nelems))
            WA, WB, V = (D.to_device(rng.normal(size=(prob.ndof, 5))) for _ in range(3))
            ref = prob.device_call_fused(WA, WB, V, 1.0, -1.0)
            prob.sharding = ModeSharding()
            got = prob.device_call_fused(WA, WB, V, 1.0, -1.0)
            errs.append(float((got - ref).abs().max() / ref.abs().max()))
        if rank == 0:
            out.put(max(errs))
    finally:
        dist.destroy_process_group()


def test_sharded_sensitivities_match_unsharded():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_sharded_worker, args=(r, 2, port, q)) for r in range(2)]
    for pr in procs:
        pr.start()
    err = q.get(timeout=600)
    for pr in procs:
        pr.join(timeout=600)
    assert err <= 1e-12
