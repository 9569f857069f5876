"""The 3-D heat-conduction model (H8ThermalProblem, ThermalTopology3DAnalysis) and the Helmholtz filter on hexahedral
meshes on the device, against tests/h8_thermal_oracle.py and dense / scipy references:

  * unit element matrices of a perturbed mesh (1e-13) and their capacity block against the solid's mass matrix (bit for
    bit), assembled K and M against scipy's COO assembly, the fused sensitivities against the oracle's einsum, the
    tangent assembly against its definition and a central difference;
  * eigenpairs of a small insulated box against scipy.linalg.eigh (one zero eigenvalue, the next ones to 1e-10);
  * the design gradient of thermal compliance + sum lambda against a central difference and the dual-number
    (complex-step) directional derivative of BasicLanczos, with the conic and the Helmholtz filter;
  * the 3-D Helmholtz filter against scipy's spsolve, its transpose and tangent, with and without a design-variable map
    and projection, and its pooled factor;
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
P, BETA = 3.0, 1e-6


def rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(b).max(), 1e-300)


@pytest.fixture(scope="module")
def mesh():
    import h8_oracle as ho
    import h8_thermal_oracle as hto
    from eigd_b200 import device as D, fe
    D.init()
    nx, ny, nz = 5, 4, 3
    conn, _ = fe.hex_mesh(nx, ny, nz)
    X = ho.perturbed_box(nx, ny, nz, (1.5, 1.0, 0.8), amp=0.25, seed=3)
    prob = fe.H8ThermalProblem(conn, X, kappa=1.3, density=1.7, heat_capacity=0.6, p=P, beta=BETA)
    K0, M0 = hto.all_element_matrices(conn, X)
    return prob, K0, M0


def _law(rhoE):
    import h8_thermal_oracle as hto
    return hto.thermal_law(rhoE, P, 1.3, 1.7 * 0.6, BETA)


def test_element_matrices_match_oracle(mesh):
    from eigd_b200 import fe
    prob, K0, M0 = mesh
    Kd = prob.K0_d.cpu().numpy().reshape(K0.shape)
    Md = prob.M0_d.cpu().numpy().reshape(M0.shape)
    assert rel(Kd, K0) < 1e-13
    assert rel(Md, M0) < 1e-13
    assert np.array_equal(Kd, Kd.transpose(0, 2, 1))
    solid = fe.H8Problem(prob.conn, prob.X, density=1.0)
    Ms = solid.M0_d.cpu().numpy().reshape(-1, 24, 24)
    assert np.array_equal(Md, Ms[:, ::3, ::3])


def test_element_matrices_of_a_partial_last_warp():
    """Element counts that are not a multiple of four leave lanes of the last warp without an element of their own."""
    import h8_thermal_oracle as hto
    from eigd_b200 import device as D, fe
    D.init()
    for nx in (1, 2, 3, 5):
        conn, X = fe.hex_mesh(nx, 1, 1, 0.5 * nx, 0.7, 0.9)
        prob = fe.H8ThermalProblem(conn, X)
        K0, M0 = hto.all_element_matrices(conn, X)
        assert rel(prob.K0_d.cpu().numpy().reshape(K0.shape), K0) < 1e-13
        assert rel(prob.M0_d.cpu().numpy().reshape(M0.shape), M0) < 1e-13


def test_assembly_matches_scipy_coo(mesh):
    import h8_thermal_oracle as hto
    prob, K0, M0 = mesh
    rhoE = np.random.default_rng(4).uniform(0.2, 1.0, prob.nelems)
    prob.set_density(rhoE=rhoE)
    K, M = prob.assemble()
    ks, ms, _, _ = _law(rhoE)
    Ko, Mo = hto.assemble(prob.conn, K0, M0, ks, ms, prob.ndof)
    Kd, Md = K.to_scipy(), M.to_scipy()
    for A, B in ((Kd, Ko), (Md, Mo)):
        assert np.array_equal(A.indptr, B.indptr) and np.array_equal(A.indices, B.indices)
        assert rel(A.data, B.data) < 1e-13


@pytest.mark.parametrize("N", [1, 7, 16])
def test_fused_sensitivities_match_einsum(mesh, N):
    from eigd_b200 import device as D
    prob, K0, M0 = mesh
    rng = np.random.default_rng(N)
    rhoE = rng.uniform(0.2, 1.0, prob.nelems)
    prob.set_density(rhoE=rhoE)
    WA, WB, V = (rng.normal(size=(prob.ndof, N)) for _ in range(3))
    cA, cB = 0.7, -1.3
    var = prob.var
    qK = np.einsum("eak,eab,ebk->e", WA[var], K0, V[var])
    qM = np.einsum("eak,eab,ebk->e", WB[var], M0, V[var])
    _, _, dk, dm = _law(rhoE)
    ref = cA * dk * qK + cB * dm * qM
    out = prob.device_call_fused(D.to_device(WA), D.to_device(WB), D.to_device(V), cA, cB).cpu().numpy()
    assert rel(out, ref) < 1e-12
    assert rel(prob.dAdx(WA, V), dk * qK) < 1e-12
    assert rel(prob.dBdx(WB, V), dm * qM) < 1e-12


def test_tangent_assembly(mesh):
    import h8_thermal_oracle as hto
    from eigd_b200 import device as D
    prob, K0, M0 = mesh
    rng = np.random.default_rng(5)
    rho, rho_t = rng.uniform(0.3, 1.0, prob.nnodes), rng.normal(size=prob.nnodes)
    prob.set_density(rho=D.to_device(rho))
    Kt, Mt = prob.assemble_tangent(D.to_device(rho_t))
    rhoE, rhoEt = rho[prob.conn].mean(axis=1), rho_t[prob.conn].mean(axis=1)
    _, _, dk, dm = _law(rhoE)
    Ko, Mo = hto.assemble(prob.conn, K0, M0, dk * rhoEt, dm * rhoEt, prob.ndof)
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


def _model(nx, ny, nz, N, solver_type="IRAM", **kw):
    from eigd_b200 import topo as T
    return T.make_thermal_3d_model(nx, ny, nz, rfact=1.5, N=N, solver_type=solver_type, seed=0, rtol=1e-12, tol=1e-14,
                                   adjoint_options={"lanczos_guess": True}, **kw)


def test_insulated_box_eigenpairs_match_dense():
    from scipy.linalg import eigh
    from eigd_b200 import device as D
    D.init()
    N = 8
    model = _model(6, 5, 4, N=N)
    assert model.nvars == 210
    model.initialize(x=np.random.default_rng(6).uniform(0.4, 1.0, model.nnodes))
    K, M = model.K.to_scipy().toarray(), model.M.to_scipy().toarray()
    lam_ref = eigh(K, M, eigvals_only=True)
    lam = np.asarray(model.lam)
    assert abs(lam_ref[0]) < 1e-10 * lam_ref[1] and lam_ref[1] > 1e-3 * lam_ref[N]      # one zero eigenvalue
    assert abs(lam[0]) < 1e-10 * lam_ref[1]
    assert rel(lam[1:], lam_ref[1:N]) < 1e-10
    Phi = model.Q.cpu().numpy()
    assert np.abs(Phi.T @ M @ Phi - np.eye(N)).max() < 1e-10


def _objective(model, vec):
    return model.get_thermal_compliance(vec) + np.sum(np.asarray(model.lam)[1:])


def _gradient_checks(ftype, fd_only=False):
    from eigd_b200 import device as D
    D.init()
    N = 5
    model = _model(5, 4, 3, N=N, ftype=ftype)
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
        fs.append(_objective(model, vec_d))
    fd = (fs[0] - fs[1]) / (2 * h)
    assert abs(g - fd) <= 1e-6 * abs(fd), (g, fd)
    if fd_only:
        return
    dual = _model(5, 4, 3, N=N, ftype=ftype, solver_type="BasicLanczos")
    dual.initialize(x=x0 + 1j * p)
    # value + i tangent: the first-order derivative of the objective, written out (complex arithmetic is not dual)
    lam_c, Q_c = np.asarray(dual.lam), np.asarray(dual.Q)
    c_r, c_t = Q_c.real.T @ vec, Q_c.imag.T @ vec
    l_r, l_t = lam_c.real[1:], lam_c.imag[1:]
    d_dual = float(np.sum((2.0 * c_r[1:] * c_t[1:] * l_r - c_r[1:] ** 2 * l_t) / l_r ** 2) + np.sum(l_t))
    assert abs(g - d_dual) <= 1e-8 * abs(d_dual), (g, d_dual)


def test_gradient_matches_central_difference_and_dual_numbers():
    _gradient_checks("spatial")


def test_helmholtz_driver_gradient_matches_central_difference():
    _gradient_checks("helmholtz", fd_only=True)


def _mirror_dvmap(nx, ny, nz):
    """Mirror symmetry in x, and the nodes of the end faces x = 0 and x = Lx not designed (dvmap -1, the filter takes
    x = 1 there)."""
    i = np.arange(nx + 1)[:, None, None] + np.zeros((1, ny + 1, nz + 1), dtype=np.int64)
    j = np.arange(ny + 1)[None, :, None] + np.zeros_like(i)
    k = np.arange(nz + 1)[None, None, :] + np.zeros_like(i)
    half = np.minimum(i, nx - i)
    dv = ((half - 1) * (ny + 1) + j) * (nz + 1) + k
    dv[half == 0] = -1
    return dv.ravel(), int(dv.max()) + 1


@pytest.mark.parametrize("dvmap,projection", [(False, False), (True, False), (False, True), (True, True)])
def test_helmholtz_filter_3d(dvmap, projection):
    import scipy.sparse.linalg as spla
    import h8_oracle as ho
    import h8_thermal_oracle as hto
    from eigd_b200 import device as D, fe
    D.init()
    nx, ny, nz = 6, 4, 3
    conn, _ = fe.hex_mesh(nx, ny, nz)
    X = ho.perturbed_box(nx, ny, nz, (1.2, 0.8, 0.6), amp=0.2, seed=12)
    r0 = 0.35
    kw = dict(projection=projection, beta=8.0, eta=0.45)
    if dvmap:
        dv, ndv = _mirror_dvmap(nx, ny, nz)
        kw.update(dvmap=dv, num_design_vars=ndv)
    flt = fe.NodeFilter(conn, X, r0=r0, ftype="helmholtz", **kw)
    # reference: A = r0^2 K + M, B = M of the unit-material scalar element, x expanded through the map
    K0, M0 = hto.all_element_matrices(conn, X)
    ones = np.ones(len(conn))
    Ko, Mo = hto.assemble(conn, K0, M0, ones, ones, X.shape[0])
    A = (r0 ** 2 * Ko + Mo).tocsc()
    rng = np.random.default_rng(13)
    x = rng.uniform(0.1, 1.0, flt.num_design_vars)
    xn = x if not dvmap else np.where(dv >= 0, x[np.maximum(dv, 0)], 1.0)
    rho_ref = spla.spsolve(A, Mo @ xn)
    if projection:
        t = np.tanh
        rho_ref = (t(8.0 * 0.45) + t(8.0 * (rho_ref - 0.45))) / (t(8.0 * 0.45) + t(8.0 * 0.55))
    assert rel(flt.apply(x), rho_ref) < 1e-12
    # the gradient is the exact transpose of the (linearised) filter
    xt, g = rng.normal(size=x.shape), rng.normal(size=X.shape[0])
    Fxt = flt.apply_tangent(D.to_device(x), D.to_device(xt)).cpu().numpy()
    FTg = flt.apply_gradient(g, x)
    assert abs(Fxt @ g - xt @ FTg) <= 1e-12 * np.abs(Fxt).max() * np.abs(g).sum()
    h = 1e-6
    fd = (flt.apply(x + h * xt) - flt.apply(x - h * xt)) / (2 * h)
    assert rel(Fxt, fd) < 1e-7
    # the filter's factor is pooled: it keeps no front workspace
    lu = flt._hA.lu
    assert lu.fronts == "pooled" and lu.pool_bytes() > 0
    resident = D.Factor(lu.sym, max_rhs=1, fronts="resident")
    assert resident.nbytes() - lu.nbytes() >= 8 * lu.sym.query("front_doubles")


def test_pooled_and_resident_fronts_are_bitwise_equal():
    from eigd_b200 import device as D
    D.init()
    N = 5
    rng = np.random.default_rng(14)
    out = []
    for fronts in ("resident", "pooled"):
        model = _model(7, 5, 4, N=N, fronts=fronts)
        if not out:
            x0 = rng.uniform(0.3, 1.0, model.nnodes)
            vec = D.to_device(rng.uniform(size=model.nnodes))
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model.initialize(x=x0)
        model.initialize_adjoint()
        model.add_thermal_compliance_derivative(1.0, vec)
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
        conn, X = fe.hex_mesh(7, 5, 4, 1.4, 1.0, 0.8)
        prob = fe.H8ThermalProblem(conn, X)
        rng = np.random.default_rng(10)
        prob.set_density(rhoE=rng.uniform(0.2, 1.0, prob.nelems))
        WA, WB, V = (D.to_device(rng.normal(size=(prob.ndof, 5))) for _ in range(3))
        ref = prob.device_call_fused(WA, WB, V, 1.0, -1.0)
        prob.sharding = ModeSharding()
        got = prob.device_call_fused(WA, WB, V, 1.0, -1.0)
        if rank == 0:
            out.put(float((got - ref).abs().max() / ref.abs().max()))
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
