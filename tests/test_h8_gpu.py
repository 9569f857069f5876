"""The 3-D H8 solid on the device against tests/h8_oracle.py and dense references:

  * unit element matrices of a perturbed mesh (1e-13), assembled K and M against scipy's COO assembly of the oracle's
    matrices, the fused sensitivity kernel against the oracle's einsum, the tangent assembly against its definition and
    a central difference;
  * eigenpairs of a small free box against scipy.linalg.eigh (six rigid modes dropped, flexible lambda to 1e-10);
  * the design gradient of sum omega_i + sum (phi_i . w_i)^2 against a central difference and the dual-number
    (complex-step) directional derivative of BasicLanczos;
  * LDL^T factor and solve of K - sigma M on the smallest H8 cube whose widest front exceeds 4096 rows;
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
P, RHO0 = 3.0, 1e-6


def rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(b).max(), 1e-300)


@pytest.fixture(scope="module")
def mesh():
    import h8_oracle as ho
    from eigd_b200 import device as D, fe
    D.init()
    nx, ny, nz = 5, 4, 3
    conn, _ = fe.hex_mesh(nx, ny, nz)
    X = ho.perturbed_box(nx, ny, nz, (1.5, 1.0, 0.8), amp=0.25, seed=3)
    E, nu, density = 2.0, 0.28, 1.7
    prob = fe.H8Problem(conn, X, E=E, nu=nu, density=density, p=P, rho0_K=RHO0)
    K0, M0 = ho.all_element_matrices(conn, X, E, nu, density)
    return prob, K0, M0


def test_element_matrices_match_oracle(mesh):
    prob, K0, M0 = mesh
    Kd = prob.K0_d.cpu().numpy().reshape(K0.shape)
    Md = prob.M0_d.cpu().numpy().reshape(M0.shape)
    assert rel(Kd, K0) < 1e-13
    assert rel(Md, M0) < 1e-13


def test_assembly_matches_scipy_coo(mesh):
    import h8_oracle as ho
    prob, K0, M0 = mesh
    rhoE = np.random.default_rng(4).uniform(0.2, 1.0, prob.nelems)
    prob.set_density(rhoE=rhoE)
    K, M = prob.assemble()
    Ko, Mo = ho.assemble(prob.conn, K0, M0, rhoE**P + RHO0, rhoE, prob.ndof)
    Kd, Md = K.to_scipy(), M.to_scipy()
    for A, B in ((Kd, Ko), (Md, Mo)):
        B.sort_indices()
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
    dk, dm = P * rhoE ** (P - 1.0), np.ones(prob.nelems)
    ref = cA * dk * qK + cB * dm * qM
    out = prob.device_call_fused(D.to_device(WA), D.to_device(WB), D.to_device(V), cA, cB).cpu().numpy()
    assert rel(out, ref) < 1e-12
    assert rel(prob.dAdx(WA, V), dk * qK) < 1e-12
    assert rel(prob.dBdx(WB, V), dm * qM) < 1e-12


def test_tangent_assembly(mesh):
    import h8_oracle as ho
    from eigd_b200 import device as D
    prob, K0, M0 = mesh
    rng = np.random.default_rng(5)
    rho, rho_t = rng.uniform(0.3, 1.0, prob.nnodes), rng.normal(size=prob.nnodes)
    prob.set_density(rho=D.to_device(rho))
    Kt, Mt = prob.assemble_tangent(D.to_device(rho_t))
    rhoE, rhoEt = rho[prob.conn].mean(axis=1), rho_t[prob.conn].mean(axis=1)
    Ko, Mo = ho.assemble(prob.conn, K0, M0, P * rhoE ** (P - 1.0) * rhoEt, rhoEt, prob.ndof)
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


def _model(nx, ny, nz, L, N, solver_type="IRAM", **kw):
    from eigd_b200 import topo as T
    return T.make_natural_frequency_3d_model(nx, ny, nz, *L, rfact=1.5, N=N, solver_type=solver_type, seed=0, rtol=1e-12,
                                             adjoint_options={"lanczos_guess": True}, **kw)


def test_free_box_eigenpairs_match_dense():
    from scipy.linalg import eigh
    from eigd_b200 import device as D
    D.init()
    model = _model(6, 3, 3, (2.0, 1.0, 1.0), N=8, tol=1e-14)
    assert model.nvars == 336 and model.nrigid == 6
    model.initialize(x=np.random.default_rng(6).uniform(0.4, 1.0, model.nnodes))
    K, M = model.K.to_scipy().toarray(), model.M.to_scipy().toarray()
    lam_ref = eigh(K, M, eigvals_only=True)
    lam0 = np.asarray(model.lam0)
    assert np.all(np.abs(lam0[:6]) < 1e-8 * lam_ref[6])
    assert rel(model.lam, lam_ref[6:6 + 8]) < 1e-10
    Phi = model.Q0.cpu().numpy()
    assert np.abs(Phi.T @ M @ Phi - np.eye(Phi.shape[1])).max() < 1e-10


def _objective(model, w_d):
    from eigd_b200 import device as D
    c = D.col_dot(model.Q, w_d).cpu().numpy()
    return float(np.sum(model.get_frequencies()) + np.sum(c**2))


def test_gradient_matches_central_difference_and_dual_numbers():
    from eigd_b200 import device as D
    D.init()
    N = 4
    model = _model(5, 3, 2, (2.0, 1.1, 0.7), N=N, tol=1e-14)
    rng = np.random.default_rng(7)
    x0 = rng.uniform(0.4, 1.0, model.nnodes)
    p = rng.uniform(-1.0, 1.0, model.nnodes)
    w = rng.normal(size=(model.nvars, N))
    w_d = D.to_device(w)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.initialize(x=x0)
    lam = np.asarray(model.lam)
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
        fs.append(_objective(model, w_d))
    fd = (fs[0] - fs[1]) / (2 * h)
    assert abs(g - fd) <= 1e-6 * abs(fd), (g, fd)
    dual = _model(5, 3, 2, (2.0, 1.1, 0.7), N=N, solver_type="BasicLanczos", tol=1e-14)
    dual.initialize(x=x0 + 1j * p)
    lam_c, Q_c = np.asarray(dual.lam), np.asarray(dual.Q)
    c_r, c_t = np.einsum("ij,ij->j", Q_c.real, w), np.einsum("ij,ij->j", Q_c.imag, w)
    d_dual = float(np.sum(0.5 * lam_c.imag / np.sqrt(lam_c.real)) + np.sum(2.0 * c_r * c_t))
    assert abs(g - d_dual) <= 1e-8 * abs(d_dual), (g, d_dual)


def test_factor_and_solve_beyond_4096_row_fronts():
    """30^3 hexahedra (89 373 DOF) is the smallest H8 cube whose widest front exceeds 4096 rows (29^3: 4050)."""
    from eigd_b200 import device as D, fe
    from eigd_b200.eigenvector_derivatives import SpLuOperator
    D.init()
    conn, X = fe.hex_mesh(30, 30, 30)
    prob = fe.H8Problem(conn, X)
    prob.set_density(rhoE=np.random.default_rng(8).uniform(0.3, 1.0, prob.nelems))
    K, M = prob.assemble()
    sigma = -10.0
    A = K.with_values(D.axpby(1.0, K.data, -sigma, M.data))
    sym = D.Symbolic(prob.indptr, prob.indices, prob.ndof, coords=X, dof_per_node=3)
    assert sym.stats()["max_front"] > 4096
    f = SpLuOperator(A, symbolic=(sym, sym.assembly_map_device(A.indptr, A.indices)))
    info = f.info
    assert info["negative_pivots"] == 0 and info["perturbed_pivots"] == 0 and info["non_finite"] == 0, info
    rng = np.random.default_rng(9)
    for k in (1, 2, 10):
        b = D.to_device(rng.normal(size=(prob.ndof, k)))
        x = f.solve_dev(b)
        r = A.spmm(x) - b
        assert float(r.norm() / b.norm()) <= 1e-10, k


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
        prob = fe.H8Problem(conn, X)
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
