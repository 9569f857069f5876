"""Parity of every CUDA kernel (through the C-ABI) against numpy / scipy on the same inputs."""
import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def D():
    from eigd_b200 import device
    device.init()
    return device


def rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def grid_matrix(nx, ny, dof, rng, spd=True):
    import fe_oracle as fo
    conn, X = fo.grid_mesh(nx, ny, 1.0, ny / nx)
    var = fo.element_dofs(conn, dof)
    i, j = fo.coo_index(var)
    v = rng.uniform(-1, 1, len(i))
    A = sp.coo_matrix((v, (i, j))).tocsr()
    A = (A + A.T) * 0.5
    if spd:
        A = A + sp.diags(np.abs(A).sum(axis=1).A1 + 0.1)
    A = A.tocsr()
    A.sort_indices()
    return A, X


@pytest.mark.parametrize("k", [1, 2, 3, 7, 10, 20, 33])
def test_spmm(D, k):
    rng = np.random.default_rng(k)
    A, _ = grid_matrix(37, 23, 2, rng)
    n = A.shape[0]
    Ad = D.CsrDevice.from_scipy(A)
    X = rng.normal(size=(n, k))
    Y0 = rng.normal(size=(n, k))
    Y = Ad.spmm(D.to_device(X), out=D.to_device(Y0.copy()), alpha=0.7, beta=-0.3).cpu().numpy()
    assert rel(Y, 0.7 * (A @ X) - 0.3 * Y0) < 1e-14
    # vector-major operands (Krylov basis layout)
    Xt = D.to_device(np.ascontiguousarray(X.T))
    Yt = D.empty(k, n)
    Ad.spmm(Xt.T, out=Yt.T)
    assert rel(Yt.cpu().numpy().T, A @ X) < 1e-14


@pytest.mark.parametrize("k1,k2", [(1, 1), (3, 5), (10, 10), (23, 9), (60, 1), (61, 10), (40, 37)])
def test_gemm_tn_nn(D, k1, k2):
    rng = np.random.default_rng(k1 * 100 + k2)
    n = 10007
    X, Y = rng.normal(size=(n, k1)), rng.normal(size=(n, k2))
    C = D.gemm_tn(D.to_device(X), D.to_device(Y)).cpu().numpy()
    assert rel(C, X.T @ Y) < 1e-13
    # vector-major X
    Xt = D.to_device(np.ascontiguousarray(X.T))
    C2 = D.gemm_tn(Xt.T, D.to_device(Y)).cpu().numpy()
    assert rel(C2, X.T @ Y) < 1e-13
    S = rng.normal(size=(k1, k2))
    Y0 = rng.normal(size=(n, k2))
    Yd = D.to_device(Y0.copy())
    D.gemm_nn(D.to_device(X), D.to_device(S), Yd, alpha=-1.5, beta=0.5)
    assert rel(Yd.cpu().numpy(), 0.5 * Y0 - 1.5 * X @ S) < 1e-13
    Yd = D.zeros(n, k2)
    D.gemm_nn(Xt.T, D.to_device(S), Yd, alpha=1.0, beta=0.0)
    assert rel(Yd.cpu().numpy(), X @ S) < 1e-13


@pytest.mark.parametrize("k", [1, 5, 10, 23, 64, 70])
def test_column_ops(D, k):
    rng = np.random.default_rng(k)
    n = 5003
    X, Y = rng.normal(size=(n, k)), rng.normal(size=(n, k))
    s = rng.uniform(0.5, 2.0, k)
    Xd, Yd, sd = D.to_device(X), D.to_device(Y), D.to_device(s)
    assert rel(D.col_dot(Xd, Yd).cpu().numpy(), np.einsum("ij,ij->j", X, Y)) < 1e-13
    D.col_axpy(Yd, sd, Xd, sign=-1.0)
    assert rel(Yd.cpu().numpy(), Y - s * X) < 1e-14
    D.col_scale(Xd, sd, mode=2)
    assert rel(Xd.cpu().numpy(), X / np.sqrt(s)) < 1e-14
    T = D.empty(k, n)
    D.copy2d(Xd, T.T)
    assert (T.cpu().numpy().T == Xd.cpu().numpy()).all()
    P = rng.normal(size=(n, 4))
    Q = rng.normal(size=(n, 4))
    Z = D.to_device(Y.copy())
    D.project(D.to_device(P), D.to_device(Q), Z)
    assert rel(Z.cpu().numpy(), Y - P @ (Q.T @ Y)) < 1e-12


CASES = [(12, 9, 1, True), (12, 9, 1, False), (40, 40, 1, True), (33, 21, 2, False), (90, 70, 1, True), (64, 48, 2, True)]


@pytest.mark.parametrize("nx,ny,dof,use_xy", CASES)
def test_factor_solve(D, nx, ny, dof, use_xy):
    import multifrontal_oracle as mo
    rng = np.random.default_rng(nx + ny)
    A, X = grid_matrix(nx, ny, dof, rng)
    n = A.shape[0]
    sym = D.Symbolic(A.indptr, A.indices, n, coords=X if use_xy else None, dof_per_node=dof)
    Ad = D.CsrDevice.from_scipy(A)
    amap_h = sym.assembly_map_host()
    amap_d = sym.assembly_map_device(Ad.indptr, Ad.indices)
    assert (amap_d.cpu().numpy() == amap_h).all()          # integer structure: bit-exact
    fac = D.Factor(sym, max_rhs=32).numeric(Ad.data, amap_d)
    info = fac.info()
    assert info["negative_pivots"] == 0 and info["perturbed_pivots"] == 0 and info["non_finite"] == 0
    for k in (1, 3, 10, 20, 32, 40):
        B = rng.normal(size=(n, k))
        Xs = fac.solve(D.to_device(B)).cpu().numpy()
        r = np.abs(A @ Xs - B).max() / np.abs(B).max()
        assert r < 1e-11, (k, r)
    # single vector, in place, vector-major layout
    b = rng.normal(size=n)
    bd = D.to_device(b.copy())
    fac.solve(bd, out=bd)
    assert np.abs(A @ bd.cpu().numpy() - b).max() < 1e-11
    if n < 3000:
        d = sym.arrays()
        d["amap"] = amap_h
        ref = mo.MultifrontalOracle(d).factor(A.data)
        xo = ref.solve(b)
        assert rel(bd.cpu().numpy(), xo) < 1e-10


@pytest.mark.parametrize("nx,ny,dof", [(250, 200, 1), (160, 120, 2)])
def test_factor_solve_front_mode(D, nx, ny, dof):
    """Sizes at which the solve plan has subtree phases: exercises the TMA-staged front kernels (k = 1 pipelined
    operands, k > 1 forward fronts + backward tile path) and the persistent level kernel between them."""
    import ctypes
    from eigd_b200 import _lib
    rng = np.random.default_rng(nx + ny + dof)
    A, X = grid_matrix(nx, ny, dof, rng)
    n = A.shape[0]
    sym = D.Symbolic(A.indptr, A.indices, n, coords=X, dof_per_node=dof)
    lib = _lib.load()
    meta = np.zeros(3, dtype=np.int64)
    lib.eigd_solve_plan_get(sym.handle, 148 * 16, 148, -2, 7, meta.ctypes.data_as(ctypes.c_void_p), 3)
    assert meta[0] >= 0, "expected subtree phases at this size"
    Ad = D.CsrDevice.from_scipy(A)
    fac = D.Factor(sym, max_rhs=32).numeric(Ad.data, sym.assembly_map_device(Ad.indptr, Ad.indices))
    for k in (1, 2, 5, 10, 16, 24):
        B = rng.normal(size=(n, k))
        Bd = D.to_device(B)
        X1 = fac.solve(Bd).cpu().numpy()
        r = np.abs(A @ X1 - B).max() / np.abs(B).max()
        assert r < 1e-11, (k, r)
        X2 = fac.solve(Bd).cpu().numpy()
        assert np.array_equal(X1, X2), "solve is not bitwise reproducible"
    b = rng.normal(size=n)
    bd = D.to_device(b.copy())
    fac.solve(bd, out=bd)                               # in place
    assert np.abs(A @ bd.cpu().numpy() - b).max() / np.abs(b).max() < 1e-11


def test_factor_indefinite(D):
    rng = np.random.default_rng(7)
    A, X = grid_matrix(50, 30, 1, rng, spd=True)
    # shift into the spectrum: a handful of negative eigenvalues, like K + sigma*G above BLF_0
    import scipy.sparse.linalg as spla
    lo = spla.eigsh(A, k=6, sigma=0.0, which="LM", return_eigenvectors=False)
    shift = 0.5 * (np.sort(lo)[3] + np.sort(lo)[4])
    As = (A - shift * sp.identity(A.shape[0])).tocsr()
    n = As.shape[0]
    sym = D.Symbolic(As.indptr, As.indices, n, coords=X)
    Ad = D.CsrDevice.from_scipy(As)
    fac = D.Factor(sym).numeric(Ad.data, sym.assembly_map_device(Ad.indptr, Ad.indices))
    info = fac.info()
    assert info["negative_pivots"] == 4      # Sylvester inertia = eigenvalues below the shift
    b = rng.normal(size=(n, 5))
    x = fac.solve(D.to_device(b)).cpu().numpy()
    assert np.abs(As @ x - b).max() / np.abs(b).max() < 1e-9


@pytest.mark.parametrize("kind,N", [("thermal", 1), ("thermal", 10), ("plane_stress", 9), ("plane_stress", 23)])
def test_q4_kernels(D, kind, N):
    import fe_oracle as fo
    rng = np.random.default_rng(N)
    conn, X = fo.grid_mesh(23, 17, 2.0, 1.3)
    X = X + 0.01 * rng.normal(size=X.shape)          # non-rectangular elements
    mdl = fo.Q4Model(conn, X, kind)
    rhoE = rng.uniform(0.2, 1.0, mdl.nelems)
    WA, WB, V = (rng.normal(size=(mdl.ndof, N)) for _ in range(3))
    ref = 1.3 * mdl.dK(rhoE, WA, V) - 0.7 * mdl.dM(rhoE, WB, V)
    kid = 0 if kind == "thermal" else 1
    conn_d = torch.as_tensor(conn.astype(np.int32), device=D.dev())
    xy_d = D.to_device(X)
    c6 = D.to_device(mdl.cmat6)
    out = D.zeros(mdl.nelems)
    D.q4_quadforms(kid, conn_d, xy_d, c6, D.to_device(WA), D.to_device(WB), D.to_device(V),
                   D.to_device(mdl.k_scale_deriv(rhoE)), D.to_device(mdl.m_scale_deriv(rhoE)), 1.3, 0.7, out)
    assert rel(out.cpu().numpy(), ref) < 1e-12
    # assembly in gather form
    K, M = mdl.assemble(rhoE)
    sp_, src, _ = mdl.assembly_sources(K)
    Kv, Mv = D.empty(K.nnz), D.empty(K.nnz)
    D.q4_assemble(kid, conn_d, xy_d, D.to_device(mdl.k_scale(rhoE)), D.to_device(mdl.m_scale(rhoE)), c6,
                  torch.as_tensor(sp_, device=D.dev()), torch.as_tensor(src, device=D.dev()), K.nnz, Kv, Mv)
    assert rel(Kv.cpu().numpy(), K.data) < 1e-12 and rel(Mv.cpu().numpy(), M.data) < 1e-12
    # element -> node gather
    nptr, nelem = mdl.node_adjacency()
    ev = rng.normal(size=mdl.nelems)
    nd = D.empty(mdl.nnodes)
    D.node_gather(torch.as_tensor(nptr, device=D.dev()), torch.as_tensor(nelem, device=D.dev()), D.to_device(ev), 0.25, nd)
    assert rel(nd.cpu().numpy(), mdl.scatter_to_nodes(ev)) < 1e-13


def test_host_device_copies(D):
    """Copies behind the numpy API: pageable, read-only and page-locked sources, transposed / sliced device
    tensors, sizes either side of the pinned-path threshold -- all bit-exact round trips."""
    rng = np.random.default_rng(5)
    for shape in [(7,), (300, 10), (200_000, 3), (150_000, 10)]:
        a = rng.standard_normal(shape)
        t = D.h2d(a)
        assert t.is_cuda and tuple(t.shape) == shape
        assert np.array_equal(D.d2h(t), a)
        ro = a.copy()
        ro.setflags(write=False)
        assert np.array_equal(D.d2h(D.h2d(ro)), a)
        p = D.pinned_empty(shape)
        p[...] = a
        tp = D.h2d(p)
        p[...] = 0.0                                  # the upload must be complete when h2d returns
        assert np.array_equal(D.d2h(tp), a)
    big = D.h2d(rng.standard_normal((150_000, 10)))
    back = D.d2h(big.T)                               # dense, transposed: strides preserved like Tensor.cpu()
    assert back.shape == (10, 150_000) and np.array_equal(back, big.cpu().numpy().T)
    sl = D.d2h(big[:, 2:9])                           # non-dense view
    assert np.array_equal(sl, big.cpu().numpy()[:, 2:9])
    out = D.d2h(big)
    out[0, 0] = 123.0                                 # returned arrays are writable and independent of the device copy
    assert float(big[0, 0]) != 123.0
    idx = rng.integers(0, 1000, 600_000).astype(np.int32)
    assert np.array_equal(D.d2h(D.h2d(idx)), idx)


def test_pattern_cache_identity_and_change(D):
    """The CSR structure is uploaded once per pattern; the same arrays are accepted again, edited or different
    arrays are compared in full (a changed pattern must never be served from the cache)."""
    rng = np.random.default_rng(9)
    A, _ = grid_matrix(41, 29, 1, rng)
    c1 = D.CsrDevice.from_scipy(A)
    c2 = D.CsrDevice.from_scipy(A)                    # identical objects -> identity path
    assert c2.indices.data_ptr() == c1.indices.data_ptr()
    B = A.copy()                                      # new arrays, same pattern -> full comparison, same entry
    c3 = D.CsrDevice.from_scipy(B)
    assert c3.indices.data_ptr() == c1.indices.data_ptr()
    C = A.copy()
    r = C.shape[0] // 2
    lo, hi = C.indptr[r], C.indptr[r + 1]
    C.indices[lo:hi] = np.sort((C.indices[lo:hi] + 3) % C.shape[1])    # same sizes, different columns
    c4 = D.CsrDevice.from_scipy(C)
    assert np.array_equal(c4.indices.cpu().numpy(), C.indices)
    x = rng.standard_normal(C.shape[1])
    assert rel(c4.spmm(D.to_device(x)).cpu().numpy(), C @ x) < 1e-13


@pytest.mark.parametrize("n,k,j", [(5003, 1, 3), (5003, 10, 7), (40_000, 10, 12), (251_001, 10, 9), (3001, 20, 5),
                                   (777, 64, 2), (100_000, 3, 70), (50, 10, 4)])
def test_mgs_sweep(D, n, k, j):
    """One cooperative launch = the reference's dot / axpy loop over the stored blocks (sequential, modified GS)."""
    rng = np.random.default_rng(n + k + j)
    w = rng.normal(size=(n, k))
    Ws = [rng.normal(size=(n, k)) / np.sqrt(n) for _ in range(j)]
    ref, hs = w.copy(), []
    for W in Ws:
        h = np.einsum("ij,ij->j", ref, W)
        ref -= h * W
        hs.append(h)
    wd = D.to_device(w)
    H = D.zeros(j + 1, k)
    D.mgs_sweep(wd, [D.to_device(W) for W in Ws], [H[t] for t in range(j)])
    assert rel(wd.cpu().numpy(), ref) < 1e-13
    assert rel(H[:j].cpu().numpy(), np.array(hs)) < 1e-12
    assert float(H[j].abs().max()) == 0.0
    # bitwise reproducible
    wd2 = D.to_device(w)
    H2 = D.zeros(j + 1, k)
    D.mgs_sweep(wd2, [D.to_device(W) for W in Ws], [H2[t] for t in range(j)])
    assert torch.equal(wd, wd2) and torch.equal(H, H2)
    # non-contiguous operands take the dot / axpy path with the same result
    wt = D.to_device(np.ascontiguousarray(w.T)).T
    H3 = D.zeros(j, k)
    D.mgs_sweep(wt, [D.to_device(W) for W in Ws], [H3[t] for t in range(j)])
    assert rel(wt.cpu().numpy(), ref) < 1e-13


@pytest.mark.parametrize("k", [1, 2, 3])
def test_factor_solve_slices_beyond_the_ring(D, k):
    """400 disjoint dense 96 x 96 blocks: level-phase tiles whose panel slice (24 576 bytes) is larger than the
    shared-memory ring of the pipelined level kernel read it from global memory (k = 1, 2); k = 3 runs the 16-warp
    level kernel on the same tile-major panels.  test_solve_plan_cpu.py checks that the plan has such slices."""
    import factor_cases as fc
    c = fc.block_diagonal_case()
    A, n = c.A, c.n
    sym = D.Symbolic(A.indptr, A.indices, n, coords=c.coords, dof_per_node=c.dof, opts=c.opts)
    Ad = D.CsrDevice.from_scipy(A)
    fac = D.Factor(sym, max_rhs=32).numeric(Ad.data, sym.assembly_map_device(Ad.indptr, Ad.indices))
    B = np.random.default_rng(k).normal(size=(n, k))
    Bd = D.to_device(B)
    X1 = fac.solve(Bd).cpu().numpy()
    r = np.abs(A @ X1 - B).max() / np.abs(B).max()
    assert r < 1e-11, (k, r)
    X2 = fac.solve(Bd).cpu().numpy()
    assert np.array_equal(X1, X2), "solve is not bitwise reproducible"
