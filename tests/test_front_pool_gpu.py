"""Pooled fronts against resident fronts on the device: the factor (pivot-block inverses, full inverses, solve panels,
D and D^-1), the pivot statistics and multi-column solves are bitwise equal, with static and restricted Bunch-Kaufman
pivoting, refined solves of an indefinite shift, and the drivers that build one or two factors per design.  A pool that
is too small and a factor used with the wrong numeric entry point are refused."""
import ctypes
import warnings

import numpy as np
import pytest

import factor_cases as fc

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def _align(b):
    return (b + 255) // 256 * 256


def factor_arrays(fac):
    """The bytes of linv, xinv, xtmp, sfwd, sbwd, dval and dinv: one contiguous span of the factor's workspace, after the
    fronts (resident) or at its start (pooled)."""
    sym = fac.sym
    a = sym.arrays()
    nc = np.diff(a["sn_first"])
    f = nc + np.diff(a["sn_rowptr"])
    linv = int(np.sum((nc + 31) // 32) * 32 * 32)
    xinv = int(np.sum(nc * nc))
    panel = int(np.sum((f * nc + 1) & ~1))
    span = _align(linv * 8) + 2 * _align(xinv * 8) + 2 * _align(panel * 8 + 16) + 2 * _align(sym.n * 8)
    start = 0 if fac.fronts == "pooled" else _align(sym.query("front_doubles") * 8)
    assert fac._workspace.data_ptr() % 256 == 0
    return fac._workspace[start:start + span]


def factor_pair(sym, d_vals, d_map, pivoting="static", max_rhs=16):
    from eigd_b200 import device as D
    out = []
    for fronts in ("resident", "pooled"):
        fac = D.Factor(sym, max_rhs=max_rhs, pivoting=pivoting, fronts=fronts)
        fac._workspace.zero_()          # the few words no kernel writes (panel padding) read the same in both
        out.append(fac.numeric(d_vals, d_map))
    return out


def assert_same_factor(res, poo, n, rng, ks=(1, 3, 16)):
    from eigd_b200 import device as D
    assert poo.nbytes() < res.nbytes()
    assert torch.equal(factor_arrays(res), factor_arrays(poo))
    assert res.info() == poo.info()
    for k in ks:
        B = D.to_device(rng.normal(size=(n, k)))
        assert torch.equal(res.solve(B), poo.solve(B)), k


def case_of(kind, args):
    return {"grid": fc.grid_case, "dense": fc.dense_case, "bordered": fc.bordered_case, "kron": fc.kron_case}[kind](*args)


CASES = [("grid", fc.FRONT_MODE[0], "static"), ("grid", fc.WIDE_6DOF, "static"), ("dense", (300, "spd"), "static"),
         ("dense", (257, "saddle"), "bunch-kaufman"), ("bordered", (fc.BORDERED[4][0], fc.BORDERED[4][1], "shifted"),
                                                       "bunch-kaufman"),
         ("bordered", (fc.BORDERED[1][0], fc.BORDERED[1][1], "shifted"), "static"), ("kron", fc.KRON[1], "static"),
         ("kron", fc.KRON[3], "bunch-kaufman")]


@pytest.mark.parametrize("kind,args,pivoting", CASES, ids=["%s-%d-%s" % (c[0], i, c[2]) for i, c in enumerate(CASES)])
def test_pooled_factor_is_bitwise_resident(kind, args, pivoting):
    from eigd_b200 import device as D
    D.init()
    case = case_of(kind, args)
    A = case.A
    sym = D.Symbolic(A.indptr, A.indices, A.shape[0], coords=case.coords, dof_per_node=case.dof, opts=case.opts)
    Ad = D.CsrDevice.from_scipy(A)
    dmap = sym.assembly_map_device(Ad.indptr, Ad.indices)
    res, poo = factor_pair(sym, Ad.data, dmap, pivoting)
    assert_same_factor(res, poo, A.shape[0], np.random.default_rng(5))
    # a second factorisation with other values on the same factor and the same (cached) entry lists
    vals2 = Ad.data * 2.0
    res.numeric(vals2, dmap)
    poo.numeric(vals2, dmap)
    assert_same_factor(res, poo, A.shape[0], np.random.default_rng(6), ks=(2,))


def test_pooled_factor_of_30_cube_is_bitwise_resident():
    """30^3 hexahedra: fronts of more than 4096 rows; the pool is a sixth of the resident fronts."""
    from eigd_b200 import device as D, fe
    D.init()
    conn, X = fe.hex_mesh(30, 30, 30)
    prob = fe.H8Problem(conn, X)
    prob.set_density(rhoE=np.random.default_rng(8).uniform(0.3, 1.0, prob.nelems))
    K, M = prob.assemble()
    A = K.with_values(D.axpby(1.0, K.data, 10.0, M.data))
    sym = D.Symbolic(prob.indptr, prob.indices, prob.ndof, coords=X, dof_per_node=3)
    assert sym.stats()["max_front"] > 4096
    dmap = sym.assembly_map_device(A.indptr, A.indices)
    res, poo = factor_pair(sym, A.data, dmap)
    assert_same_factor(res, poo, prob.ndof, np.random.default_rng(9), ks=(1, 10))


def test_refined_solves_of_an_indefinite_shift():
    from eigd_b200 import device as D
    from eigd_b200.eigenvector_derivatives import SpLuOperator
    D.init()
    case = fc.kron_case(*fc.KRON[1])
    ops = [SpLuOperator(case.A, coords=case.coords, dof_per_node=case.dof, fronts=fr) for fr in ("resident", "pooled")]
    assert ops[0].info == ops[1].info and ops[0].info["negative_pivots"] == case.nneg
    assert ops[0].refine == ops[1].refine
    b = np.random.default_rng(3).normal(size=(case.n, 4))
    x0, x1 = ops[0].solve(b), ops[1].solve(b)
    assert np.array_equal(x0, x1)
    r = np.abs(case.A @ x0 - b).max() / np.abs(b).max()
    assert r < 1e-10, r


def test_too_small_pool_and_wrong_entry_point_are_refused():
    from eigd_b200 import _lib, device as D
    D.init()
    case = fc.grid_case(*fc.FRONT_MODE[0])
    A = case.A
    sym = D.Symbolic(A.indptr, A.indices, A.shape[0], coords=case.coords, dof_per_node=case.dof, opts=case.opts)
    Ad = D.CsrDevice.from_scipy(A)
    dmap = sym.assembly_map_device(Ad.indptr, Ad.indices)
    poo = D.Factor(sym, fronts="pooled")
    res = D.Factor(sym, fronts="resident")
    seg, ent = sym.pool_scatter(dmap)
    need = 8 * sym.query("pool_doubles")
    pool = torch.empty(need, dtype=torch.uint8, device=D.dev())
    lib = _lib.load()
    p = ctypes.c_void_p
    rc = lib.eigd_factor_numeric_pool(poo.handle, Ad.nnz, p(Ad.data.data_ptr()), p(seg.data_ptr()), p(ent.data_ptr()),
                                      p(pool.data_ptr()), need - 8)
    assert rc == 3 and b"front pool" in lib.eigd_last_error()
    rc = lib.eigd_factor_numeric(poo.handle, Ad.nnz, p(Ad.data.data_ptr()), p(dmap.data_ptr()))
    assert rc != 0 and b"pooled" in lib.eigd_last_error()
    rc = lib.eigd_factor_numeric_pool(res.handle, Ad.nnz, p(Ad.data.data_ptr()), p(seg.data_ptr()), p(ent.data_ptr()),
                                      p(pool.data_ptr()), need)
    assert rc != 0 and b"resident" in lib.eigd_last_error()
    assert lib.eigd_factor_workspace_bytes_fronts(sym.handle, 16, 2) == -1
    # the full-size pool works
    rc = lib.eigd_factor_numeric_pool(poo.handle, Ad.nnz, p(Ad.data.data_ptr()), p(seg.data_ptr()), p(ent.data_ptr()),
                                      p(pool.data_ptr()), need)
    assert rc == 0
    res.numeric(Ad.data, dmap)
    B = D.to_device(np.random.default_rng(1).normal(size=(A.shape[0], 2)))
    assert torch.equal(res.solve(B), poo.solve(B))


def _quiet(fn, *a, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return fn(*a, **kw)


def test_natural_frequency_3d_gradient_is_bitwise_resident():
    from eigd_b200 import device as D, topo as T
    D.init()
    out = []
    for fronts in ("resident", "pooled"):
        model = T.make_natural_frequency_3d_model(6, 4, 4, 2.0, 1.0, 1.0, rfact=1.5, N=4, seed=0, rtol=1e-12,
                                                  adjoint_options={"lanczos_guess": True}, fronts=fronts)
        assert model.fronts == fronts
        rng = np.random.default_rng(7)
        x0 = rng.uniform(0.4, 1.0, model.nnodes)
        w_d = D.to_device(rng.normal(size=(model.nvars, 4)))
        _quiet(model.initialize, x=x0)
        assert model.factor.lu.fronts == fronts
        model.initialize_adjoint()
        model.add_modal_function_derivative(w_d)
        model.finalize_adjoint()
        out.append((np.asarray(model.lam), model.xb.cpu().numpy()))
    assert np.array_equal(out[0][0], out[1][0])
    assert np.array_equal(out[0][1], out[1][1])


@pytest.mark.parametrize("pivoting", ["static", "bunch-kaufman"])
def test_buckling_3d_factors_share_the_pool(pivoting):
    """K_r and K_r + sigma G_r of one design are both pooled: neither keeps fronts, both factor on a pool borrowed
    in turn, and the load factors and the gradient are those of resident fronts bit for bit."""
    from eigd_b200 import device as D, topo as T
    D.init()
    out = []
    for fronts in ("resident", "pooled"):
        model = T.make_buckling_3d_model(4, 3, 16, 1.0, 0.75, 4.0, rfact=1.5, N=6, m=40, seed=0, rtol=1e-12,
                                         adjoint_options={"lanczos_guess": True}, pivoting=pivoting, fronts=fronts)
        x0 = np.random.default_rng(8).uniform(0.3, 0.7, model.fltr.num_design_vars)
        _quiet(model.initialize, x=x0)
        assert model.Kfact.lu.fronts == fronts and model.factor.lu.fronts == fronts
        node = int(np.argmax(np.abs(model.prob.full_vector(model.Qr[:, 0].contiguous()).cpu().numpy())))
        model.initialize_adjoint()
        model.add_eigenvector_aggregate_derivative(1.0, 100.0, node, mode="tanh")
        model.finalize_adjoint()
        out.append((np.asarray(model.BLF), model.xb.cpu().numpy(), model.factor.info,
                    model.Kfact.lu.nbytes() + model.factor.lu.nbytes()))
    assert np.array_equal(out[0][0], out[1][0])
    assert np.array_equal(out[0][1], out[1][1])
    assert out[0][2] == out[1][2]
    sym = model.symbolic[0]
    assert out[0][3] - out[1][3] == 2 * _align(8 * sym.query("front_doubles"))
