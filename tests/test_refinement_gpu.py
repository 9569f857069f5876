"""Iterative refinement inside the factor's solve (eigd_factor_apply, csrc/solve.cu) on an indefinite shifted thermal Q4
pencil: SpLuOperator.solve_dev returns bitwise the X of the refinement loop written out with the plain solve, the SpMM,
axpby and col_axpy, in every operand layout the solvers use, with the same number of library launches.  A k above the
scratch registered with the native factor is an error; device.Factor grows its scratch instead."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from test_block_lanczos_gpu import q4_thermal  # noqa: E402

SIGMA = 60.0                                      # between 5 pi^2 and 8 pi^2: LDL^T with negative pivots


@pytest.fixture(scope="module")
def D():
    from eigd_b200 import device
    device.init()
    return device


@pytest.fixture(scope="module", params=[1, 2], ids=["depth1", "depth2"])
def op(request, D):
    import eigd_b200 as E
    K, M = q4_thermal(73, 61)
    f = E.SpLuOperator((K - SIGMA * M).tocsc(), refine=request.param)
    assert f.info["negative_pivots"] > 0 and f.refine == request.param
    return f


def loop_solve(D, op, Bd, out=None):
    """x = F b, then op.refine times x += F(b - mat x), one library call per step."""
    k = 1 if Bd.dim() == 1 else Bd.shape[1]
    if out is not None and out.data_ptr() == Bd.data_ptr():
        Bd = Bd.clone()
    X = op.lu.solve(Bd, out=out)
    for _ in range(op.refine):
        R = op.mat.spmm(X)
        Bc = Bd if Bd.is_contiguous() else Bd.contiguous()
        D.axpby(1.0, Bc.reshape(-1), -1.0, R.reshape(-1), out=R.reshape(-1))
        dX = op.lu.solve(R)
        if X.is_contiguous():
            D.axpby(1.0, X.reshape(-1), 1.0, dX.reshape(-1), out=X.reshape(-1))
        else:
            D.col_axpy(X, D.to_device(np.ones(k)), dX, sign=1.0)
    return X


def rhs(n, k, seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return torch.rand(n, k, dtype=torch.float64, device="cuda", generator=g) - 0.5


def launches(D, fn):
    torch.cuda.synchronize()
    l0 = D.launch_count()
    out = fn()
    torch.cuda.synchronize()
    return out, D.launch_count() - l0


@pytest.mark.parametrize("k", [1, 2, 3, 10, 20, 33])
def test_contiguous(D, op, k):
    n = op.shape[0]
    B = rhs(n, k, k)
    X, l_new = launches(D, lambda: op.solve_dev(B))
    R, l_ref = launches(D, lambda: loop_solve(D, op, B))
    assert torch.equal(X, R)
    assert l_new == l_ref
    if k == 1:                                    # a 1-D right-hand side: the same one-column products
        assert torch.equal(op.solve_dev(B[:, 0]), loop_solve(D, op, B[:, 0]))


@pytest.mark.parametrize("P", [1, 2, 3])
def test_vector_major_output(D, op, P):
    n = op.shape[0]
    B = rhs(n, P, 100 + P)
    Vt, Rt = D.zeros(P + 2, n), D.zeros(P + 2, n)
    op.solve_dev(B, out=Vt[:P].T)                 # the start block of the block Lanczos
    loop_solve(D, op, B, out=Rt[:P].T)
    assert torch.equal(Vt, Rt)


@pytest.mark.parametrize("k", [1, 3, 20])
def test_column_slice_input(D, op, k):
    n = op.shape[0]
    Bw = rhs(n, 40, 200 + k)
    B = Bw[:, 5:5 + k]
    assert torch.equal(op.solve_dev(B), loop_solve(D, op, B))


@pytest.mark.parametrize("k", [1, 2, 10, 33])
def test_out_aliases_b(D, op, k):
    n = op.shape[0]
    B = rhs(n, k, 300 + k)
    B1, B2 = B.clone(), B.clone()
    op.solve_dev(B1, out=B1)
    loop_solve(D, op, B2, out=B2)
    assert torch.equal(B1, B2)
    Bt1, Bt2 = B.T.contiguous(), B.T.contiguous()  # vector-major, in place
    op.solve_dev(Bt1.T, out=Bt1.T)
    loop_solve(D, op, Bt2.T, out=Bt2.T)
    assert torch.equal(Bt1, Bt2)


def test_scratch_bound(D, op):
    from eigd_b200 import _lib
    n = op.shape[0]
    cols = op.lu._refine_work.numel() // (2 * n)
    k = cols + 1
    B = rhs(n, k, 400)
    X = torch.empty_like(B)
    lib = _lib.load()
    rc = lib.eigd_factor_apply(op.lu.handle, ctypes.c_void_p(B.data_ptr()), k, 1, ctypes.c_void_p(X.data_ptr()), k, 1, k)
    assert rc != 0 and b"scratch" in lib.eigd_last_error()
    assert torch.equal(op.solve_dev(B), loop_solve(D, op, B))      # device.Factor grows the scratch
    assert op.lu._refine_work.numel() == 2 * n * k
