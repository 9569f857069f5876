"""The device supernodal LDL^T (factor.cu) and its triangular solves (solve.cu) against plain float64 references, on the
matrices of tests/factor_cases.py (whose shapes test_factor_shapes_cpu.py checks on the host):

  * one dense supernode of every width 1 .. 512 around the 32-column edges, SPD, indefinite and saddle-point, with the
    static and the Bunch-Kaufman factor: backward error of the unrefined solve, forward error against
    numpy.linalg.solve scaled by the condition number, exact inertia from eigvalsh, and (Bunch-Kaufman) the pivot
    decisions of tests/bunch_kaufman_oracle.py;
  * bordered block-diagonal matrices (child fronts with a controlled number of rows below), grid patterns with 1, 2, 3
    and 6 DOF per node under supernode caps 32 .. 512 with and without relaxation, the two front-mode sizes;
  * shifted Kronecker-sum Laplacians at 40 000 - 50 000 DOF whose inertia is known in closed form;
  * every right-hand-side count 1 .. 16 and wider ones, and max_rhs 1 .. 16, in a level-only and a front-mode plan:
    the k columns solved together agree with each column solved alone, repeated solves are bitwise identical;
  * operand layouts (row-major, column-major, column and row slices of wider buffers, mixed, in place): the solve
    writes exactly its n x k view -- every other bit of the surrounding buffer stays a NaN sentinel -- leaves B
    untouched, and gives bitwise the same X for every layout.

Residuals are accumulated in long double, so the check's own rounding stays out of the backward error
eta = |b - A x|_inf / (|A|_inf |x|_inf + |b|_inf)."""
import numpy as np
import pytest
import scipy.sparse.linalg as spla

import factor_cases as fc

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

ETA_SPD = 1e-14             # SPD matrices, static or pivoted factor
ETA_INDEFINITE = 1e-13      # indefinite matrices, Bunch-Kaufman factor (and static where its growth permits)


@pytest.fixture(scope="module")
def D():
    from eigd_b200 import device
    device.init()
    return device


def eta(A, x, b):
    """Normwise backward error of every column, residual in long double; -> max over columns."""
    Al = A.astype(np.longdouble)
    x = np.asarray(x).reshape(A.shape[0], -1)
    b = np.asarray(b).reshape(A.shape[0], -1)
    r = b.astype(np.longdouble) - Al @ x.astype(np.longdouble)
    anorm = float(abs(Al).sum(axis=1).max())
    return max(float(np.abs(r[:, j]).max()) / (anorm * np.abs(x[:, j]).max() + np.abs(b[:, j]).max())
               for j in range(x.shape[1]))


def symbolic(D, c):
    return D.Symbolic(c.A.indptr, c.A.indices, c.n, coords=c.coords, dof_per_node=c.dof, opts=c.opts)


def factor(D, c, sym, pivoting="static", max_rhs=32):
    Ad = D.CsrDevice.from_scipy(c.A)
    return D.Factor(sym, max_rhs=max_rhs, pivoting=pivoting).numeric(Ad.data, sym.assembly_map_device(Ad.indptr,
                                                                                                       Ad.indices))


def oracle(c, sym):
    from bunch_kaufman_oracle import BunchKaufmanOracle
    d = sym.arrays()
    d["amap"] = sym.assembly_map_host()
    return BunchKaufmanOracle(d)


def doubling_inverse(L):
    """Inverse of a unit lower triangular pivot block the way factor.cu forms it: 32 x 32 diagonal blocks, then
    recursive doubling, X21 = -B^-1 (C A^-1) for pairs of hb-wide blocks, hb = 32, 64, 128, 256."""
    n = L.shape[0]
    X = np.zeros_like(L)
    for k0 in range(0, n, 32):
        X[k0:k0 + 32, k0:k0 + 32] = np.linalg.inv(L[k0:k0 + 32, k0:k0 + 32])
    hb = 32
    while hb < n:
        for lo0 in range(0, n - hb, 2 * hb):
            hi0 = lo0 + hb
            hi1 = min(n, hi0 + hb)
            X[hi0:hi1, lo0:hi0] = -X[hi0:hi1, hi0:hi1] @ (L[hi0:hi1, lo0:hi0] @ X[lo0:hi0, lo0:hi0])
        hb *= 2
    return X


def inverse_based_eta(c, sym, pivoting, b):
    """The oracle's factor of c.A (same ordering, same pivots), solved the way the device solves: products with the
    explicit doubling inverses of the pivot blocks instead of substitution.  -> (oracle, backward error).  The
    explicit inverse loses accuracy with the condition number of the unit lower pivot block, which an indefinite
    matrix can make large (1e5 for a 255-wide Bunch-Kaufman block, 1e9 without pivoting)."""
    o = oracle(c, sym).factor(c.A.data, pivoting=pivoting)
    s = o.sym
    perm = s["perm"]
    y = b[perm].copy()
    inv = []
    for k in range(o.ns):
        Fk, nc, nb = o._front_view(o.F, k)
        L11 = o.L11[k] if o.L11 is not None else np.tril(Fk[:nc, :nc], -1) + np.eye(nc)
        inv.append(doubling_inverse(L11))
        c0 = s["sn_first"][k]
        y[c0:c0 + nc] = inv[k] @ y[c0:c0 + nc]
        y[s["sn_rows"][s["sn_rowptr"][k]:s["sn_rowptr"][k + 1]]] -= Fk[nc:, :nc] @ y[c0:c0 + nc]
    y *= o.dinv[:, None]
    for k in range(o.ns - 1, -1, -1):
        Fk, nc, nb = o._front_view(o.F, k)
        c0 = s["sn_first"][k]
        rows = s["sn_rows"][s["sn_rowptr"][k]:s["sn_rowptr"][k + 1]]
        y[c0:c0 + nc] = inv[k].T @ (y[c0:c0 + nc] - Fk[nc:, :nc].T @ y[rows])
    x = np.empty_like(y)
    x[perm] = y
    return o, eta(c.A, x, b)


def check_case(D, c, pivoting, dense_ref, seed=0):
    """Factor c.A on the device and check info(), the inertia and the unrefined solve of three right-hand sides.
    dense_ref: inertia from eigvalsh, forward error against numpy.linalg.solve (small cases); else the closed-form
    inertia c.nneg and, where the spectrum is known (Kronecker cases), the forward error against scipy's splu."""
    sym = symbolic(D, c)
    fac = factor(D, c, sym, pivoting)
    info = fac.info()
    rng = np.random.default_rng(seed + c.n)
    b = rng.normal(size=(c.n, 3))
    x = fac.solve(D.to_device(b)).cpu().numpy()
    assert info["non_finite"] == 0, info
    assert info["perturbed_pivots"] == 0, info
    if dense_ref:
        Ad = c.A.toarray()
        ev = np.linalg.eigvalsh(Ad)
        nneg = int((ev < 0).sum())
        if c.nneg is not None:
            assert nneg == c.nneg
        x_ref = np.linalg.solve(Ad, b)
        cond = np.abs(ev).max() / np.abs(ev).min()
    else:
        nneg = c.nneg
        cond = None
        if hasattr(c, "spectrum"):                   # Kronecker cases: the condition number is known too
            x_ref = spla.splu(c.A.tocsc()).solve(b)
            cond = np.abs(c.spectrum).max() / np.abs(c.spectrum).min()
    assert info["negative_pivots"] == nneg, (info, nneg)
    e = eta(c.A, x, b)
    if nneg == 0:
        bound = ETA_SPD
    else:
        # indefinite: the element growth of the static factor is not bounded, and the explicit inverses of the pivot
        # blocks lose accuracy with their condition: the device may not lose more than a factor 10 against the same
        # algorithm carried out in numpy, nor exceed ETA_INDEFINITE where that algorithm stays below it
        o, e_ref = inverse_based_eta(c, sym, pivoting, b)
        assert o.info == (nneg, 0)
        bound = max(ETA_INDEFINITE, 10.0 * e_ref)
    assert e <= bound, (c.name, pivoting, e, bound)
    if cond is not None:
        fwd = np.abs(x - x_ref).max() / np.abs(x_ref).max()
        assert fwd <= cond * bound, (c.name, fwd, cond)
    return sym, fac, info


DENSE_RUNS = [(w, kind, piv) for w in fc.DENSE_WIDTHS
              for kind, piv in [("spd", "static"), ("spd", "bunch-kaufman"), ("indefinite", "static"),
                                ("indefinite", "bunch-kaufman"), ("saddle", "bunch-kaufman")]
              if not (kind == "saddle" and w < 2)]


@pytest.mark.parametrize("w,kind,pivoting", DENSE_RUNS)
def test_dense_supernode(D, w, kind, pivoting):
    """One supernode of width w: the 32-column pivot blocks, the partial last block (a 2x2 pivot must not cross its
    edge), the 64 / 128 / 256 stages of the recursive-doubling inverse (hb = 256 only for w > 256)."""
    c = fc.dense_case(w, kind)
    sym, fac, info = check_case(D, c, pivoting, dense_ref=True)
    if pivoting == "bunch-kaufman":
        ref = oracle(c, sym).factor(c.A.data, pivoting="bunch-kaufman")
        # pivot decisions compare computed entries: only where none lies within rounding of its threshold
        if ref.margin > 1e-8:
            for key in ("negative_pivots", "two_by_two_pivots", "interchanges"):
                assert info[key] == ref.counts[key], (key, info[key], ref.counts[key])


@pytest.mark.parametrize("pivoting", ["static", "bunch-kaufman"])
@pytest.mark.parametrize("kind", ["spd", "shifted"])
@pytest.mark.parametrize("blocks,border", fc.BORDERED)
def test_bordered(D, blocks, border, kind, pivoting):
    check_case(D, fc.bordered_case(blocks, border, kind), pivoting, dense_ref=True)


@pytest.mark.parametrize("case", fc.GRID_CASES, ids=lambda g: "x".join(map(str, g)))
def test_grid(D, case):
    """Grid patterns with 1, 2, 3 and 6 DOF per node; 6 x 51 x 45 has a 420-column top separator (shell-like front
    sizes); 250 x 200 x 1 and 160 x 120 x 2 are solved in front mode."""
    c = fc.grid_case(*case)
    check_case(D, c, "static", dense_ref=False)
    if case == fc.WIDE_6DOF:
        check_case(D, c, "bunch-kaufman", dense_ref=False)


@pytest.mark.parametrize("pivoting", ["static", "bunch-kaufman"])
@pytest.mark.parametrize("nx,ny,dof,target", fc.KRON)
def test_kron_inertia(D, nx, ny, dof, target, pivoting):
    """Shifted Kronecker-sum Laplacian: the number of negative pivots is the closed-form count of eigenvalues below the
    shift (hundreds of them, spread over many supernodes and the subtree phases)."""
    c = fc.kron_case(nx, ny, dof, target)
    sym, fac, info = check_case(D, c, pivoting, dense_ref=False)
    if pivoting == "bunch-kaufman":
        ref = oracle(c, sym).factor(c.A.data, pivoting="bunch-kaufman")
        assert ref.margin > 1e-8
        for key in ("negative_pivots", "two_by_two_pivots", "interchanges"):
            assert info[key] == ref.counts[key], (key, info[key], ref.counts[key])


# ---- right-hand-side counts ----------------------------------------------------------------------------------------
RHS_K = list(range(1, 17)) + [17, 20, 24, 31, 32, 33, 40, 48]
KMAX = max(RHS_K)


@pytest.fixture(scope="module", params=fc.RHS_CASES, ids=["level-only", "front-mode"])
def rhs_case(request, D):
    """(case, symbolic, factor with max_rhs = 32, B (n x 48), X of every column solved alone)."""
    c = fc.grid_case(*request.param)
    sym = symbolic(D, c)
    fac = factor(D, c, sym)
    B = np.random.default_rng(c.n).normal(size=(c.n, KMAX))
    X1 = np.stack([fac.solve(D.to_device(B[:, j].copy())).cpu().numpy() for j in range(KMAX)], axis=1)
    assert eta(c.A, X1, B) <= ETA_SPD
    return c, sym, fac, B, X1


def agree_with_single_columns(X, X1):
    """Columns solved together against alone: relative to each column (another KT may sum in another order)."""
    d = np.abs(X - X1).max(axis=0) / np.abs(X1).max(axis=0)
    return float(d.max())


@pytest.mark.parametrize("k", RHS_K)
def test_rhs_count(D, rhs_case, k):
    """k -> balanced chunks of at most 16 columns, each on the template KT in {1, 2, 4, 6, 8, 10, 12, 16} with
    zero-padded lanes: every KT and every padded width, in both plan kinds."""
    c, sym, fac, B, X1 = rhs_case
    Bd = D.to_device(B[:, :k].copy())
    X = fac.solve(Bd).cpu().numpy()
    assert eta(c.A, X, B[:, :k]) <= ETA_SPD
    assert agree_with_single_columns(X, X1[:, :k]) <= 1e-14
    assert np.array_equal(X, fac.solve(Bd).cpu().numpy()), "solve is not bitwise reproducible"


@pytest.mark.parametrize("max_rhs", [1, 2, 4, 8, 16])
def test_max_rhs(D, rhs_case, max_rhs):
    """A factor created for fewer right-hand sides (the workspace slabs are sized by max_rhs) splits wider solves
    into chunks of at most max_rhs columns."""
    c, sym, _, B, X1 = rhs_case
    fac = factor(D, c, sym, max_rhs=max_rhs)
    for k in (1, 3, 5, 9, 17):
        X = fac.solve(D.to_device(B[:, :k].copy())).cpu().numpy()
        assert eta(c.A, X, B[:, :k]) <= ETA_SPD, (max_rhs, k)
        assert agree_with_single_columns(X, X1[:, :k]) <= 1e-14, (max_rhs, k)


# ---- operand layouts -----------------------------------------------------------------------------------------------
SENTINEL = 0x7FF8DEADBEEF0001      # a quiet NaN with a payload; compared bit for bit


def view_row(buf, n, k):           # (a) row-major (n, k), inside a longer buffer
    return buf[5:5 + n * k].view(n, k)


def view_col(buf, n, k):           # (b) column-major: the transpose of a (k, n) tensor
    return buf[3:3 + n * k].view(k, n).t()


def view_colslice(buf, n, k):      # (c) columns 3 .. 3+k of a wider row-major array (row stride k + 7)
    return buf[:(n + 2) * (k + 7)].view(n + 2, k + 7)[1:n + 1, 3:3 + k]


def view_rowslice(buf, n, k):      # (d) rows 1 .. 1+k of a vector-major basis with n + 9 columns (column stride > n)
    return buf[:(k + 2) * (n + 9)].view(k + 2, n + 9)[1:k + 1, 4:4 + n].t()


VIEWS = {"row": view_row, "col": view_col, "colslice": view_colslice, "rowslice": view_rowslice}
LAYOUTS = {"row": ("row", "row"), "col": ("col", "col"), "colslice": ("colslice", "colslice"),
           "rowslice": ("rowslice", "rowslice"), "mixed": ("row", "col"), "inplace": ("row", None)}


def buffer_size(n, k):
    return (n + 9) * (k + 7) + 16


def sentinel_buffer(D, size):
    return torch.full((size,), SENTINEL, dtype=torch.int64, device=D.dev()).view(torch.float64)


def solve_in_layout(D, fac, B, layout):
    """-> X (host), after checking that the solve wrote nothing outside X's view and left B's buffer untouched."""
    n, k = B.shape
    size = buffer_size(n, k)
    bl, xl = LAYOUTS[layout]
    bbuf = sentinel_buffer(D, size)
    Bv = VIEWS[bl](bbuf, n, k)
    Bv.copy_(torch.from_numpy(B))
    inside_b = np.zeros(size, dtype=bool)
    inside_b[VIEWS[bl](torch.arange(size), n, k).reshape(-1).numpy()] = True
    before = bbuf.view(torch.int64).cpu().numpy().copy()
    if xl is None:                                   # in place: X is B's view
        xbuf, Xv, inside_x = bbuf, Bv, inside_b
    else:
        xbuf = sentinel_buffer(D, size)
        Xv = VIEWS[xl](xbuf, n, k)
        inside_x = np.zeros(size, dtype=bool)
        inside_x[VIEWS[xl](torch.arange(size), n, k).reshape(-1).numpy()] = True
    fac.solve(Bv, out=Xv)
    after_x = xbuf.view(torch.int64).cpu().numpy()
    assert (after_x[~inside_x] == SENTINEL).all(), (layout, k, "the solve wrote outside its output view")
    if xl is not None:
        assert np.array_equal(bbuf.view(torch.int64).cpu().numpy(), before), (layout, k, "B was modified")
    X = Xv.cpu().numpy()
    assert np.isfinite(X).all(), (layout, k, "entries of X left unwritten")
    return X


@pytest.mark.parametrize("k", [1, 2, 5, 8, 16, 20, 40])
def test_layouts(D, rhs_case, k):
    """B is gathered through the permutation with its own strides and X scattered with its own, so every layout gives
    bitwise the same X as the row-major one."""
    c, sym, fac, B, X1 = rhs_case
    Bk = np.ascontiguousarray(B[:, :k])
    layouts = list(LAYOUTS) if k != 40 else ["row", "inplace"]     # k = 40: chunked solve in place
    Xs = {lay: solve_in_layout(D, fac, Bk, lay) for lay in layouts}
    ref = Xs["row"]
    assert eta(c.A, ref, Bk) <= ETA_SPD
    assert agree_with_single_columns(ref, X1[:, :k]) <= 1e-14
    for lay, X in Xs.items():
        assert np.array_equal(X.view(np.int64), ref.view(np.int64)), (lay, k)
