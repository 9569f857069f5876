"""TEST INFRASTRUCTURE ONLY -- matrices for the supernodal LDL^T tests (test_factor_shapes_cpu.py checks what each case
covers, test_factor_dense_ref_gpu.py factors and solves them on the device against dense / scipy references).

numpy / scipy only.  Every builder returns a Case: the symmetric matrix as a CSR with sorted indices (explicit zeros
kept in the pattern), optional node coordinates, dof_per_node, the symbolic options the case needs, and the number of
negative eigenvalues when it is known without an eigensolve (None otherwise).

  * dense_case: a fully dense pattern, which the symbolic analysis turns into ONE supernode of width n (n <= 512, with
    max_super_cols raised to 512): the widths straddle the 32-column pivot blocks and the 64 / 128 / 256 stages of the
    recursive-doubling inverse of the pivot block.
  * bordered_case: dense diagonal blocks joined by a dense border -- child fronts with a controlled number of rows
    below the pivot block (partial extend-add, TRSM and trailing-update tiles).
  * grid_case: finite-element grid patterns with 1, 2, 3 or 6 DOF per node, under several supernode caps and with or
    without relaxed amalgamation.
  * block_diagonal_case: disjoint dense blocks, whose solve plan has level-phase panel slices larger than the
    shared-memory ring of the pipelined level kernel.
  * kron_case: a shifted Kronecker-sum Laplacian whose spectrum is known in closed form, so that the number of
    eigenvalues below the shift (the inertia of the shifted factor) is exact at 50 000 DOF."""
import numpy as np
import scipy.sparse as sp

import fe_oracle as fo

# Symbolic(opts=...) pads the list with zeros and opts[3] = 0 means "no relaxation": pass -1 for the default
DENSE_OPTS = [0, 512, 0, -1]


class Case:
    def __init__(self, name, A, coords=None, dof=1, opts=None, nneg=None):
        self.name, self.A, self.coords, self.dof, self.opts = name, A, coords, dof, opts
        self.nneg = nneg            # eigenvalues below zero, when known in closed form

    @property
    def n(self):
        return self.A.shape[0]

    def __repr__(self):
        return "Case(%s, n=%d)" % (self.name, self.n)


def csr_from_dense(M, mask=None):
    """CSR of M on the pattern `mask` (default: every entry), zeros included."""
    n = M.shape[0]
    if mask is None:
        mask = np.ones((n, n), dtype=bool)
    i, j = np.nonzero(mask)
    A = sp.csr_matrix((M[i, j], (i, j)), shape=(n, n))
    A.sort_indices()
    assert A.nnz == mask.sum()
    return A


def random_orthogonal(n, rng):
    Q, R = np.linalg.qr(rng.normal(size=(n, n)))
    return Q * np.sign(np.diag(R))


def symmetric_with_spectrum(s, rng):
    Q = random_orthogonal(len(s), rng)
    M = (Q * s) @ Q.T
    return (M + M.T) * 0.5


DENSE_WIDTHS = [1, 2, 31, 32, 33, 63, 64, 65, 96, 127, 128, 129, 255, 256, 257, 300, 383, 511, 512]


def dense_case(w, kind, seed=0):
    """One supernode of width w.  kind:
      "spd"        Q diag(s) Q^T, s log-uniform in [1, 1e4] (both ends included);
      "indefinite" Q diag(s) Q^T with w // 3 (at least one) negative entries, |s| log-uniform in [1, 1e2];
      "saddle"     [[H, B^T], [B, 0]], H (w - p) x (w - p) SPD, B p x (w - p) random, p = max(1, w // 4): exactly p
                   negative eigenvalues, and a zero diagonal block that only a pivoted factor handles without
                   perturbation."""
    rng = np.random.default_rng(1000 * w + {"spd": 0, "indefinite": 1, "saddle": 2}[kind] + 7 * seed)
    if kind == "spd":
        s = np.exp(rng.uniform(0.0, np.log(1e4), w))
        s[0], s[-1] = 1.0, 1e4
        return Case("dense-spd-%d" % w, csr_from_dense(symmetric_with_spectrum(s, rng)), opts=DENSE_OPTS, nneg=0)
    if kind == "indefinite":
        nneg = max(1, w // 3)
        s = np.exp(rng.uniform(0.0, np.log(1e2), w))
        s[rng.permutation(w)[:nneg]] *= -1.0
        return Case("dense-indefinite-%d" % w, csr_from_dense(symmetric_with_spectrum(s, rng)), opts=DENSE_OPTS,
                    nneg=nneg)
    if kind == "saddle":
        assert w >= 2
        p = max(1, w // 4)
        m = w - p
        H = symmetric_with_spectrum(np.exp(rng.uniform(0.0, np.log(10.0), m)), rng)
        B = rng.normal(size=(p, m))
        M = np.zeros((w, w))
        M[:m, :m], M[m:, :m], M[:m, m:] = H, B, B.T
        # interleave the constraint rows with the others: the zero diagonal entries land inside every pivot block
        P = rng.permutation(w)
        return Case("dense-saddle-%d" % w, csr_from_dense(M[np.ix_(P, P)]), opts=DENSE_OPTS, nneg=p)
    raise ValueError(kind)


# (diagonal block widths, border width): widths either side of the 32-column edges
BORDERED_OPTS = [1, 512, 1, 0]
BORDERED = [((1, 31, 33, 65, 100, 257), 1), ((33, 65, 100, 7, 1), 40), ((31, 33, 64, 96), 31),
            ((65, 129, 32), 33), ((100, 31, 257), 97)]


def bordered_case(blocks, border, kind="spd", seed=0):
    """Dense diagonal blocks of the given widths, and a dense border of `border` rows / columns coupled to all of them,
    numbered last.  Options [1, 512, 1, 0]: no collapsed leaf subtrees (leaf_cols = 1) and no relaxation (relax = 0),
    so that every block stays one supernode with `border` rows below; nested dissection down to single vertices of the
    compressed graph (nd_leaf = 1), so that the border is the top separator; max_super_cols = 512 so that a 257-wide
    block stays whole.  kind "spd": random entries on the pattern plus a dominant diagonal; "shifted": that matrix
    minus the mid-point of the widest eigenvalue gap just above its 40 % quantile (indefinite, inertia from eigvalsh)."""
    rng = np.random.default_rng(seed + sum(blocks) + 31 * border)
    n = sum(blocks) + border
    mask = np.zeros((n, n), dtype=bool)
    o = 0
    for b in blocks:
        mask[o:o + b, o:o + b] = True
        o += b
    mask[o:, :] = mask[:, o:] = True
    M = np.where(mask, rng.uniform(-1.0, 1.0, (n, n)), 0.0)
    M = (M + M.T) * 0.5
    M[np.diag_indices(n)] = np.abs(M).sum(axis=1) + 0.1
    nneg = 0
    if kind == "shifted":
        ev = np.linalg.eigvalsh(M)
        m = int(0.4 * n)
        m = m + int(np.argmax(np.diff(ev[m:m + 20])))        # widest gap among the next few
        M[np.diag_indices(n)] -= 0.5 * (ev[m] + ev[m + 1])
        nneg = m + 1
    elif kind != "spd":
        raise ValueError(kind)
    name = "bordered-%s-%s+%d" % (kind, "/".join(map(str, blocks)), border)
    return Case(name, csr_from_dense(M, mask), opts=BORDERED_OPTS, nneg=nneg)


def block_diagonal_case(nblocks=400, w=96, seed=0):
    """nblocks disjoint dense SPD w x w blocks: one w-wide supernode each, all on one level of the tree and no subtree
    phases.  With w = 96 the level has 3 * nblocks 32-output tiles per direction, enough to give every warp of 148 SMs a
    tile of its own (ws = 1), so each front's widest tile multiplies a 96 x 32 panel slice of 24 576 bytes, larger than
    the 16 KB shared-memory ring of the pipelined level kernel: those tiles read their slice from global memory."""
    rng = np.random.default_rng(seed + nblocks + 7 * w)
    blocks = []
    for _ in range(nblocks):
        M = rng.uniform(-1.0, 1.0, (w, w))
        M = (M + M.T) * 0.5
        M[np.diag_indices(w)] = np.abs(M).sum(axis=1) + 0.1
        blocks.append(M)
    A = sp.block_diag(blocks, format="csr")
    A.sort_indices()
    return Case("block-diagonal-%dx%d" % (nblocks, w), A, nneg=0)


def grid_matrix(nx, ny, dof, seed):
    """SPD finite-element pattern (Q4 grid, `dof` DOF per node): random entries plus a dominant diagonal."""
    rng = np.random.default_rng(seed)
    conn, X = fo.grid_mesh(nx, ny, 1.0, ny / nx)
    i, j = fo.coo_index(fo.element_dofs(conn, dof))
    A = sp.coo_matrix((rng.uniform(-1, 1, len(i)), (i, j))).tocsr()
    A = (A + A.T) * 0.5
    A = (A + sp.diags(np.abs(A).sum(axis=1).A1 + 0.1)).tocsr()
    A.sort_indices()
    return A, X


# (dof per node, nx, ny): about 2 500 DOF each
GRID_SIZES = [(1, 60, 45), (2, 40, 30), (3, 32, 24), (6, 22, 17)]
GRID_CAPS = [32, 64, 256, 512]
# the 6-DOF case whose top separator (6 x 45 columns) is wider than 256 under the 512-column cap, and the two sizes of
# test_kernels_gpu.py whose solve plans have subtree phases (front mode) and thin tiles
WIDE_6DOF = (6, 50, 44, 512, 1)
FRONT_MODE = [(1, 250, 200, 0, -1), (2, 160, 120, 0, -1)]
# the right-hand-side sweep: one plan without subtree phases (level kernels only), one in front mode
RHS_LEVEL_ONLY = (1, 90, 70, 0, -1)
RHS_CASES = [RHS_LEVEL_ONLY, FRONT_MODE[0]]
GRID_CASES = ([(d, nx, ny, cap, relax) for d, nx, ny in GRID_SIZES for cap in GRID_CAPS for relax in (0, 1)]
              + [WIDE_6DOF] + FRONT_MODE)


def grid_case(dof, nx, ny, cap, relax):
    """cap = 0 keeps the default supernode cap (256); relax = -1 the default relaxation."""
    A, X = grid_matrix(nx, ny, dof, seed=nx * ny + dof)
    return Case("grid-%dx%dx%d-cap%d-relax%d" % (nx, ny, dof, cap, relax), A, coords=X, dof=dof,
                opts=[0, cap, 0, relax], nneg=0)


def dirichlet_eigenvalues(m):
    """Eigenvalues of the m x m second difference tridiag(-1, 2, -1)."""
    return 2.0 - 2.0 * np.cos(np.arange(1, m + 1) * np.pi / (m + 1))


def second_difference(m):
    return sp.diags([-np.ones(m - 1), 2.0 * np.ones(m), -np.ones(m - 1)], [-1, 0, 1])


KRON_C = np.array([[2.0, 0.6], [0.6, 1.0]])        # SPD node block of the 2-DOF variant
# (nx, ny, dof, shift target): coprime sides, about 30 ("shallow") and several hundred ("deep") eigenvalues below
KRON = [(251, 199, 1, 30), (251, 199, 1, 400), (163, 121, 2, 30), (163, 121, 2, 600)]
GAP_REL = 1e-6


def kron_spectrum(nx, ny, dof):
    lam = (dirichlet_eigenvalues(nx)[:, None] + dirichlet_eigenvalues(ny)[None, :]).ravel()
    if dof == 2:
        lam = (lam[:, None] * np.linalg.eigvalsh(KRON_C)[None, :]).ravel()
    return np.sort(lam)


def kron_shift(ev, target):
    """Shift in the widest gap of the sorted spectrum ev among positions target-10 .. target+10; -> (sigma, number of
    eigenvalues below sigma, relative gap)."""
    lo = target - 10
    m = lo + int(np.argmax(ev[lo + 1:target + 11] - ev[lo:target + 10]))
    sigma = 0.5 * (ev[m] + ev[m + 1])
    gap = min(sigma - ev[m], ev[m + 1] - sigma) / sigma
    assert gap >= GAP_REL, (target, gap)
    return sigma, m + 1, gap


def kron_case(nx, ny, dof, target):
    """A = (T_nx (x) I + I (x) T_ny) (x) C - sigma I on the nx x ny grid of nodes (C = 1 for one DOF per node), with
    node coordinates: its eigenvalues are (2 - 2cos(i pi/(nx+1)) + 2 - 2cos(j pi/(ny+1))) mu, mu an eigenvalue of C."""
    L = sp.kron(second_difference(nx), sp.identity(ny)) + sp.kron(sp.identity(nx), second_difference(ny))
    if dof == 2:
        L = sp.kron(L, sp.csr_matrix(KRON_C))
    ev = kron_spectrum(nx, ny, dof)
    sigma, nneg, gap = kron_shift(ev, target)
    A = (L - sigma * sp.identity(L.shape[0])).tocsr()
    A.sort_indices()
    X = np.stack(np.meshgrid(np.arange(nx, dtype=float), np.arange(ny, dtype=float), indexing="ij"), -1).reshape(-1, 2)
    c = Case("kron-%dx%dx%d-below%d" % (nx, ny, dof, nneg), A, coords=X, dof=dof, opts=None, nneg=nneg)
    c.sigma, c.gap, c.spectrum = sigma, gap, ev - sigma
    return c
