"""Device-side finite-element operators for the Q4 problems of the reference examples, the 3-D solid and 3-D heat
conduction on trilinear hexahedra (H8) and quadratic tetrahedra (T10).

Host part (numpy, runs once per mesh): mesh numbering, DOF maps, the CSR pattern of K/M and the
integer assembly maps (element, a, b) -> CSR non-zero, node -> element adjacency, the conic
filter pattern.  Device part (kernels of csrc/fe.cu): material interpolation, gather-form
assembly of K and M, the bilinear sensitivity forms ``w^T (dK/drho_e) v`` / ``w^T (dM/drho_e) v``
summed over modes, element -> node gather, filter products.

Mirrors (paths relative to the reference root):
  mesh / connectivity       examples/thermal.py:1475-1498, examples/natural_frequency.py:850-894
  DOF map and COO lists     examples/thermal.py:79-92, examples/natural_frequency.py:90-104
  K, M assembly             examples/thermal.py:126-148,192-214, examples/natural_frequency.py:134-160,205-236
  dK, dM callbacks          examples/thermal.py:150-190,216-246, examples/natural_frequency.py:162-203,238-284
  node scatter              examples/thermal.py:612-615
  node filter               examples/node_filter.py:61-88 (construction), :164-217 (apply / gradient)
"""
import numpy as np
import torch

from . import device as D
from ._hostdev import to_dev, like_input


def grid_mesh(nx, ny, Lx=1.0, Ly=1.0):
    """Structured Q4 mesh with the examples' numbering: node(i, j) = i*(ny+1) + j,
    element e = i + nx*j, counter-clockwise connectivity (examples/thermal.py:1475-1498)."""
    nodes = np.arange((nx + 1) * (ny + 1), dtype=np.int64).reshape(nx + 1, ny + 1)
    X = np.zeros(((nx + 1) * (ny + 1), 2))
    X[:, 0] = np.repeat(np.linspace(0, Lx, nx + 1), ny + 1)
    X[:, 1] = np.tile(np.linspace(0, Ly, ny + 1), nx + 1)
    conn = np.empty((nx * ny, 4), dtype=np.int64)
    conn[:, 0] = nodes[:-1, :-1].T.ravel()
    conn[:, 1] = nodes[1:, :-1].T.ravel()
    conn[:, 2] = nodes[1:, 1:].T.ravel()
    conn[:, 3] = nodes[:-1, 1:].T.ravel()
    return conn, X


def hex_mesh(nx, ny, nz, Lx=1.0, Ly=1.0, Lz=1.0):
    """Structured H8 mesh extending the numbering of ``grid_mesh``: node(i, j, k) = (i*(ny+1) + j)*(nz+1) + k,
    element e = i + nx*(j + ny*k); nodes 0-3 counter-clockwise (seen from +z) on the element's bottom face, 4-7 above
    them, so that detJ > 0.  Returns conn (nelems, 8) and X (nnodes, 3)."""
    nodes = np.arange((nx + 1) * (ny + 1) * (nz + 1), dtype=np.int64).reshape(nx + 1, ny + 1, nz + 1)
    grid = np.meshgrid(np.linspace(0, Lx, nx + 1), np.linspace(0, Ly, ny + 1), np.linspace(0, Lz, nz + 1), indexing="ij")
    X = np.stack([g.ravel() for g in grid], axis=1)
    corners = [(0, 0), (1, 0), (1, 1), (0, 1)]              # (di, dj) counter-clockwise
    conn = np.empty((nx * ny * nz, 8), dtype=np.int64)
    for dk in (0, 1):
        for a, (di, dj) in enumerate(corners):
            c = nodes[di:di + nx, dj:dj + ny, dk:dk + nz]
            conn[:, 4 * dk + a] = c.transpose(2, 1, 0).ravel()      # i fastest, then j, then k
    return conn, X


# corner pairs of the T10 midside nodes 4-9 (VTK quadratic tetra)
TET10_EDGES = ((0, 1), (1, 2), (2, 0), (0, 3), (1, 3), (2, 3))


def tet10_mesh(nx, ny, nz, Lx=1.0, Ly=1.0, Lz=1.0):
    """Structured T10 mesh of a box: nx x ny x nz cubes, each split into 6 tetrahedra around its main diagonal (the
    Kuhn split, conforming across cubes), with quadratic 10-node elements in VTK order.  The nodes are exactly the
    (2nx+1)(2ny+1)(2nz+1) points of the half-step lattice, numbered and placed as ``hex_mesh(2nx, 2ny, 2nz, ...)`` does,
    so that T10 and H8 models on the same nodes can be compared at equal DOF.  Element 6 c + t is tetrahedron t of cube
    c = i + nx*(j + ny*k); corner volumes are positive.  Returns conn (nelems, 10) and X (nnodes, 3)."""
    _, X = hex_mesh(2 * nx, 2 * ny, 2 * nz, Lx, Ly, Lz)
    cube = np.stack([a.transpose(2, 1, 0).ravel() for a in np.meshgrid(np.arange(nx), np.arange(ny), np.arange(nz),
                                                                        indexing="ij")], axis=1)   # i fastest
    unit = np.eye(3, dtype=np.int64)
    conn = np.empty((nx * ny * nz, 6, 10), dtype=np.int64)
    ny2, nz2 = 2 * ny + 1, 2 * nz + 1
    # the path (0,0,0) -> +e_a -> +e_b -> (1,1,1) of every axis order (a, b, c); odd orders have negative volume and
    # get corners 1 and 2 swapped
    for t, (order, odd) in enumerate((((0, 1, 2), 0), ((1, 2, 0), 0), ((2, 0, 1), 0),
                                      ((0, 2, 1), 1), ((2, 1, 0), 1), ((1, 0, 2), 1))):
        v1 = unit[order[0]]
        corners = [np.zeros(3, dtype=np.int64), v1, v1 + unit[order[1]], np.ones(3, dtype=np.int64)]
        if odd:
            corners[1], corners[2] = corners[2], corners[1]
        offsets = [2 * c for c in corners] + [corners[a] + corners[b] for a, b in TET10_EDGES]   # half-step lattice
        for a, off in enumerate(offsets):
            L = 2 * cube + off[None, :]
            conn[:, t, a] = (L[:, 0] * ny2 + L[:, 1]) * nz2 + L[:, 2]
    return conn.reshape(-1, 10), X


def tet10_from_tet4(conn4, X):
    """Quadratic tetrahedra from a linear tetrahedral mesh (conn4 (nelems, 4), X (nnodes, 3)), such as one a mesher
    writes: each edge gets one midside node at its midpoint, numbered after the corner nodes in the order of the sorted
    edge list.  Negatively oriented elements are flipped (corners 1 and 2 swapped); degenerate elements
    (|6 V| <= 1e-12 (longest edge)^3) raise ValueError.  Returns conn (nelems, 10) and X (nnodes + nedges, 3)."""
    conn4 = np.array(conn4, dtype=np.int64)
    X = np.asarray(X, dtype=np.float64)
    if conn4.ndim != 2 or conn4.shape[1] != 4 or X.ndim != 2 or X.shape[1] != 3:
        raise ValueError("tet10_from_tet4 needs conn (nelems, 4) and X (nnodes, 3)")
    xe = X[conn4]
    d = xe[:, 1:] - xe[:, :1]
    vol6 = np.einsum("ei,ei->e", d[:, 0], np.cross(d[:, 1], d[:, 2]))
    lmax = np.max([np.linalg.norm(xe[:, a] - xe[:, b], axis=1) for a, b in TET10_EDGES], axis=0)
    bad = np.abs(vol6) <= 1e-12 * lmax ** 3
    if bad.any():
        raise ValueError("tet10_from_tet4: %d degenerate element(s), the first is element %d"
                         % (bad.sum(), np.nonzero(bad)[0][0]))
    neg = vol6 < 0
    conn4[neg, 1], conn4[neg, 2] = conn4[neg, 2], conn4[neg, 1].copy()
    nn = np.int64(X.shape[0])
    ends = np.stack([conn4[:, [a, b]] for a, b in TET10_EDGES], axis=1)           # (nelems, 6, 2)
    key = ends.min(axis=2) * nn + ends.max(axis=2)
    ukey, inv = np.unique(key.ravel(), return_inverse=True)
    Xm = 0.5 * (X[ukey // nn] + X[ukey % nn])
    conn = np.concatenate([conn4, nn + inv.reshape(-1, 6)], axis=1)
    return conn, np.concatenate([X, Xm], axis=0)


def element_dofs(conn, dof):
    """var[e] = the element's global DOF list (examples/natural_frequency.py:90-92)."""
    conn = np.asarray(conn, dtype=np.int64)
    return (conn[:, :, None] * dof + np.arange(dof)[None, None, :]).reshape(conn.shape[0], -1)


def assembly_structure(var, ndof):
    """CSR pattern of sum_e P_e^T K_e P_e plus, for every non-zero, the list of (e, a, b) sources.

    The (i, j) lists are in ``Ke.flatten()`` order (examples/natural_frequency.py:94-104) and the
    CSR is what ``coo_matrix((vals, (i, j))).tocsr()`` produces (:157-158): duplicates summed,
    column indices sorted.  Returns indptr (int32), indices (int32), src_ptr (int64, nnz+1),
    src (int64, flat COO positions e*ne*ne + a*ne + b grouped by non-zero, ascending)."""
    ne = var.shape[1]
    i = np.repeat(var, ne, axis=1).ravel()
    j = np.tile(var, (1, ne)).ravel()
    key = i * np.int64(ndof) + j
    order = np.argsort(key, kind="stable")
    skey = key[order]
    first = np.ones(len(skey), dtype=bool)
    first[1:] = skey[1:] != skey[:-1]
    ukey = skey[first]
    rows = (ukey // ndof).astype(np.int64)
    indices = (ukey % ndof).astype(np.int32)
    indptr = np.zeros(ndof + 1, dtype=np.int64)
    np.add.at(indptr, rows + 1, 1)
    indptr = np.cumsum(indptr).astype(np.int32)
    src_ptr = np.concatenate([np.nonzero(first)[0], [len(skey)]]).astype(np.int64)
    return indptr, indices, src_ptr, order.astype(np.int64)


def node_adjacency(conn, nnodes):
    """CSR node -> elements (gather form of the ``np.add.at`` scatter, examples/thermal.py:612-615)."""
    conn = np.asarray(conn, dtype=np.int64)
    e = np.repeat(np.arange(conn.shape[0], dtype=np.int64), conn.shape[1])
    v = conn.ravel()
    order = np.lexsort((e, v))
    nptr = np.zeros(nnodes + 1, dtype=np.int64)
    np.add.at(nptr, v + 1, 1)
    return np.cumsum(nptr).astype(np.int32), e[order].astype(np.int32)


class AssemblyPattern:
    """The CSR pattern of assembled K/M matrices (``assembly_structure``) and, for every non-zero, the list of its
    (element, a, b) sources: ``indptr``, ``indices`` on the host, all four arrays in HBM.  The host copies of the source
    lists are not kept; ``reduced`` downloads them when it needs them."""

    def __init__(self, indptr, indices, src_ptr, src):
        dev = D.dev()
        self.indptr, self.indices = indptr, indices
        self.nnz = len(indices)
        self.shape = (len(indptr) - 1, len(indptr) - 1)
        self.indptr_d = torch.as_tensor(indptr, device=dev)
        self.indices_d = torch.as_tensor(indices, device=dev)
        self.src_ptr_d = torch.as_tensor(src_ptr, device=dev)
        self.src_d = torch.as_tensor(src, device=dev)

    def csr(self, vals):
        """The matrix with values ``vals`` (device, (nnz,)) on this pattern."""
        return D.CsrDevice(self.indptr_d, self.indices_d, vals, self.shape)

    def reduced(self, reduced):
        """The pattern of ``matrix[reduced, :][:, reduced]`` (``reduced_structure``)."""
        return AssemblyPattern(*reduced_structure(self.indptr, self.indices, to_host_i64(self.src_ptr_d),
                                                  to_host_i64(self.src_d), reduced, self.shape[0]))


def _penalty_law(name, ptype, p, q, c0, rho0):
    """Law and parameters of eigd_q4_material for the structural penalisation ``ptype`` ("simp": rho^p + rho0, "ramp":
    rho/(1+q(1-rho)) + rho0), mass factor c0 rho; ``name`` is the option the error message names."""
    if ptype == "simp":
        return 1, np.array([p, 1.0, c0, rho0])
    if ptype == "ramp":
        return 2, np.array([q, 1.0, c0, rho0])
    raise ValueError("unknown %s %r" % (name, ptype))


def _cols(t):
    """(n,) or (n, N) device operand -> contiguous (n, N)."""
    if t is None:
        return None
    t = t if t.dim() == 2 else t.unsqueeze(1)
    return t if t.is_contiguous() else t.contiguous()


class _SensitivityCallback:
    """A reference sensitivity callback such as ``dAdx(w, v)``: ``which`` of the operators of ``parent``, called with
    host or device operands; subclasses give its device form ``device_call(W, V)``."""

    def __init__(self, parent, which):
        self.parent, self.which = parent, which

    def __call__(self, w, v):
        return like_input(self.device_call(to_dev(w), to_dev(v)), w)


class _Half(_SensitivityCallback):
    """One of the two reference callbacks ``dAdx(w, v)`` / ``dBdx(w, v)``."""

    fused_with = None       # the other half: add_eig_total_derivative then evaluates both in one fused call

    def device_call(self, W, V):
        if self.which == "A":
            return self.parent.device_call_fused(W, None, V, 1.0, 0.0)
        return self.parent.device_call_fused(None, W, V, 0.0, 1.0)


class _ElementModel:
    """What the models with one density per element share: the mesh and its dof numbering, the assembly pattern, node
    adjacency, nodal density -> element density (the mean over the element's ``npe`` nodes) -> penalised material
    factors ks, ms and their derivatives dk, dm (eigd_q4_material with ``law``, ``par``), the assembly of K, M and of
    their tangent, and the element-range sharding of the fused sensitivities.  Subclasses give the element kernels:
    ``_assemble_values(ck, cm)`` and ``_quadforms(lo, hi, WA, WB, V, cA, cB)`` on the elements [lo, hi)."""

    def _setup(self, conn, X, nnodes, dof, law, par):
        dev = D.dev()
        self.conn, self.X = conn, X
        self.nelems, self.nnodes, self.dof = conn.shape[0], nnodes, dof
        self.ndof = dof * nnodes
        self.var = element_dofs(conn, dof)
        self.pattern = AssemblyPattern(*assembly_structure(self.var, self.ndof))
        self.indptr, self.indices, self.nnz = self.pattern.indptr, self.pattern.indices, self.pattern.nnz
        nptr, nelem = node_adjacency(conn, nnodes)
        self.conn_d = torch.as_tensor(conn.astype(np.int32), device=dev)
        self.nptr_d = torch.as_tensor(nptr, device=dev)
        self.nelem_d = torch.as_tensor(nelem, device=dev)
        self.law, self.par = law, par
        self.rhoE_d = D.empty(self.nelems)
        self.ks_d, self.ms_d = D.empty(self.nelems), D.empty(self.nelems)
        self.dk_d, self.dm_d = D.empty(self.nelems), D.empty(self.nelems)
        self.sharding = None          # dist.ModeSharding: element-range shards of the df/dx reduction
        self.dAdx, self.dBdx = _Half(self, "A"), _Half(self, "B")
        self.dAdx.fused_with, self.dBdx.fused_with = self.dBdx, self.dAdx

    # ---- material -------------------------------------------------------------------------------
    def set_density(self, rho=None, rhoE=None):
        """Nodal density rho (filtered design) -> element density + material factors, or set the
        element densities directly."""
        out = dict(ks=self.ks_d, ms=self.ms_d, dk=self.dk_d, dm=self.dm_d)
        if rhoE is not None:
            self.rhoE_d.copy_(to_dev(rhoE))
            D.element_material(self.law, self.par, self.rhoE_d, **out)
        else:
            D.element_material(self.law, self.par, to_dev(rho), conn=self.conn_d, rhoE=self.rhoE_d, **out)
        return self.rhoE_d

    def _element_mean(self, rho_t):
        """Element mean of the nodal vector ``rho_t``."""
        rhoEt = D.empty(self.nelems)
        D.element_material(self.law, self.par, to_dev(rho_t), conn=self.conn_d, rhoE=rhoEt)
        return rhoEt

    # ---- assembly -------------------------------------------------------------------------------
    def assemble(self):
        """K(rho), M(rho) as CsrDevice sharing one pattern (values computed in gather form)."""
        Kv, Mv = self._assemble_values(self.ks_d, self.ms_d)
        return self.pattern.csr(Kv), self.pattern.csr(Mv)

    def assemble_tangent(self, rho_t):
        """Directional derivative of (K, M) along the nodal density direction ``rho_t`` (device, (nnodes,)), on the same
        pattern: the assembly with the material factors replaced by (dk/drho_e) rho_e', (dm/drho_e) rho_e'.
        Used by the dual-number (complex-step) mode of the drivers."""
        rhoEt = self._element_mean(rho_t)
        Kv, Mv = self._assemble_values(self.dk_d * rhoEt, self.dm_d * rhoEt)
        return self.pattern.csr(Kv), self.pattern.csr(Mv)

    def dof_coords(self):
        """Node coordinates for geometric nested dissection (``SpLuOperator(coords=..., dof_per_node=...)``)."""
        return self.X, self.dof

    # ---- sensitivities ----------------------------------------------------------------------------
    def device_call_fused(self, WA, WB, V, cA, cB):
        """cA * sum_k WA_k^T (dK/drho_e) V_k + cB * sum_k WB_k^T (dM/drho_e) V_k per element (device).  With
        ``sharding``, every rank evaluates its element range and one all-gather joins them (dist.py)."""
        args = (_cols(WA), _cols(WB), _cols(V), float(cA), float(cB))
        shard = self.sharding
        if shard is None or shard.world == 1:
            return self._quadforms(0, self.nelems, *args)
        lo, hi = shard.my_range(self.nelems)
        return shard.allgather_ranges(self._quadforms(lo, hi, *args), self.nelems)

    def scatter_to_nodes(self, evals, scale=None):
        """rho_b[v] = scale * sum_{e ni v} evals[e] (examples/thermal.py:612-615); default scale 1 / npe, the transpose
        of the element mean."""
        ev = to_dev(evals)
        out = D.empty(self.nnodes)
        D.node_gather(self.nptr_d, self.nelem_d, ev, 1.0 / self.npe if scale is None else scale, out)
        return like_input(out, evals)


class Q4Problem(_ElementModel):
    """Thermal (1 DOF/node) or plane-stress (2 DOF/node) Q4 model with its operators in HBM.

    kind "thermal": K_e = kappa(rho_e) sum_q detJ Be^T Be, M_e = c(rho_e) sum_q detJ N N^T
      with kappa = kappa0((1-beta) rho^p + beta), c = cp*density*((1-beta) rho + beta)
      (examples/thermal.py:23-28,132,198).
    kind "plane_stress": K_e = s(rho_e) sum_q detJ Be^T C0 Be, M_e = density*rho_e sum_q detJ He^T He
      with s = rho^p + rho0_K (SIMP) or rho/(1+q(1-rho)) + rho0_K (RAMP)
      (examples/natural_frequency.py:83-86,140-155,219-231).
    """

    npe = 4

    def __init__(self, conn, X, kind="thermal", E=1.0, nu=0.3, kappa=1.0, density=1.0, heat_capacity=1.0, p=3.0,
                 beta=1e-6, rho0_K=1e-6, ptype_K="simp", q=5.0):
        if kind not in ("thermal", "plane_stress"):
            raise ValueError("unknown kind %r" % kind)
        self.kind = kind
        self.kid = 0 if kind == "thermal" else 1
        conn = np.asarray(conn, dtype=np.int64)
        if kind == "thermal":
            law, par = 0, np.array([p, kappa, heat_capacity * density, beta])
        else:
            law, par = _penalty_law("ptype_K", ptype_K, p, q, density, rho0_K)
        self._setup(conn, np.asarray(X, dtype=np.float64), int(conn.max()) + 1, 1 if kind == "thermal" else 2, law, par)
        C0 = E * np.array([[1.0, nu, 0.0], [nu, 1.0, 0.0], [0.0, 0.0, 0.5 * (1.0 - nu)]]) / (1.0 - nu**2)
        self.C0 = C0
        self.xy_d = to_dev(self.X)
        self.cmat6_d = to_dev(np.array([C0[0, 0], C0[0, 1], C0[0, 2], C0[1, 1], C0[1, 2], C0[2, 2]]))

    def _assemble_values(self, ck, cm):
        p = self.pattern
        Kv, Mv = D.empty(self.nnz), D.empty(self.nnz)
        D.q4_assemble(self.kid, self.conn_d, self.xy_d, ck, cm, self.cmat6_d, p.src_ptr_d, p.src_d, self.nnz, Kv, Mv)
        return Kv, Mv

    def _quadforms(self, lo, hi, WA, WB, V, cA, cB):
        out = D.zeros(hi - lo)
        D.q4_quadforms(self.kid, self.conn_d[lo:hi], self.xy_d, self.cmat6_d, WA, WB, V, self.dk_d[lo:hi], self.dm_d[lo:hi],
                       cA, -cB, out)
        return out


class _StoredMatrixModel(_ElementModel):
    """Element models whose unit element matrices are computed once per mesh and stay resident: ``K0_d``, ``M0_d``
    (nelems * NE * NE each, row-major) and the element dof map ``dofmap_d`` (nelems, NE).  Per design, assembly and
    the sensitivities are the stored-matrix kernels (eigd_stored_assemble, eigd_stored_quadform)."""

    def _setup_hex(self, conn, X, dof, law, par):
        """``_setup`` on a hexahedral mesh, conn (nelems, 8) and X (nnodes, 3) (ValueError otherwise), the element dof
        map and room for K0, M0, which the subclass's element kernel fills."""
        conn = np.asarray(conn, dtype=np.int64)
        X = np.asarray(X, dtype=np.float64)
        if conn.ndim != 2 or conn.shape[1] != 8 or X.ndim != 2 or X.shape[1] != 3:
            raise ValueError("%s needs conn (nelems, 8) and X (nnodes, 3)" % type(self).__name__)
        self._setup(conn, X, X.shape[0], dof, law, par)
        self.X_d = to_dev(np.ascontiguousarray(self.X))
        self.dofmap_d = torch.as_tensor(self.var.astype(np.int32), device=D.dev())
        ne2 = self.NE * self.NE
        self.K0_d, self.M0_d = D.empty(self.nelems * ne2), D.empty(self.nelems * ne2)

    def _setup_tet(self, conn, X, dof, law, par):
        """``_setup`` on a quadratic tetrahedral mesh, conn (nelems, 10) and X (nnodes, 3) (ValueError otherwise), the
        element dof map and room for K0, M0, which the subclass's element kernel fills."""
        conn = np.asarray(conn, dtype=np.int64)
        X = np.asarray(X, dtype=np.float64)
        if conn.ndim != 2 or conn.shape[1] != 10 or X.ndim != 2 or X.shape[1] != 3:
            raise ValueError("%s needs conn (nelems, 10) and X (nnodes, 3)" % type(self).__name__)
        self._setup(conn, X, X.shape[0], dof, law, par)
        self.X_d = to_dev(np.ascontiguousarray(self.X))
        self.dofmap_d = torch.as_tensor(self.var.astype(np.int32), device=D.dev())
        ne2 = self.NE * self.NE
        self.K0_d, self.M0_d = D.empty(self.nelems * ne2), D.empty(self.nelems * ne2)

    def _assemble_values(self, ck, cm):
        p = self.pattern
        Kv, Mv = D.empty(self.nnz), D.empty(self.nnz)
        D.stored_assemble(p.src_ptr_d, p.src_d, self.NE, self.K0_d, ck, Kv, F1=self.M0_d, d1=cm, vals2=Mv)
        return Kv, Mv

    def _quadforms(self, lo, hi, WA, WB, V, cA, cB):
        """Both terms in one pass of eigd_stored_quadform over the gathered V."""
        ne2 = self.NE * self.NE
        terms = [(W, U[lo * ne2:hi * ne2], c[lo:hi], s)
                 for W, U, c, s in ((WA, self.K0_d, self.dk_d, cA), (WB, self.M0_d, self.dm_d, cB)) if W is not None]
        (W1, U1, c1, s1), second = terms[0], terms[1:]
        out = D.zeros(hi - lo)
        if second:
            W2, F1, d1, s2 = second[0]
            D.stored_quadform(self.dofmap_d[lo:hi], U1, c1, W1, V, out, F1=F1, d1=d1, W2=W2, s1=s1, s2=s2)
        else:
            D.stored_quadform(self.dofmap_d[lo:hi], U1, c1, W1, V, out)
            if s1 != 1.0:
                out.mul_(s1)
        return out


class H8Problem(_StoredMatrixModel):
    """Free 3-D isotropic solid on trilinear hexahedra (3 DOF/node) with its operators in HBM.

    K_e = s(rho_e) K0_e, M_e = rho_e M0_e with s = rho^p + rho0_K (SIMP) or rho/(1+q(1-rho)) + rho0_K (RAMP), the laws
    of the plane-stress ``Q4Problem``; rho_e is the mean of the 8 nodal densities.  The unit matrices
    K0_e = sum_q detJ B^T C B and M0_e = density sum_q detJ (N N^T (x) I_3) (2x2x2 Gauss) are computed once per mesh on
    the device (eigd_h8_element_matrices, 9.2 KB per element) and stay resident; per design, assembly and the
    sensitivities are the stored-matrix kernels (eigd_stored_assemble, eigd_stored_quadform)."""

    npe = 8
    NE = 24

    def __init__(self, conn, X, E=1.0, nu=0.3, density=1.0, p=3.0, rho0_K=1e-6, ptype_K="simp", q=5.0):
        self._setup_hex(conn, X, 3, *_penalty_law("ptype_K", ptype_K, p, q, 1.0, rho0_K))
        D.h8_element_matrices(self.conn_d, self.X_d, E, nu, density, self.K0_d, self.M0_d)


class H8ThermalProblem(_StoredMatrixModel):
    """Heat conduction on trilinear hexahedra (1 DOF/node), the 3-D counterpart of ``Q4Problem(kind="thermal")``.

    K_e = kappa(rho_e) K0_e, M_e = c(rho_e) M0_e with the thermal law of ``Q4Problem``: kappa = kappa0((1-beta) rho^p
    + beta), c = heat_capacity * density * ((1-beta) rho + beta); rho_e is the mean of the 8 nodal densities.  The unit
    matrices K0_e = sum_q detJ grad N grad N^T and M0_e = sum_q detJ N N^T (2x2x2 Gauss) are computed once per mesh on
    the device (eigd_h8_thermal_element_matrices, 1 KB per element for the pair) and stay resident; per design, assembly
    and the sensitivities are the stored-matrix kernels, as for ``H8Problem``."""

    npe = 8
    NE = 8

    def __init__(self, conn, X, kappa=1.0, density=1.0, heat_capacity=1.0, p=3.0, beta=1e-6):
        self._setup_hex(conn, X, 1, 0, np.array([p, kappa, heat_capacity * density, beta]))
        D.h8_thermal_element_matrices(self.conn_d, self.X_d, self.K0_d, self.M0_d)


class T10Problem(_StoredMatrixModel):
    """Free 3-D isotropic solid on quadratic tetrahedra (T10, 3 DOF/node), with the material laws and interface of
    ``H8Problem``: K_e = s(rho_e) K0_e, M_e = rho_e M0_e, rho_e the mean of the 10 nodal densities.  The unit matrices
    K0_e = sum_q w_q detJ B^T C B and M0_e = density sum_q w_q detJ (N N^T (x) I_3) (14-point degree-5 rule) are
    computed once per mesh on the device (eigd_t10_element_matrices, 14.4 KB per element for the pair) and stay
    resident; per design, assembly and the sensitivities are the stored-matrix kernels.  Node order: ``tet10_mesh``."""

    npe = 10
    NE = 30

    def __init__(self, conn, X, E=1.0, nu=0.3, density=1.0, p=3.0, rho0_K=1e-6, ptype_K="simp", q=5.0):
        self._setup_tet(conn, X, 3, *_penalty_law("ptype_K", ptype_K, p, q, 1.0, rho0_K))
        D.t10_element_matrices(self.conn_d, self.X_d, E, nu, density, self.K0_d, self.M0_d)


class T10ThermalProblem(_StoredMatrixModel):
    """Heat conduction on quadratic tetrahedra (1 DOF/node), with the thermal law and interface of
    ``H8ThermalProblem``; rho_e is the mean of the 10 nodal densities.  The unit matrices K0_e = sum_q w_q detJ
    grad N grad N^T and M0_e = sum_q w_q detJ N N^T are computed once per mesh on the device
    (eigd_t10_thermal_element_matrices, 1.6 KB per element for the pair) and stay resident."""

    npe = 10
    NE = 10

    def __init__(self, conn, X, kappa=1.0, density=1.0, heat_capacity=1.0, p=3.0, beta=1e-6):
        self._setup_tet(conn, X, 1, 0, np.array([p, kappa, heat_capacity * density, beta]))
        D.t10_thermal_element_matrices(self.conn_d, self.X_d, self.K0_d, self.M0_d)


def reduced_structure(indptr, indices, src_ptr, src, reduced, ndof):
    """Pattern and (e, a, b) source lists of ``matrix[reduced, :][:, reduced]`` (examples/buckling.py:505-510)
    taken from those of the full matrix; the result equals scipy's fancy-indexed CSR bit for bit
    (``reduced`` ascending keeps rows and sorted columns in order)."""
    reduced = np.asarray(reduced, dtype=np.int64)
    f2r = np.full(ndof, -1, dtype=np.int64)
    f2r[reduced] = np.arange(len(reduced))
    rows = np.repeat(np.arange(ndof, dtype=np.int64), np.diff(indptr))
    keep = (f2r[rows] >= 0) & (f2r[indices] >= 0)
    cnt = np.zeros(len(reduced) + 1, dtype=np.int64)
    np.add.at(cnt, f2r[rows[keep]] + 1, 1)
    r_indptr = np.cumsum(cnt).astype(np.int32)
    r_indices = f2r[indices[keep]].astype(np.int32)
    lens = np.diff(src_ptr)[keep]
    r_src_ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    start = src_ptr[:-1][keep]
    pos = np.repeat(start - r_src_ptr[:-1], lens) + np.arange(int(r_src_ptr[-1]), dtype=np.int64)
    return r_indptr, r_indices, r_src_ptr, src[pos]


class _BucklingCallback(_SensitivityCallback):
    """dAdu / dAdx / dBdx of examples/buckling.py:924-979 as device operators on REDUCED (n_r, N) operands."""

    def device_call(self, Wr, Vr):
        return self.parent.sensitivity(self.which, Wr, Vr)


def node_local_index(conn):
    """For every (node, element) pair of ``node_adjacency`` order: the node's local index inside the element."""
    conn = np.asarray(conn, dtype=np.int64)
    nelems, npe = conn.shape
    e = np.repeat(np.arange(nelems, dtype=np.int64), npe)
    loc = np.tile(np.arange(npe, dtype=np.int64), nelems)
    return loc[np.lexsort((e, conn.ravel()))].astype(np.int32)


class _BucklingProblem:
    """What the Q4 and H8 buckling problems share around their element problem ``base`` (``Q4Problem`` /
    ``H8Problem``, which owns the mesh, K law and element density): Dirichlet conditions and loads on ``dof`` components
    per node, the reduced pattern and its source lists, the G material law, the Dirichlet maps, the fundamental path
    and the three sensitivity callbacks (``sensitivity`` of the subclass)."""

    def _setup(self, base, bcs, forces, p, q, density, rho0_G, ptype_G):
        dev = D.dev()
        self.base = b = base
        self.conn, self.X = b.conn, b.X
        self.nelems, self.nnodes, self.ndof, self.dof = b.nelems, b.nnodes, b.ndof, b.dof
        self.conn_d, self.nptr_d, self.nelem_d = b.conn_d, b.nptr_d, b.nelem_d
        # Dirichlet conditions {node: [components]} and loads {node: [f_0, .., f_dof-1]} (:120-150)
        dof = self.dof
        fixed = np.zeros(self.ndof, dtype=bool)
        for node, comps in bcs.items():
            for index in comps:
                if not 0 <= int(index) < dof:
                    raise ValueError("boundary condition on component %r of node %r: %d components per node"
                                     % (index, node, dof))
                fixed[dof * int(node) + int(index)] = True
        self.reduced = np.nonzero(~fixed)[0]
        self.nred = len(self.reduced)
        self.f = np.zeros(self.ndof)
        for node, fv in forces.items():
            for j in range(dof):
                self.f[dof * int(node) + j] += fv[j]
        self.pattern = b.pattern.reduced(self.reduced)
        self.indptr, self.indices, self.nnz = self.pattern.indptr, self.pattern.indices, self.pattern.nnz
        self.reduced_d = torch.as_tensor(self.reduced.astype(np.int32), device=dev)
        self.fr_d = to_dev(self.f[self.reduced])
        # local index of every node inside each adjacent element (dof gather of :318-320)
        self.nlocal_d = torch.as_tensor(node_local_index(self.conn), device=dev)
        # G material law (:231-234) and the RAMP parameters the reference differentiates it with (:333-336)
        self.lawG, self._parG = _penalty_law("ptype_G", ptype_G, p, q, density, rho0_G)
        self._pardG = [q + 1.0, 1.0, density, rho0_G]
        self.kg_d, self.dkg_d = D.empty(self.nelems), D.empty(self.nelems)
        self.u_d = None
        self.dGdu = _BucklingCallback(self, "dGdu")
        self.dGdx = _BucklingCallback(self, "dGdx")
        self.dKdx = _BucklingCallback(self, "dKdx")

    # ---- Dirichlet maps (:499-518) ----------------------------------------------------------------
    def full_vector(self, vr):
        return D.expand_rows(self.reduced_d, vr, self.ndof)

    def reduce_vector(self, v):
        return D.reduce_rows(self.reduced_d, v)

    def dof_coords(self):
        """Per-dof coordinates of the reduced system for geometric nested dissection."""
        return self.X[self.reduced // self.dof], 1

    # ---- material ------------------------------------------------------------------------------------
    def set_density(self, rho=None, rhoE=None):
        rhoE_d = self.base.set_density(rho=rho, rhoE=rhoE)
        D.element_material(self.lawG, self._parG, rhoE_d, ks=self.kg_d, dk=self.dkg_d)
        if self.lawG == 2:      # the reference differentiates the RAMP law of G with q + 1 (:336)
            D.element_material(self.lawG, self._pardG, rhoE_d, dk=self.dkg_d)
        return rhoE_d

    def set_displacement(self, ur_d):
        """u = full_vector(u_r): the fundamental path the stress stiffness is linearised about (:561-562)."""
        self.ur_d = ur_d
        self.u_d = self.full_vector(ur_d)
        return self.u_d

    def scatter_to_nodes(self, evals, scale=None):
        """rho_b[v] = scale * sum_{e ni v} evals[e]; default scale 1 / (nodes per element), the transpose of the element
        mean."""
        return self.base.scatter_to_nodes(evals, scale)


class BucklingQ4Problem(_BucklingProblem):
    """Plane-stress Q4 column of examples/buckling.py in HBM: K(x) with Dirichlet rows removed, the fundamental
    path K_r u_r = f_r, the stress stiffness G(u, x) and the three sensitivity callbacks.

    Element-level outputs stay per element (the node scatter ``np.add.at ... *0.25`` of :212-216, :337-341 is
    linear and is applied once at the end by the driver).  Reference: examples/buckling.py:152-343, 499-518.
    """

    def __init__(self, conn, X, bcs, forces, E=1.0, nu=0.3, density=1.0, p=3.0, q=5.0, rho0_K=1e-6, rho0_G=1e-9,
                 ptype_K="simp", ptype_G="simp"):
        base = Q4Problem(conn, X, "plane_stress", E=E, nu=nu, density=density, p=p, rho0_K=rho0_K, ptype_K=ptype_K, q=q)
        self._setup(base, bcs, forces, p, q, density, rho0_G, ptype_G)
        self.xy_d, self.cmat6_d = base.xy_d, base.cmat6_d

    # ---- assembly -------------------------------------------------------------------------------------
    def assemble_K(self):
        """K_r(rho) = reduce_matrix(get_stiffness_matrix(rhoE)) (:152-176, 505-510), values gathered directly
        through the reduced source lists."""
        b, p = self.base, self.pattern
        Kv = D.empty(self.nnz)
        D.q4_assemble(1, self.conn_d, self.xy_d, b.ks_d, b.ms_d, self.cmat6_d, p.src_ptr_d, p.src_d, self.nnz, Kv, None)
        return p.csr(Kv)

    def assemble_G(self):
        """G_r(u, rho) = reduce_matrix(get_stress_stiffness_matrix(rhoE, u)) (:220-255)."""
        p = self.pattern
        sdet = D.empty(self.nelems, 4, 3)
        D.q4_stress(self.conn_d, self.xy_d, self.cmat6_d, self.kg_d, self.u_d, sdet)
        Gv = D.empty(self.nnz)
        D.q4_assemble_geometric(self.conn_d, self.xy_d, sdet, p.src_ptr_d, p.src_d, self.nnz, Gv)
        return p.csr(Gv)

    def dK_single(self, psi_full, u_full):
        """psi^T (dK/drho_e) u per element for one pair of full vectors (:178-218 before the node scatter)."""
        out = D.zeros(self.nelems)
        b = self.base
        D.q4_quadforms(1, self.conn_d, self.xy_d, self.cmat6_d, psi_full.reshape(-1, 1), None, u_full.reshape(-1, 1),
                       b.dk_d, b.dm_d, 1.0, 0.0, out)
        return out

    # ---- sensitivities --------------------------------------------------------------------------------
    def sensitivity(self, which, Wr, Vr):
        """dGdu (full dof vector), dGdx or dKdx (per element) of sum_k w_k^T (.) v_k for reduced (n_r, N) W, V."""
        W2, V2 = _cols(self.full_vector(Wr)), _cols(self.full_vector(Vr))
        if which == "dGdu":
            due = D.empty(self.nelems, 8)
            D.q4_gderiv(self.conn_d, self.xy_d, self.cmat6_d, W2, V2, self.kg_d, self.dkg_d, self.u_d, 1.0, None, due)
            return D.dof_gather(self.nptr_d, self.nelem_d, self.nlocal_d, due, D.empty(self.ndof))
        out = D.zeros(self.nelems)
        if which == "dGdx":
            D.q4_gderiv(self.conn_d, self.xy_d, self.cmat6_d, W2, V2, self.kg_d, self.dkg_d, self.u_d, 1.0, out, None)
        else:                                                                     # dKdx
            D.q4_quadforms(1, self.conn_d, self.xy_d, self.cmat6_d, W2, None, V2, self.base.dk_d, self.base.dm_d, 1.0, 0.0,
                           out)
        return out


class BucklingH8Problem(_BucklingProblem):
    """Linearised buckling of a 3-D isotropic solid on trilinear hexahedra, with the interface of ``BucklingQ4Problem``:
    K_r(x) with the Dirichlet rows removed, the fundamental path K_r u_r = f_r, the stress stiffness G_r(u, x) and the
    three sensitivity callbacks.  ``bcs`` is {node: [components 0..2]}, ``forces`` {node: [fx, fy, fz]}.

    K_e = s(rho_e) K0_e as in ``H8Problem`` (whose unit matrices it uses), G_e = kg(rho_e) G0_e(u) with the G law of
    ``BucklingQ4Problem``.  Per design, eigd_h8_stress_stiffness writes the unit stress stiffness G0_e of the current
    fundamental path (24 x 24 per element, the layout of K0: 4.6 KB per element), so the assembly of G_r and dG/dx are
    the stored-matrix kernels, as K_r and dK/dx are.  The reduced operands are read through a reduced element dofmap
    (-1 on clamped dofs): no expansion to full vectors."""

    def __init__(self, conn, X, bcs, forces, E=1.0, nu=0.3, density=1.0, p=3.0, q=5.0, rho0_K=1e-6, rho0_G=1e-9,
                 ptype_K="simp", ptype_G="simp"):
        base = H8Problem(conn, X, E=E, nu=nu, density=density, p=p, rho0_K=rho0_K, ptype_K=ptype_K, q=q)
        self._setup(base, bcs, forces, p, q, density, rho0_G, ptype_G)
        self.E, self.nu = float(E), float(nu)
        self.X_d = base.X_d
        f2r = np.full(self.ndof, -1, dtype=np.int64)
        f2r[self.reduced] = np.arange(self.nred)
        self.dofmap_r_d = torch.as_tensor(f2r[base.var].astype(np.int32), device=D.dev())
        self.G0_d = D.empty(self.nelems * H8Problem.NE ** 2)
        self.stress_d = D.empty(self.nelems, 8, 6)          # kg C B_q u_e at the 8 Gauss points of every element

    def _assemble(self, E1, c1):
        p = self.pattern
        return p.csr(D.stored_assemble(p.src_ptr_d, p.src_d, H8Problem.NE, E1, c1, D.empty(self.nnz)))

    def _quadform(self, dofmap, E1, c1, W, V):
        return D.stored_quadform(dofmap, E1, c1, _cols(W), _cols(V), D.zeros(self.nelems))

    def assemble_K(self):
        """K_r(rho), gathered directly through the reduced source lists."""
        return self._assemble(self.base.K0_d, self.base.ks_d)

    def assemble_G(self):
        """G_r(u, rho) about the displacement of ``set_displacement``: element stresses and G0 of this path, then
        the gather-form assembly with the coefficients kg."""
        D.h8_stress_stiffness(self.conn_d, self.X_d, self.E, self.nu, self.kg_d, self.dofmap_r_d, self.ur_d, self.stress_d,
                              self.G0_d)
        return self._assemble(self.G0_d, self.kg_d)

    def dK_single(self, psi_full, u_full):
        """psi^T (dK/drho_e) u per element for one pair of full vectors."""
        return self._quadform(self.base.dofmap_d, self.base.K0_d, self.base.dk_d, psi_full, u_full)

    def sensitivity(self, which, Wr, Vr):
        """dGdu (full dof vector), dGdx or dKdx (per element) of sum_k w_k^T (.) v_k for reduced (n_r, N) W, V."""
        if which == "dGdu":
            W2, V2 = _cols(Wr), _cols(Vr)
            due = D.h8_gderiv_u(self.conn_d, self.X_d, self.E, self.nu, self.kg_d, self.dofmap_r_d, W2, V2,
                                D.empty(self.nelems, H8Problem.NE))
            return D.dof_gather(self.nptr_d, self.nelem_d, self.nlocal_d, due, D.empty(self.ndof))
        if which == "dGdx":
            return self._quadform(self.dofmap_r_d, self.G0_d, self.dkg_d, Wr, Vr)
        return self._quadform(self.dofmap_r_d, self.base.K0_d, self.base.dk_d, Wr, Vr)


def _contig1(t):
    return t if t.is_contiguous() else t.contiguous()


def to_host_i64(t):
    return t.detach().cpu().numpy().astype(np.int64)


class NodeFilter:
    """Conic node filter F[i, j] ~ max(0, r0 - |X_i - X_j|), rows normalised to 1
    (examples/node_filter.py:61-88), applied on the device as CSR products (:164-217).
    Spatial filter with optional design-variable map (the symmetric column of examples/buckling.py:1331-1344)
    and optional tanh projection (``projection=True``, ``beta``, ``eta``).  ``ftype="helmholtz"`` is the PDE filter
    (``_init_helmholtz``) on a Q4 mesh (2-D coordinates) or a hexahedral or T10 mesh (3-D coordinates); in 3-D it replaces the
    conic filter's pair search and its two CSR operators by one scalar LDL^T of the mesh, factored once."""

    ftype = "spatial"

    def __init__(self, conn, X, r0=1.0, ftype="spatial", dvmap=None, num_design_vars=None, beta=10.0, eta=0.5,
                 projection=False):
        from scipy import sparse, spatial
        if ftype not in ("spatial", "helmholtz"):
            raise ValueError("unknown filter type %r" % ftype)
        self.ftype = ftype
        self.projection = bool(projection)
        self.beta = 10.0 if beta is None else float(beta)      # reference default (node_filter.py:30-31)
        self.eta = float(eta)
        self.X = np.asarray(X, dtype=np.float64)
        self.nnodes = self.X.shape[0]
        self.r0 = r0
        self.dvmap = None if dvmap is None else np.asarray(dvmap, dtype=np.int64)
        self.offset_d = None
        if ftype == "helmholtz":
            self._init_helmholtz(conn, r0, num_design_vars)
            return
        tree = spatial.cKDTree(self.X)
        Dm = tree.sparse_distance_matrix(tree, r0, output_type="coo_matrix")
        w = r0 - Dm.data
        F = sparse.coo_matrix((w, (Dm.row, Dm.col)), shape=(self.nnodes, self.nnodes)).tocsr()
        rs = np.asarray(F.sum(axis=1)).ravel()
        F = (sparse.diags(1.0 / rs) @ F).tocsr()
        self.dvmap = None if dvmap is None else np.asarray(dvmap, dtype=np.int64)
        self.offset_d = None
        if self.dvmap is None:
            self.num_design_vars = self.nnodes
        else:
            # design-variable map (examples/node_filter.py:164-168, 211-214): rho = F x[dvmap] with x := 1 where
            # dvmap < 0, gradient scattered back with np.add.at.  Folded into the operator: F <- F P,
            # P[i, dvmap[i]] = 1, plus the constant F 1_{dvmap<0}; the transpose product is then the gather form
            # of the np.add.at scatter.
            self.num_design_vars = int(num_design_vars if num_design_vars is not None else self.dvmap.max() + 1)
            act = self.dvmap >= 0
            P = sparse.coo_matrix((np.ones(int(act.sum())), (np.nonzero(act)[0], self.dvmap[act])),
                                  shape=(self.nnodes, self.num_design_vars)).tocsr()
            if not act.all():
                self.offset_d = to_dev(F @ (~act).astype(np.float64))
            F = (F @ P).tocsr()
        F.sort_indices()
        FT = F.T.tocsr()
        FT.sort_indices()
        self.F, self.FT = F, FT
        self.F_d = D.CsrDevice.from_scipy(F)
        self.FT_d = D.CsrDevice.from_scipy(FT)

    def _init_helmholtz(self, conn, r0, num_design_vars):
        """Helmholtz (PDE) filter of examples/node_filter.py:90-162: rho = A^-1 (B x) with A = r0^2 int grad N . grad N +
        int N N and B = int N N on the element mesh: Q4 for 2-D coordinates with 4-node ``conn``, trilinear hexahedra or
        quadratic tetrahedra for 3-D coordinates with 8- or 10-node ``conn``.  A and B are the unit-material conductivity
        / capacity matrices of ``Q4Problem(kind="thermal")``, ``H8ThermalProblem`` or ``T10ThermalProblem`` (assembled
        by the same kernels), A is factored once by the
        GPU LDL^T (the reference uses scipy's ``factorized``) and applied to one right-hand side per call."""
        from .eigenvector_derivatives import SpLuOperator
        conn = np.asarray(conn, dtype=np.int64)
        dim, npe = self.X.shape[1] if self.X.ndim == 2 else 0, conn.shape[1] if conn.ndim == 2 else 0
        fronts = "resident"
        if (dim, npe) == (2, 4):
            prob = Q4Problem(conn, self.X, "thermal", kappa=1.0, density=1.0, heat_capacity=1.0, p=1.0, beta=0.0)
        elif (dim, npe) in ((3, 8), (3, 10)):
            prob = (H8ThermalProblem if npe == 8 else T10ThermalProblem)(conn, self.X, p=1.0, beta=0.0)
            # A is factored once and only solved with afterwards, so a pooled factor keeps no dense fronts for the
            # filter's life (17 GB at 80 x 64 x 48 hexahedra); it is bitwise the resident factor.
            fronts = "pooled"
        else:
            raise ValueError("the Helmholtz filter needs 2-D coordinates with 4-node (Q4) conn or 3-D coordinates with "
                             "8-node (H8) or 10-node (T10) conn; got %d-D coordinates with %d-node conn" % (dim, npe))
        prob.set_density(rhoE=np.ones(prob.nelems))
        K, M = prob.assemble()
        self._hB = M
        vals = D.axpby(float(r0) ** 2, K.data, 1.0, M.data)
        self._hA = SpLuOperator(K.with_values(vals), coords=self.X, dof_per_node=1, max_rhs=1, fronts=fronts)
        self._hprob = prob
        if self.dvmap is None:
            self.num_design_vars = self.nnodes
            self._dv_d = self._act_d = None
        else:
            dev = D.dev()
            self.num_design_vars = int(num_design_vars if num_design_vars is not None else self.dvmap.max() + 1)
            act = self.dvmap >= 0
            self._dv_d = torch.as_tensor(np.where(act, self.dvmap, 0), device=dev)
            self._act_d = torch.as_tensor(act, device=dev)
            self._act_idx = torch.as_tensor(np.nonzero(act)[0], device=dev)
            self._act_dv = torch.as_tensor(self.dvmap[act], device=dev)

    def _expand_design(self, x_d):
        if self.dvmap is None:
            return x_d
        xn = x_d.index_select(0, self._dv_d)                     # x[dvmap], and x := 1 where dvmap < 0 (:166-168)
        return torch.where(self._act_d, xn, torch.ones_like(xn))

    def _filtered(self, x_d):
        if self.ftype == "helmholtz":
            return self._hA.solve_dev(self._hB.spmm(self._expand_design(x_d)))
        rho = self.F_d.spmm(x_d)
        if self.offset_d is not None:
            D.axpby(1.0, rho, 1.0, self.offset_d, out=rho)
        return rho

    def _project(self, rho, g=None):
        return D.filter_project(rho, self.beta, self.eta, g)

    def apply_tangent(self, x, xt):
        """Directional derivative of ``apply`` at x along xt (dual-number mode of the drivers)."""
        x_d, xt_d = to_dev(x), to_dev(xt)
        if self.ftype == "helmholtz":
            xt_n = xt_d if self.dvmap is None else torch.where(self._act_d, xt_d.index_select(0, self._dv_d), torch.zeros_like(self._dv_d, dtype=xt_d.dtype))
            rt = self._hA.solve_dev(self._hB.spmm(xt_n))
        else:
            rt = self.F_d.spmm(xt_d)                       # the constant offset of the dv-map has no derivative
        if self.projection:
            rt = self._project(self._filtered(x_d), _contig1(rt))
        return rt

    def apply(self, x):
        rho = self._filtered(to_dev(x))
        if self.projection:                                    # node_filter.py:174-181
            rho = self._project(rho)
        return like_input(rho, x)

    def apply_gradient(self, g, x=None, rho=None):
        g_d = to_dev(g)
        if self.projection:                                    # node_filter.py:187-203: needs the unprojected field
            if x is None:
                raise ValueError("apply_gradient with projection needs the design x")
            g_d = self._project(self._filtered(to_dev(x)), _contig1(g_d))
        if self.ftype == "helmholtz":                          # g0 = B^T A^-1 grad (:205-209), then the dv-map scatter (:211-214)
            g0 = self._hB.spmm(self._hA.solve_dev(_contig1(g_d)))
            if self.dvmap is not None:
                out = D.zeros(self.num_design_vars)
                out.index_add_(0, self._act_dv, g0.index_select(0, self._act_idx))
                g0 = out
            return like_input(g0, g)
        return like_input(self.FT_d.spmm(g_d), g)
