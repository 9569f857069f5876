"""CRM-scale synthetic shell model on the device: the driver of reference ``examples/crm.py`` without TACS.

The reference's fourth example takes K, M and the design sensitivities from TACS (a shell finite-element code that is
not available here) and calls the eigd solvers with the per-mode "vector" derivative form (crm.py:212-376: ``IRAM`` /
``BasicLanczos`` -> ``solve_adjoint`` -> ``add_eig_total_derivative`` without ``deriv_type``, i.e. one ``dAdx(w, v)`` /
``dBdx(w, v)`` call per mode, each returning one value per design variable; SURVEY.md section 8 config C4).  This module
supplies a self-contained model of the same shape:

  * a structured Q4 mesh on a curved surface in 3-D, 6 DOF per node (u, v, w, theta_x, theta_y, theta_z);
  * flat facet shell elements: membrane (plane stress) + Mindlin bending and transverse shear + a drilling
    penalty, 2 x 2 Gauss, rotated into global axes -> 24 x 24 element matrices
        K_e = t E1_e + t^3 E3_e,      M_e = t F1_e + t^3 F3_e
    (E1: membrane + shear + drilling, E3: bending; F1: translational inertia, F3: rotary inertia);
  * design variables = one shell thickness per component (patches of elements), x = scale * t as in crm.py:113;
  * clamped nodes removed from the system (crm.py:143-181 ``_create_reduced_indices`` / ``_delete_rows_and_columns``).

The unit matrices E1, E3, F1, F3 are computed once on the host (vectorised numpy) and stay resident in HBM (3 GB at
1 M DOF); per design the device assembles K(t), M(t) in gather form (``eigd_stored_assemble``) and evaluates the
sensitivities w^T (dK/dt_c) v per component with one warp per element and a warp-shuffle segmented reduction
(``eigd_stored_quadform``, ``eigd_segment_sum``).
"""
import numpy as np
import torch

from . import device as D
from . import fe
from ._hostdev import to_dev, to_host, small_to_dev
from .eigenvector_derivatives import SpLuOperator, add_eig_total_derivative
from .topo import _EigenAnalysis, _now


# ------------------------------------------------------------------------------------------
# host: mesh and unit element matrices
# ------------------------------------------------------------------------------------------
def cylindrical_panel(nx, ny, Ls=1.0, Ly=1.0, radius=2.0):
    """Structured nx x ny Q4 mesh on a cylindrical panel: arc length s in [0, Ls] around the y axis, y in [0, Ly].
    Node (i, j) = i * (ny + 1) + j, element e = i + nx * j (the numbering of the reference's 2-D examples).
    Returns conn (nelems, 4), X (nnodes, 3), the parametric grid coordinates (nnodes, 2)."""
    conn, P = fe.grid_mesh(nx, ny, Ls, Ly)
    s, y = P[:, 0], P[:, 1]
    X = np.stack([radius * np.sin(s / radius), y, radius * (1.0 - np.cos(s / radius))], axis=1)
    return conn, X, P


def shell_unit_matrices(conn, X, E=73.1e9, nu=0.33, rho=2780.0, kshear=5.0 / 6.0, kdrill=1e-3):
    """(E1, E3, F1, F3), each (nelems, 24, 24) in GLOBAL axes, element dof order node-major (u, v, w, tx, ty, tz)."""
    conn = np.asarray(conn, dtype=np.int64)
    p = np.asarray(X, dtype=np.float64)[conn]                      # (ne, 4, 3)
    ne = p.shape[0]
    c = p.mean(axis=1, keepdims=True)
    v1 = (p[:, 1] + p[:, 2] - p[:, 0] - p[:, 3])
    v2 = (p[:, 2] + p[:, 3] - p[:, 0] - p[:, 1])
    e1 = v1 / np.linalg.norm(v1, axis=1, keepdims=True)
    nrm = np.cross(e1, v2)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    e2 = np.cross(nrm, e1)
    R = np.stack([e1, e2, nrm], axis=1)                            # (ne, 3, 3): local = R @ global
    xl = np.einsum("eaj,ej->ea", p - c, e1)
    yl = np.einsum("eaj,ej->ea", p - c, e2)
    Dp = E / (1.0 - nu * nu) * np.array([[1.0, nu, 0.0], [nu, 1.0, 0.0], [0.0, 0.0, 0.5 * (1.0 - nu)]])
    G = E / (2.0 * (1.0 + nu))
    K1 = np.zeros((ne, 24, 24))
    K3 = np.zeros((ne, 24, 24))
    M1 = np.zeros((ne, 24, 24))
    M3 = np.zeros((ne, 24, 24))
    area = np.zeros(ne)
    gp = 1.0 / np.sqrt(3.0)
    iu, iv, iw, itx, ity, itz = (np.arange(4) * 6 + d for d in range(6))
    for xi in (-gp, gp):
        for eta in (-gp, gp):
            N = 0.25 * np.array([(1 - xi) * (1 - eta), (1 + xi) * (1 - eta), (1 + xi) * (1 + eta), (1 - xi) * (1 + eta)])
            Nxi = 0.25 * np.array([-(1 - eta), (1 - eta), (1 + eta), -(1 + eta)])
            Neta = 0.25 * np.array([-(1 - xi), -(1 + xi), (1 + xi), (1 - xi)])
            J00, J01 = xl @ Nxi, yl @ Nxi
            J10, J11 = xl @ Neta, yl @ Neta
            det = J00 * J11 - J01 * J10
            Nx = (J11[:, None] * Nxi[None, :] - J01[:, None] * Neta[None, :]) / det[:, None]
            Ny = (-J10[:, None] * Nxi[None, :] + J00[:, None] * Neta[None, :]) / det[:, None]
            area += det
            Bm = np.zeros((ne, 3, 24))                              # membrane strains
            Bm[:, 0, iu] = Nx
            Bm[:, 1, iv] = Ny
            Bm[:, 2, iu] = Ny
            Bm[:, 2, iv] = Nx
            Bb = np.zeros((ne, 3, 24))                              # curvatures: u = z ty, v = -z tx
            Bb[:, 0, ity] = Nx
            Bb[:, 1, itx] = -Ny
            Bb[:, 2, ity] = Ny
            Bb[:, 2, itx] = -Nx
            Bs = np.zeros((ne, 2, 24))                              # transverse shear
            Bs[:, 0, iw] = Nx
            Bs[:, 0, ity] = N[None, :]
            Bs[:, 1, iw] = Ny
            Bs[:, 1, itx] = -N[None, :]
            bt = lambda B: np.ascontiguousarray(B.transpose(0, 2, 1))   # noqa: E731
            K1 += det[:, None, None] * (np.matmul(bt(Bm), np.matmul(Dp[None], Bm)) + kshear * G * np.matmul(bt(Bs), Bs))
            K3 += det[:, None, None] * np.matmul(bt(Bb), np.matmul(Dp[None] / 12.0, Bb))
            NN = np.outer(N, N)
            for idx in (iu, iv, iw):
                M1[:, idx[:, None], idx[None, :]] += rho * det[:, None, None] * NN[None]
            for idx in (itx, ity, itz):
                M3[:, idx[:, None], idx[None, :]] += rho / 12.0 * det[:, None, None] * NN[None]
    K1[:, itz, itz] += (kdrill * E * area / 4.0)[:, None]           # drilling penalty (Zienkiewicz), ~ t
    T = np.zeros((ne, 24, 24))
    for a in range(8):
        T[:, 3 * a:3 * a + 3, 3 * a:3 * a + 3] = R
    Tt = np.ascontiguousarray(T.transpose(0, 2, 1))
    rot = lambda A: np.matmul(np.matmul(Tt, A), T)                  # noqa: E731   T^T A T (batched)
    return rot(K1), rot(K3), rot(M1), rot(M3)


# ------------------------------------------------------------------------------------------
# device operators
# ------------------------------------------------------------------------------------------
class _ShellCallback(fe._SensitivityCallback):
    """``dAdx(w, v)`` / ``dBdx(w, v)`` of crm.py:331-355: one value per design variable (component thickness)."""

    def device_call(self, W, V):
        return self.parent._sensitivity(self.which, W, V)


class ShellProblem:
    """Flat-shell Q4 model with its unit element matrices in HBM; K(t), M(t) and their thickness sensitivities."""

    NE = 24

    def __init__(self, conn, X, comp, fixed_nodes, order_coords=None, scale=100.0, **material):
        dev = D.dev()
        self.conn = np.asarray(conn, dtype=np.int64)
        self.X = np.asarray(X, dtype=np.float64)
        self.nelems, self.nnodes = self.conn.shape[0], self.X.shape[0]
        self.ndof_full = 6 * self.nnodes
        self.comp = np.asarray(comp, dtype=np.int64)
        self.ncomp = int(self.comp.max()) + 1
        self.scale = float(scale)
        fixed = np.zeros(self.nnodes, dtype=bool)
        fixed[np.asarray(fixed_nodes, dtype=np.int64)] = True
        self.free_nodes = np.nonzero(~fixed)[0]
        self.reduced = (self.free_nodes[:, None] * 6 + np.arange(6)[None, :]).ravel()     # crm.py self.dof
        self.ndof = len(self.reduced)
        var = fe.element_dofs(self.conn, 6)                                          # (nelems, 24) full dofs
        # only the reduced pattern goes to HBM: the full one is reduced on the host
        self.pattern = fe.AssemblyPattern(*fe.reduced_structure(*fe.assembly_structure(var, self.ndof_full), self.reduced,
                                                                self.ndof_full))
        self.indptr, self.indices, self.nnz = self.pattern.indptr, self.pattern.indices, self.pattern.nnz
        f2r = np.full(self.ndof_full, -1, dtype=np.int64)
        f2r[self.reduced] = np.arange(self.ndof)
        self.dofmap = f2r[var].astype(np.int32)                                      # -1 = clamped
        oc = self.X if order_coords is None else np.asarray(order_coords, dtype=np.float64)
        self._order_coords = np.ascontiguousarray(oc[self.free_nodes])
        E1, E3, F1, F3 = shell_unit_matrices(self.conn, self.X, **material)
        self.E1_d, self.E3_d = to_dev(E1.reshape(-1)), to_dev(E3.reshape(-1))
        self.F1_d, self.F3_d = to_dev(F1.reshape(-1)), to_dev(F3.reshape(-1))
        del E1, E3, F1, F3
        self.dofmap_d = torch.as_tensor(self.dofmap, device=dev)
        # elements sorted by component: segments of the per-component reduction
        order = np.argsort(self.comp, kind="stable")
        seg = np.zeros(self.ncomp + 1, dtype=np.int64)
        np.add.at(seg, self.comp + 1, 1)
        self.seg_ptr_d = torch.as_tensor(np.cumsum(seg).astype(np.int32), device=dev)
        self.perm_d = torch.as_tensor(order.astype(np.int32), device=dev)
        self.comp_d = torch.as_tensor(self.comp, device=dev)
        self.t_d = None
        self.sharding = None
        self.dAdx, self.dBdx = _ShellCallback(self, "A"), _ShellCallback(self, "B")

    def dof_coords(self):
        return self._order_coords, 6

    def set_design(self, x):
        """x = scale * thickness per component (crm.py:110-114)."""
        x_d = to_dev(x)
        self.t_d = (x_d / self.scale)[self.comp_d].contiguous()      # per-element thickness
        self.t3_d = (self.t_d ** 3).contiguous()
        self.dt3_d = (3.0 * self.t_d ** 2).contiguous()
        self.one_d = torch.ones_like(self.t_d)
        return self.t_d

    def assemble(self):
        """K(t), M(t) as CsrDevice sharing one pattern (reduced system)."""
        p = self.pattern
        Kv, Mv = D.empty(self.nnz), D.empty(self.nnz)
        D.stored_assemble(p.src_ptr_d, p.src_d, self.NE, self.E1_d, self.t_d, Kv, E3=self.E3_d, c3=self.t3_d, F1=self.F1_d,
                          d1=self.t_d, vals2=Mv, F3=self.F3_d, d3=self.t3_d)
        return p.csr(Kv), p.csr(Mv)

    def _sensitivity(self, which, W, V):
        """d/dx_c of W^T A(x) V summed over the columns: (ncomp,) device vector."""
        U1, U3 = (self.E1_d, self.E3_d) if which == "A" else (self.F1_d, self.F3_d)
        oute = D.stored_quadform(self.dofmap_d, U1, self.one_d, fe._cols(W), fe._cols(V), D.empty(self.nelems), E3=U3,
                                 c3=self.dt3_d)
        return D.segment_sum(self.seg_ptr_d, self.perm_d, oute, 1.0 / self.scale, D.empty(self.ncomp))


class ShellModalAnalysis(_EigenAnalysis):
    """The ``CRM`` driver of examples/crm.py (:19-376) on the synthetic shell: same method names, same ``profile`` keys,
    modal-compliance objective with f[1::6] = 1 (:267-293), per-mode "vector" total derivative (:357-370)."""

    def __init__(self, prob, N=10, m=None, omega0=10.0, solver_type="IRAM", tol=1e-14, rtol=1e-10, eig_atol=1e-5,
                 adjoint_method="sibk", adjoint_options=None, deriv_type="vector", seed=0, fronts="resident"):
        super().__init__(prob, N, m, solver_type, tol, rtol, eig_atol, adjoint_method, adjoint_options, deriv_type, seed,
                         fronts)
        self.omega0 = omega0
        self.x = np.ones(prob.ncomp)                       # crm.py: t = 0.01, scale 100
        f = np.zeros(prob.ndof_full)
        f[1::6] = 1.0
        self.fr_d = to_dev(f[prob.reduced])

    def get_design_vars(self):
        return np.array(self.x)

    def set_design_vars(self, x0):
        self.x = np.array(x0, dtype=float)

    def initialize(self):
        p = self.prob
        self.profile.update({"solver_type": self.solver_type, "adjoint_method": self.adjoint_method, "N": self.N})
        t0 = _now()
        p.set_design(self.x)
        self.Kr, self.Mr = p.assemble()
        t1 = _now()
        self.profile["matrix assembly time"] = t1 - t0
        sigma = self.omega0 ** 2
        self.sigma = sigma
        vals = D.axpby(1.0, self.Kr.data, -float(sigma), self.Mr.data)
        if self._symbolic_once(self.Kr) is not None:
            t1 = _now()                                    # the eigensolve time excludes the analysis
        self.factor = SpLuOperator(self.Kr.with_values(vals), symbolic=self.symbolic, fronts=self.fronts)
        self._new_eig_solver(self.N)
        self.lam = np.asarray(self._eigensolve(self.Kr, self.Mr, sigma, t1))
        self.Q = self.eig_solver._Phi_d

    def initialize_adjoint(self):
        self.Qb = D.zeros(self.prob.ndof, self.N)
        self.lamb = np.zeros(self.N)

    def get_compliance(self):
        """sum_i (phi_i . f)^2 / lam_i  (crm.py:267-280)"""
        val = to_host(D.gemm_tn(self.Q, self.fr_d)).ravel()
        return float(np.sum(val * val / self.lam))

    def add_compliance_derivative(self, compb=1.0):
        """crm.py:282-293"""
        val = to_host(D.gemm_tn(self.Q, self.fr_d)).ravel()
        D.gemm_nn(self.fr_d.unsqueeze(1), small_to_dev((2.0 * compb * val / self.lam)[None, :]), self.Qb, alpha=1.0, beta=1.0)
        self.lamb -= compb * (val * val) / self.lam ** 2

    def _eigenvector_seeds(self):
        return self.Qb

    def _total_derivative(self, psi, corr_data):
        self.psi = psi
        grad = D.zeros(self.prob.ncomp)
        shard = self.sharding
        if shard is not None and shard.world > 1 and self.deriv_type == "vector":
            # the per-mode derivative calls shard by mode like the adjoint solves: this rank's modes, one all-reduce
            self.grad = _sharded_vector_derivative(self, psi, corr_data, shard)
        else:
            self.grad = add_eig_total_derivative(self.lam, self.Q, self.lamb, self.Qb, psi, self.prob.dAdx, self.prob.dBdx, grad,
                                                 adj_corr_data=corr_data, deriv_type=self.deriv_type)


def _sharded_vector_derivative(model, psi, corr_data, shard):
    """Per-mode ("vector") total derivative with the modes spread over the ranks: rank r evaluates the dA/dx, dB/dx
    inner products of modes r, r + world, ... and the (ncomp,) partial gradients meet in one all-reduce."""
    import torch.distributed as dist
    from .eigenvector_derivatives import _total_derivative_weights
    WA, WB, signB = _total_derivative_weights(model.lam, model.Q, model.lamb, model.Qb, psi, corr_data, "normal")
    grad = D.zeros(model.prob.ncomp)
    for i in shard.my_cols(model.N):
        qi = model.Q[:, i].contiguous()
        D.axpby(1.0, grad, 1.0, model.prob.dAdx.device_call(WA[:, i].contiguous(), qi), out=grad)
        D.axpby(1.0, grad, signB, model.prob.dBdx.device_call(WB[:, i].contiguous(), qi), out=grad)
    dist.all_reduce(grad, group=shard.group)
    return grad


def make_shell_model(nx=64, ny=64, ncx=8, ncy=8, Ls=1.0, Ly=1.0, radius=2.0, scale=100.0, material=None, **kwargs):
    """Cylindrical panel clamped along y = 0, ncx x ncy thickness components (crm-like: one DV per component).
    nx = ny = 408 gives 409^2 nodes x 6 = 1 003 686 DOF (BASELINE configs[3])."""
    conn, X, P = cylindrical_panel(nx, ny, Ls, Ly, radius)
    ei = np.arange(nx * ny) % nx
    ej = np.arange(nx * ny) // nx
    comp = (ei * ncx // nx) + ncx * (ej * ncy // ny)
    nodes = np.arange((nx + 1) * (ny + 1)).reshape(nx + 1, ny + 1)
    prob = ShellProblem(conn, X, comp, fixed_nodes=nodes[:, 0], order_coords=P, scale=scale, **(material or {}))
    return ShellModalAnalysis(prob, **kwargs)
