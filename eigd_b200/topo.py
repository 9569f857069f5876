"""Device-resident counterparts of the reference's example drivers (``TopologyAnalysis`` classes).

They keep the method names, the ``profile`` timer keys and the data flow of

  examples/thermal.py            :268-342 (solve_eigenvalue_problem), :344-372 (initialize /
                                 initialize_adjoint), :428-442 (thermal compliance), :560-623 (finalize_adjoint)
  examples/natural_frequency.py  :317-392, :394-440, :442-519 (three rigid-body modes computed and dropped)

but every array of length n or nelems lives in HBM between the stages: design x -> filter ->
element densities -> K, M values (gather-form assembly) -> shifted matrix -> numeric LDL^T ->
restarted Lanczos -> adjoint right-hand sides -> lock-step sibk -> fused sensitivity kernel ->
node gather -> filter transpose -> xb.  Host code only sequences kernels and does the small
dense algebra the reference also does on the host.
"""
import time

import numpy as np
import torch

from . import device as D
from . import fe
from ._hostdev import is_dev, like_input, small_to_dev, to_dev, to_host
from .eigenvector_derivatives import IRAM, BasicLanczos, SpLuOperator


def _now():
    torch.cuda.synchronize()
    return time.perf_counter()


class _EigenAnalysis:
    """Forward and reverse pipeline shared by the model drivers.

    A driver's forward pass assembles its pencil, analyses the pattern with ``_symbolic_once``, factors the shifted
    matrix into ``self.factor`` and runs ``_new_eig_solver`` and ``_eigensolve``.  Its reverse pass is
    ``finalize_adjoint`` here, with the driver's eigenvector seeds (``_eigenvector_seeds``) and total derivative
    (``_total_derivative``)."""

    def __init__(self, prob, N, m, solver_type, tol, rtol, eig_atol, adjoint_method, adjoint_options, deriv_type, seed,
                 fronts="resident"):
        self.prob = prob
        self.fronts = D.check_fronts(fronts)      # front memory of every factor the driver builds (SpLuOperator)
        self.N, self.m = N, m
        self.solver_type, self.tol, self.rtol, self.eig_atol = solver_type, tol, rtol, eig_atol
        if adjoint_method == "shift-invert":          # the examples' historical alias (thermal.py:37)
            adjoint_method = "sibk"
        self.adjoint_method = adjoint_method
        self.adjoint_options = dict(adjoint_options or {})
        self.deriv_type = deriv_type
        self.seed = seed              # IRAM start vector (deterministic: the eigensolve is replicated when sharded)
        self.Q = self.lam = None
        self.symbolic = None
        self.sharding = None          # dist.ModeSharding for the per-mode adjoint / element-range shards
        self.profile = {}

    # ---- forward ------------------------------------------------------------------------------
    def _symbolic_once(self, K):
        """Symbolic analysis of the pattern of ``self.prob``'s system matrix K, once per sparsity pattern.  Returns its
        time, or None when the analysis of an earlier call is reused."""
        if self.symbolic is not None:
            return None
        ts = _now()
        coords, dofpn = self.prob.dof_coords()
        sym = D.Symbolic(self.prob.indptr, self.prob.indices, K.shape[0], coords=coords, dof_per_node=dofpn)
        self.symbolic = (sym, sym.assembly_map_device(K.indptr, K.indices))
        self.profile["symbolic analysis time"] = dt = _now() - ts
        return dt

    def _new_eig_solver(self, N, iram=None, lanczos=None):
        """``self.eig_solver`` for N modes: IRAM or BasicLanczos by ``solver_type``, with the driver's own extra arguments
        of each (``iram``, ``lanczos``).  ``self.m`` gets its default on the first call and keeps it."""
        if self.solver_type == "IRAM":
            if self.m is None:
                self.m = max(2 * N + 1, 60)
            self.eig_solver = IRAM(N=N, m=self.m, eig_atol=self.eig_atol, **(iram or {}))
            self.eig_solver.seed = self.seed
        else:
            if self.m is None:
                self.m = max(3 * N + 1, 60)
            self.eig_solver = BasicLanczos(N=N, m=self.m, eig_atol=self.eig_atol, tol=self.tol, **(lanczos or {}))

    def _eigensolve(self, A, B, sigma, t1):
        """``self.eig_solver`` on the pencil (A, B) about ``sigma`` with ``self.factor``; the eigenvalue solve time runs
        from ``t1``.  Returns the eigenvalues."""
        self.factor.count = 0
        self.eig_solver.sharding = self.sharding
        lam, _ = self.eig_solver.solve(A, B, self.factor, sigma)
        t2 = _now()
        self.profile["solve preconditioner count"] = self.factor.count
        self.profile["eigenvalue solve time"] = t2 - t1
        self.profile["m"] = self.m
        self.profile["eig_solver.m"] = str(self.eig_solver.m)
        return lam

    # ---- reverse ------------------------------------------------------------------------------
    def finalize_adjoint(self):
        res_list = []
        self.factor.count = 0
        t0 = _now()
        psi, corr_data = self.eig_solver.solve_adjoint(self._eigenvector_seeds(), rtol=self.rtol, method=self.adjoint_method,
                                                       callback=res_list.append, **self.adjoint_options)
        t1 = _now()
        self.profile["adjoint preconditioner count"] = self.factor.count
        self.profile["adjoint solution time"] = t1 - t0
        self.profile["adjoint residuals"] = res_list
        self.profile["adjoint iterations"] = len(res_list)
        self.profile["adjoint correction data"] = corr_data
        self._total_derivative(psi, corr_data)
        self.profile["total derivative time"] = _now() - t1

    def time_to_gradient(self):
        p = self.profile
        return p["eigenvalue solve time"] + p["adjoint solution time"] + p["total derivative time"]


class _Q4Analysis(_EigenAnalysis):
    kind = "thermal"
    nrigid = 0            # leading modes computed but dropped (rigid-body modes of the free structure)

    def __init__(self, fltr, conn, X, sigma, N=10, m=None, Ntarget=None, solver_type="IRAM", tol=0.0, rtol=1e-10,
                 eig_atol=1e-5, adjoint_method="sibk", adjoint_options=None, deriv_type="tensor", seed=0, fronts="resident",
                 **material):
        self.fltr = fltr
        self.conn, self.X = np.asarray(conn), np.asarray(X)
        super().__init__(self._make_problem(**material), N, m, solver_type, tol, rtol, eig_atol, adjoint_method,
                         adjoint_options, deriv_type, seed, fronts)
        self.nelems, self.nnodes, self.nvars = self.prob.nelems, self.prob.nnodes, self.prob.ndof
        self.sigma, self.Ntarget = sigma, Ntarget
        self.x = 0.95 * np.ones(self.fltr.num_design_vars)      # thermal.py:71, natural_frequency.py:75
        self.profile.update(nnodes=self.nnodes, nelems=self.nelems, solver_type=solver_type,
                            adjoint_method=self.adjoint_method, N=N)

    def _make_problem(self, **material):
        return fe.Q4Problem(self.conn, self.X, self.kind, **material)

    def _rigid_count(self, lam0):
        """How many of the computed modes ``lam0`` (ascending) are rigid-body modes."""
        return self.nrigid

    def _keep_flexible(self, lam0):
        """``self.keep``: the modes the driver reports, len(lam0) - nrigid of them, after the rigid ones."""
        r = self._rigid_count(lam0)
        self.keep = slice(r, r + len(lam0) - self.nrigid)

    # ---- forward ------------------------------------------------------------------------------
    def solve_eigenvalue_problem(self, store=False):
        t0 = _now()
        K, M = self.prob.assemble()
        t1 = _now()
        self.profile["matrix assembly time"] = t1 - t0
        shifted = K.with_values(D.axpby(1.0, K.data, -float(self.sigma), M.data))    # K - sigma M on the shared pattern
        if self._symbolic_once(K) is not None:
            t1 = _now()                                                   # the eigensolve time excludes the analysis
        self.factor = SpLuOperator(shifted, symbolic=self.symbolic, fronts=self.fronts)
        self.K, self.M = K, M
        self._new_eig_solver(self.N + self.nrigid, iram=dict(tol=self.tol), lanczos=dict(Ntarget=self.Ntarget))
        self.prob.sharding = self.sharding
        lam = self._eigensolve(K, M, self.sigma, t1)
        self.lam0 = np.asarray(lam)
        self.Q0 = self.eig_solver._Phi_d                                   # (n, N + nrigid) device
        self._keep_flexible(self.lam0)
        return self.lam0[self.keep], self.Q0[:, self.keep]

    def initialize(self, store=False, x=None):
        if x is not None:
            self.x = x
        if not is_dev(self.x) and np.iscomplexobj(self.x):
            return self._initialize_dual(store)
        self.x_d = to_dev(self.x)
        self.rho = self.fltr.apply(self.x_d)
        self.rhoE = self.prob.set_density(rho=self.rho)
        self.lam, self.Q = self.solve_eigenvalue_problem(store)
        self.N = len(self.lam)
        return

    def _initialize_dual(self, store=False):
        """Complex design x + i h p (the complex-step check of the examples, thermal.py:652-661): the imaginary part is
        carried as a first-order tangent through the real fp64 kernels -- filter, material law, assembly, LDL^T, Lanczos
        (eigd_b200/dual.py) -- and ``lam`` / ``Q`` come back as complex host arrays (value + i tangent), which is what
        the reference's complex run returns.  As in the reference, only ``BasicLanczos`` supports it."""
        if self.solver_type == "IRAM":
            raise NotImplementedError("complex-step designs need solver_type='BasicLanczos' (as in the reference: ARPACK is real)")
        x = np.asarray(self.x)
        xr, xt = np.ascontiguousarray(x.real), np.ascontiguousarray(x.imag)
        self.x_d = to_dev(xr)
        self.rho = self.fltr.apply(self.x_d)
        rho_t = self.fltr.apply_tangent(self.x_d, to_dev(xt))
        self.rhoE = self.prob.set_density(rho=self.rho)
        K, M = self.prob.assemble()
        Kt, Mt = self.prob.assemble_tangent(rho_t)
        self._symbolic_once(K)
        shifted = K.with_values(D.axpby(1.0, K.data, -float(self.sigma), M.data))
        self.factor = SpLuOperator(shifted, symbolic=self.symbolic, fronts=self.fronts)
        self.factor.tangent = K.with_values(D.axpby(1.0, Kt.data, -float(self.sigma), Mt.data))
        self.factor.dtype = np.dtype(np.complex128)
        self.K, self.M = K, M
        self._new_eig_solver(self.N + self.nrigid, lanczos=dict(Ntarget=self.Ntarget))
        lam, Phi = self.eig_solver.solve((K, Kt), (M, Mt), self.factor, self.sigma)
        self.lam0, self.Q0 = np.asarray(lam), np.asarray(Phi)               # complex host arrays
        self._keep_flexible(self.lam0)
        self.lam, self.Q = self.lam0[self.keep], self.Q0[:, self.keep]
        self.N = len(self.lam)
        return

    def initialize_adjoint(self):
        self.xb = D.zeros(self.x_d.shape[0])
        self.rhoEb = D.zeros(self.nelems)
        self.lamb = np.zeros(self.N)
        self.Q0b = D.zeros(self.nvars, self.N + self.nrigid)
        self.Qb = self.Q0b[:, self.keep]

    # ---- reverse ------------------------------------------------------------------------------
    def _eigenvector_seeds(self):
        return self.Q0b

    def _total_derivative(self, psi0, corr_data):
        self.psi0 = psi0
        self.psi = psi0[:, self.keep]
        nr = self.keep.start
        if nr:                                                            # natural_frequency.py:484-494
            data0 = {}
            for i, items in corr_data.items():
                keep = [(j, xi, eta) for (j, xi, eta) in items if j >= nr]
                if i >= nr and keep:
                    data0[i] = keep
            corr_data = data0
        lamb0 = np.zeros(self.N + self.nrigid)
        lamb0[self.keep] = self.lamb
        self.eig_solver.add_total_derivative(lamb0, self.Q0b, psi0, self.prob.dAdx, self.prob.dBdx, self.rhoEb,
                                             adj_corr_data=corr_data, deriv_type=self.deriv_type)
        rhob = self.prob.scatter_to_nodes(self.rhoEb)
        g = self.fltr.apply_gradient(rhob, self.x_d)
        D.axpby(1.0, self.xb, 1.0, g, out=self.xb)


class ThermalTopologyAnalysis(_Q4Analysis):
    """examples/thermal.py ``ThermalTopologyAnalysis`` (scalar heat conduction, one zero mode)."""

    kind = "thermal"

    def __init__(self, fltr, conn, X, kappa=1.0, density=1.0, heat_capacity=1.0, p=3, beta=1e-6, sigma=-0.1, N=10,
                 **kw):
        super().__init__(fltr, conn, X, sigma, N=N, kappa=kappa, density=density, heat_capacity=heat_capacity,
                         p=float(p), beta=beta, **kw)

    def get_thermal_compliance(self, vec):
        """sum_{i>=1} (phi_i . vec)^2 / lam_i   (thermal.py:428-434)"""
        if not is_dev(self.Q):                      # dual-number mode: complex host eigenpairs, N-sized host algebra
            c = np.asarray(self.Q).T @ (to_host(vec) if is_dev(vec) else np.asarray(vec))
            return np.sum(c[1:] ** 2 / self.lam[1:])
        c = to_host(D.gemm_tn(self.Q, to_dev(vec))).ravel()
        return float(np.sum(c[1:] ** 2 / self.lam[1:]))

    def add_thermal_compliance_derivative(self, compb, vec):
        """thermal.py:436-442: Qb_i += 2 compb (phi_i . vec) vec / lam_i ; lamb_i -= compb (phi_i . vec)^2 / lam_i^2"""
        vec_d = to_dev(vec)
        c = to_host(D.gemm_tn(self.Q, vec_d)).ravel()
        coef = 2.0 * compb * c / self.lam
        coef[0] = 0.0
        D.gemm_nn(vec_d.unsqueeze(1), small_to_dev(coef[None, :]), self.Qb, alpha=1.0, beta=1.0)
        dl = compb * (c * c) / self.lam ** 2
        dl[0] = 0.0
        self.lamb -= dl


class ThermalTopology3DAnalysis(ThermalTopologyAnalysis):
    """The heat-conduction problem of ``ThermalTopologyAnalysis`` on a 3-D body of trilinear hexahedra
    (``fe.H8ThermalProblem``): same material law, shift sigma, forward and reverse pipeline, thermal compliance (mode 0,
    the constant temperature of the insulated body, is skipped) and dual-number designs."""

    def _make_problem(self, **material):
        return fe.H8ThermalProblem(self.conn, self.X, **material)


class ThermalTopologyTetAnalysis(ThermalTopologyAnalysis):
    """The heat-conduction problem of ``ThermalTopologyAnalysis`` on a 3-D body of quadratic tetrahedra
    (``fe.T10ThermalProblem``, conn (nelems, 10)): everything else as ``ThermalTopology3DAnalysis``."""

    def _make_problem(self, **material):
        return fe.T10ThermalProblem(self.conn, self.X, **material)


class NaturalFrequencyAnalysis(_Q4Analysis):
    """examples/natural_frequency.py ``TopologyAnalysis``: free plane-stress structure, N + 3 modes
    computed with sigma < 0 and the three rigid-body modes dropped (:348, :383-384, :457-458)."""

    kind = "plane_stress"
    nrigid = 3

    def __init__(self, fltr, conn, X, E=1.0, nu=0.3, density=1.0, p=3, rho0_K=1e-6, ptype_K="simp", q=5.0,
                 sigma=-10.0, N=6, **kw):
        super().__init__(fltr, conn, X, sigma, N=N, E=E, nu=nu, density=density, p=float(p), rho0_K=rho0_K,
                         ptype_K=ptype_K, q=q, **kw)

    # ---- objective helpers of examples/natural_frequency.py:521-563 -------------------------------------
    def get_frequencies(self):
        return np.sqrt(np.asarray(self.lam))

    def add_frequency_derivatives(self, omegab):
        """lamb_i += omegab_i / (2 sqrt(lam_i))   (:524-529)"""
        self.lamb += 0.5 * np.asarray(omegab) / np.sqrt(np.asarray(self.lam))

    def _set_rows(self, name):
        if name not in self.node_sets:
            raise ValueError("Unrecognized point name")
        nodes = np.asarray(self.node_sets[name], dtype=np.int64)
        key = ("rows", name)
        if key not in self.__dict__.setdefault("_cache", {}):
            self._cache[key] = (torch.as_tensor(2 * nodes, device=D.dev()), torch.as_tensor(2 * nodes + 1, device=D.dev()))
        return nodes, self._cache[key]

    def get_point_coefficients(self, name):
        """Mean position of a node set and the mean modal displacement over it, (3, N) (:531-551)."""
        nodes, (rx, ry) = self._set_rows(name)
        weight = 1.0 / len(nodes)
        x0 = np.zeros(3)
        x0[0], x0[1] = weight * np.sum(self.X[nodes, 0]), weight * np.sum(self.X[nodes, 1])
        xcoef = None
        if self.Q is not None:
            xcoef = np.zeros((3, self.N))
            xcoef[0] = weight * to_host(self.Q.index_select(0, rx).sum(dim=0))
            xcoef[1] = weight * to_host(self.Q.index_select(0, ry).sum(dim=0))
        return x0, xcoef

    def add_point_derivative(self, name, x0b, xcoefb):
        """Qb[2 nodes, i] += w xcoefb[0, i], Qb[2 nodes + 1, i] += w xcoefb[1, i]   (:553-563)"""
        if xcoefb is None:
            return
        nodes, (rx, ry) = self._set_rows(name)
        weight = 1.0 / len(nodes)
        self.Qb.index_add_(0, rx, small_to_dev(weight * np.asarray(xcoefb)[0][None, :]).expand(len(nodes), self.N).contiguous())
        self.Qb.index_add_(0, ry, small_to_dev(weight * np.asarray(xcoefb)[1][None, :]).expand(len(nodes), self.N).contiguous())

    def add_modal_function_derivative(self, w):
        """Seed of a smooth function f = sum_i (phi_i . w_i)^2 of the flexible modes (used by the tests and
        the bench; the KS minimum-frequency objective of the example is host-side numpy)."""
        w_d = to_dev(w)
        val = to_host(D.col_dot(self.Q, w_d))
        D.col_axpy(self.Qb, small_to_dev(2.0 * val), w_d, sign=1.0)
        return float(np.sum(val**2))


class NaturalFrequency3DAnalysis(NaturalFrequencyAnalysis):
    """The natural-frequency problem of ``NaturalFrequencyAnalysis`` on a free 3-D solid of trilinear hexahedra
    (``fe.H8Problem``): N + 6 modes computed with sigma < 0 and the six rigid-body modes (three translations, three
    rotations) dropped.  Same forward and reverse pipeline and objective helpers; the 2-D node-set helpers are not
    offered."""

    nrigid = 6

    def _make_problem(self, **material):
        return fe.H8Problem(self.conn, self.X, **material)

    def _rigid_count(self, lam0):
        """The leading modes with lambda ~ 0.  IRAM returns all six copies of the six-fold zero eigenvalue; single-vector
        Lanczos (BasicLanczos) resolves only some of them from one start vector, and the rest of its N + 6 Ritz pairs
        are flexible modes, so the rigid ones are counted by value, not assumed."""
        lam = np.abs(np.asarray(lam0).real)
        return int(min(self.nrigid, np.count_nonzero(lam < 1e-8 * lam.max())))

    def get_point_coefficients(self, name):
        raise NotImplementedError("node-set point coefficients are defined for the 2-D model only")

    def add_point_derivative(self, name, x0b, xcoefb):
        raise NotImplementedError("node-set point derivatives are defined for the 2-D model only")


class NaturalFrequencyTetAnalysis(NaturalFrequency3DAnalysis):
    """The natural-frequency problem of ``NaturalFrequency3DAnalysis`` on a free 3-D solid of quadratic tetrahedra
    (``fe.T10Problem``, conn (nelems, 10)): six rigid-body modes dropped, same pipeline and objective helpers."""

    def _make_problem(self, **material):
        return fe.T10Problem(self.conn, self.X, **material)


class MinFreqOpt:
    """KS-aggregated minimum natural frequency of the structure with a point mass attached at each node set in turn
    (examples/natural_frequency.py ``MinFreqOpt`` :693-803).  For node set s with modal coefficients c (3 x N) the
    frequencies of structure + mass are those of the N x N pencil (diag(omega^2), I + m c^T c); the objective is the
    soft minimum (KS, parameter ks_param) over all sets and modes.  Only N x N host algebra: the n-sized work is the
    eigensolve and the adjoint of ``topo``."""

    def __init__(self, topo, ks_param=1.0, fixed_mass=1.0):
        if isinstance(topo, NaturalFrequency3DAnalysis):
            raise ValueError("MinFreqOpt attaches point masses to the node sets of the 2-D model; it is not offered for "
                             "the 3-D solid")
        self.topo, self.ks_param, self.fixed_mass = topo, ks_param, fixed_mass
        self.ks_min = 0.0
        self.node_sets = topo.node_sets
        self.coef, self.coefb, self.omega, self.omegab = {}, {}, None, None

    def initialize(self, store=False):
        self.topo.initialize(store)
        self.omega = self.topo.get_frequencies()
        self.coef = {name: self.topo.get_point_coefficients(name)[1] for name in self.node_sets}
        self.ks_min, self.omegab, self.coefb = self._eval_min_frequency(self.omega, self.coef, self.ks_param, self.fixed_mass)

    def initialize_adjoint(self):
        self.topo.initialize_adjoint()

    def finalize_adjoint(self):
        self.topo.add_frequency_derivatives(self.omegab)
        for name in self.node_sets:
            self.topo.add_point_derivative(name, None, self.coefb[name])
        self.topo.finalize_adjoint()

    def get_min_frequency(self):
        return self.ks_min

    @staticmethod
    def _soft_min(vals, p):
        lo = np.min(vals)
        e = np.exp(-p * (vals - lo))
        return lo - np.log(np.sum(e)) / p, e / np.sum(e)

    def _eval_min_frequency(self, omega, xcoef, ks_param=30.0, fixed_mass=1.0):
        from scipy.linalg import eigh
        N = len(omega)
        names = list(xcoef)
        pencil = {}
        inner = {}
        for name in names:
            c0 = xcoef[name]
            lam0, Q0 = eigh(np.diag(omega ** 2), np.eye(N) + fixed_mass * (c0.T @ c0))
            om0 = np.sqrt(lam0)
            pencil[name] = (om0, Q0)
            inner[name] = self._soft_min(om0, ks_param)                      # (KS of this set, weights over its modes)
        # outer soft minimum over the sets, anchored at min(omega, KS values) as the reference does (:757-768)
        vals = np.array([inner[name][0] for name in names])
        anchor = min(np.min(omega), np.min(vals)) if len(vals) else np.min(omega)
        e = np.exp(-ks_param * (vals - anchor))
        ks = anchor - np.log(np.sum(e)) / ks_param
        wset = e / np.sum(e)
        omegab = np.zeros(N)
        xcoefb = {}
        for name, ws in zip(names, wset):
            c0 = xcoef[name]
            om0, Q0 = pencil[name]
            wb = 0.5 * inner[name][1] * ws / om0                             # d ks / d lam0_i
            omegab += 2.0 * omega * np.einsum("ik,k,ik->i", Q0, wb, Q0)      # through K0 = diag(omega^2)
            # through M0 = I + m c^T c:  d lam0_i = -lam0_i q_i^T dM0 q_i
            sc = 2.0 * wb * fixed_mass * om0 ** 2
            xcoefb[name] = -(c0 @ Q0) * sc[None, :] @ Q0.T
        return ks, omegab, xcoefb


def make_thermal_model(nx=128, ny=128, Lx=1.0, Ly=1.0, rfact=4.0, **kwargs):
    """examples/thermal.py ``make_model`` (:1475-1509)."""
    conn, X = fe.grid_mesh(nx, ny, Lx, Ly)
    fltr = fe.NodeFilter(conn, X, r0=rfact * (Ly / ny))
    return ThermalTopologyAnalysis(fltr, conn, X, **kwargs)


def make_thermal_3d_model(nx=80, ny=64, nz=48, Lx=1.0, Ly=0.8, Lz=0.6, rfact=4.0, ftype="spatial", **kwargs):
    """Insulated nx x ny x nz hexahedral box (``fe.hex_mesh``) of ``ThermalTopology3DAnalysis``, one design variable per
    node, filter of radius rfact * Ly / ny (the radius of ``make_thermal_model``): conic (``ftype="spatial"``) or
    Helmholtz (``"helmholtz"``, one scalar LDL^T of the mesh instead of the conic filter's pair search and CSR
    operators).  The box is not a cube: a cube, or any box with two equal sides, has repeated eigenvalues at a uniform
    design, where eigenvector derivatives are undefined.  With sides 1 : 0.8 : 0.6 the first 14 eigenvalues of the
    continuous Neumann Laplacian, pi^2 (i^2 + j^2 / 0.64 + k^2 / 0.36) = pi^2 (0, 1, 1.5625, 2.5625, 2.778, 3.778, 4,
    4.34, ...), are simple.  The default 80 x 64 x 48 box has 257 985 DOF, the size of the 2-D bench grid (251 001);
    ``fronts="pooled"`` (forwarded through ``kwargs``) factors it in a 2.3 GB pool instead of 17 GB of resident
    fronts."""
    conn, X = fe.hex_mesh(nx, ny, nz, Lx, Ly, Lz)
    fltr = fe.NodeFilter(conn, X, r0=rfact * (Ly / ny), ftype=ftype)
    return ThermalTopology3DAnalysis(fltr, conn, X, **kwargs)


def make_thermal_tet_model(nx=40, ny=32, nz=24, Lx=1.0, Ly=0.8, Lz=0.6, rfact=4.0, ftype="spatial", **kwargs):
    """Insulated box of nx x ny x nz cubes, 6 quadratic tetrahedra each (``fe.tet10_mesh``), of
    ``ThermalTopologyTetAnalysis``, one design variable per node.  Its nodes are those of
    ``make_thermal_3d_model(2 nx, 2 ny, 2 nz)``: the default has the 257 985 DOF of the H8 default, and the filter
    radius, rfact times the node spacing Ly / (2 ny), is the H8 model's on the same lattice.  Conic
    (``ftype="spatial"``) or Helmholtz (``"helmholtz"``) filter; ``fronts=`` and the solver options go to the driver."""
    conn, X = fe.tet10_mesh(nx, ny, nz, Lx, Ly, Lz)
    fltr = fe.NodeFilter(conn, X, r0=rfact * (Ly / (2 * ny)), ftype=ftype)
    return ThermalTopologyTetAnalysis(fltr, conn, X, **kwargs)


def natural_frequency_design_map(nx, ny, rfact=4.0, Mx=3, My=3, ns=2):
    """Design-variable map, node sets and element sets of examples/natural_frequency.py ``make_model`` (:896-954):
    Mx x My patches of non-design material (dvmap = -1, the filter treats them as x = 1) and a four-fold mirror
    symmetry of the remaining nodes.  Same visiting order as the reference, so the design-variable numbering is
    bit-identical (checked against the reference's own ``fltr.dvmap`` in tests/test_fullsize_golden_gpu.py)."""
    nodes = np.arange((nx + 1) * (ny + 1), dtype=np.int64).reshape(nx + 1, ny + 1)
    dvmap = np.zeros((nx + 1, ny + 1), dtype=np.int64)
    node_sets, element_sets = {}, {}
    ns = max(int(ns * ny // 32), int(rfact // 2))
    sx, sy = nx // (Mx - 1), ny // (My - 1)
    for i in range(Mx):
        for j in range(My):
            if i < Mx // 2:
                imin, imax = max(0, sx * i - ns + 1), min(nx, sx * i + ns + 1)
            else:
                lo, hi = max(0, sx * (Mx - i - 1) - ns + 1), min(nx, sx * (Mx - i - 1) + ns + 1)
                imin, imax = max(0, nx - hi), min(nx, nx - lo)
            if j < My // 2:
                jmin, jmax = max(0, sy * j - ns), min(ny, sy * j + ns)
            else:
                lo, hi = max(0, sy * (My - j - 1) - ns), min(ny, sy * (My - j - 1) + ns)
                jmin, jmax = max(0, ny - hi), min(ny, ny - lo)
            ii, jj = np.meshgrid(np.arange(imin, imax), np.arange(jmin, jmax), indexing="ij")
            name = "node[%d,%d]" % (i, j)
            node_sets[name] = nodes[ii, jj].ravel()
            element_sets[name] = (ii + nx * jj).ravel()
            dvmap[imin:imax, jmin:jmax] = -1
    index = 0
    for i in range(nx // 2 + 1):
        js = np.nonzero(dvmap[i, : ny // 2 + 1] >= 0)[0]         # ascending j, as the reference's inner loop (:945-951)
        ids = index + np.arange(len(js))
        for a in (i, nx - i):
            dvmap[a, js] = ids
            dvmap[a, ny - js] = ids
        index += len(js)
    return dvmap.ravel(), index, node_sets, element_sets


def make_natural_frequency_model(nx=128, ny=64, Lx=1.0, Ly=1.0, rfact=4.0, N=10, Mx=3, My=3, ns=2, symmetry=True,
                                 projection=False, b0=None, **kwargs):
    """examples/natural_frequency.py ``make_model`` (:850-976), including its symmetric design-variable map and the
    non-design patches (``symmetry=False``: one design variable per node)."""
    conn, X = fe.grid_mesh(nx, ny, Lx, Ly)
    if symmetry:
        dvmap, ndv, node_sets, element_sets = natural_frequency_design_map(nx, ny, rfact, Mx, My, ns)
        fltr = fe.NodeFilter(conn, X, r0=rfact * (Ly / ny), dvmap=dvmap, num_design_vars=ndv, projection=bool(projection),
                             beta=b0)
    else:
        node_sets, element_sets = {}, {}
        fltr = fe.NodeFilter(conn, X, r0=rfact * (Ly / ny), projection=bool(projection), beta=b0)
    model = NaturalFrequencyAnalysis(fltr, conn, X, N=N, **kwargs)
    model.node_sets, model.element_sets = node_sets, element_sets
    return model


def make_natural_frequency_3d_model(nx, ny, nz, Lx=2.0, Ly=1.0, Lz=1.0, rfact=4.0, **kwargs):
    """Free nx x ny x nz hexahedral box (``fe.hex_mesh``), one design variable per node, conic filter of radius
    rfact * Ly / ny on the 3-D nodes.  With the default resident fronts the largest box one 180 GB B200 factors is
    about 80 x 40 x 40 (408k DOF); ``fronts="pooled"`` (forwarded through ``kwargs``) borrows a lifetime-ordered front
    pool per factorisation instead, which takes 96 x 48 x 48 (699k DOF) (DESIGN.md section 8b)."""
    conn, X = fe.hex_mesh(nx, ny, nz, Lx, Ly, Lz)
    fltr = fe.NodeFilter(conn, X, r0=rfact * (Ly / ny))
    return NaturalFrequency3DAnalysis(fltr, conn, X, **kwargs)


def make_natural_frequency_tet_model(nx=32, ny=16, nz=16, Lx=2.0, Ly=1.0, Lz=1.0, rfact=4.0, **kwargs):
    """Free box of nx x ny x nz cubes, 6 quadratic tetrahedra each (``fe.tet10_mesh``), of
    ``NaturalFrequencyTetAnalysis``, one design variable per node, conic filter of radius rfact times the node spacing
    Ly / (2 ny).  Its nodes are those of ``make_natural_frequency_3d_model(2 nx, 2 ny, 2 nz)``: the default has the
    212 355 DOF of the H8 64 x 32 x 32 box and the same filter radius.  ``fronts=`` and the solver options go to the
    driver."""
    conn, X = fe.tet10_mesh(nx, ny, nz, Lx, Ly, Lz)
    fltr = fe.NodeFilter(conn, X, r0=rfact * (Ly / (2 * ny)))
    return NaturalFrequencyTetAnalysis(fltr, conn, X, **kwargs)


# ------------------------------------------------------------------------------------------
# linearised buckling -- examples/buckling.py
# ------------------------------------------------------------------------------------------
class BucklingTopologyAnalysis(_EigenAnalysis):
    """examples/buckling.py ``TopologyAnalysis`` (:19-118): (K + BLF * G(u)) phi = 0 on the reduced dofs, with
    the fundamental path K_r u_r = f_r, shift-invert about ``sigma`` (mode="buckling": A = G_r, B = K_r,
    factor of K_r + sigma G_r, :548-640), and the gradient of an eigenvector functional including the
    fundamental-path adjoint (:896-982).  Every vector of length n, 2*nnodes or nelems stays in HBM.
    ``pivoting`` (not in the reference) is the pivot strategy of the shifted factor K_r + sigma G_r (SpLuOperator);
    the fundamental-path factor of K_r is SPD and always static."""

    def __init__(self, fltr, conn, X, bcs, forces={}, E=1.0, nu=0.3, ptype_K="simp", ptype_M="simp", ptype_G="simp",
                 rho0_K=1e-6, rho0_M=1e-9, rho0_G=1e-9, p=3.0, q=5.0, density=1.0, sigma=3.0, N=10, m=None,
                 solver_type="IRAM", tol=0.0, rtol=1e-10, eig_atol=1e-5, adjoint_method="shift-invert",
                 adjoint_options=None, cost=1, deriv_type="tensor", seed=0, pivoting="static", fronts="resident"):
        self.fltr = fltr
        self.pivoting = pivoting          # of the shifted factor K_r + sigma G_r (SpLuOperator); K_r alone is SPD
        self.conn, self.X = np.asarray(conn), np.asarray(X)
        prob = self._make_problem(bcs, forces, E=E, nu=nu, density=density, p=float(p), q=float(q), rho0_K=rho0_K,
                                  rho0_G=rho0_G, ptype_K=ptype_K.lower(), ptype_G=ptype_G.lower())
        super().__init__(prob, N, m, solver_type, tol, rtol, eig_atol, adjoint_method, adjoint_options, deriv_type, seed,
                         fronts)
        self.nelems, self.nnodes, self.nvars = self.prob.nelems, self.prob.nnodes, self.prob.ndof
        self.reduced, self.f = self.prob.reduced, self.prob.f
        self.E, self.nu, self.p, self.q, self.density = E, nu, p, q, density
        self.rho0_K, self.rho0_G = rho0_K, rho0_G
        self.sigma, self.cost = sigma, cost
        self.x = 0.5 * np.ones(self.fltr.num_design_vars)                 # buckling.py:81
        self.profile.update(nnodes=self.nnodes, nelems=self.nelems, solver_type=solver_type,
                            adjoint_method=self.adjoint_method, N=N)

    def _make_problem(self, bcs, forces, **material):
        return fe.BucklingQ4Problem(self.conn, self.X, bcs, forces, **material)

    # ---- forward (:548-640, 811-838) ----------------------------------------------------------------
    def solve_eigenvalue_problem(self, store=False):
        t0 = _now()
        Kr = self.prob.assemble_K()
        t0 += self._symbolic_once(Kr) or 0.0                              # the assembly time excludes the analysis
        self.Kfact = SpLuOperator(Kr, symbolic=self.symbolic, max_rhs=1, fronts=self.fronts)  # fundamental path K_r u_r = f_r
        ur = self.Kfact.solve_dev(self.prob.fr_d)
        self.u_d = self.prob.set_displacement(ur)
        Gr = self.prob.assemble_G()
        t1 = _now()
        self.profile["matrix assembly time"] = t1 - t0
        vals = D.axpby(1.0, Kr.data, float(self.sigma), Gr.data)          # K_r + sigma G_r on the shared pattern
        self.factor = SpLuOperator(Kr.with_values(vals), symbolic=self.symbolic, pivoting=self.pivoting, fronts=self.fronts)
        self.Kr, self.Gr = Kr, Gr
        self._new_eig_solver(self.N, iram=dict(mode="buckling"), lanczos=dict(mode="buckling"))
        if self.solver_type == "IRAM":
            self.eig_solver.reference_pairing = getattr(self, "reference_pairing", False)
            self.eig_solver.block_size = getattr(self, "block_size", None)
        mu = self._eigensolve(Gr, Kr, self.sigma, t1)
        self.BLF = np.asarray(mu)[: self.N]
        self.Qr = self.eig_solver._Phi_d                                   # (n_r, N) device
        return self.BLF, self.Qr

    def initialize(self, store=False, x=None):
        if x is not None:
            self.x = x
        self.x_d = to_dev(self.x)
        self.rho = self.fltr.apply(self.x_d)
        self.rhoE = self.prob.set_density(rho=self.rho)
        self.lam, self.Qr = self.solve_eigenvalue_problem(store)
        return

    @property
    def u(self):
        return to_host(self.u_d)

    def compliance(self):
        return float(np.dot(self.f, self.u))

    def initialize_adjoint(self):
        self.xb = D.zeros(self.x_d.shape[0])
        self.rhoEb = D.zeros(self.nelems)
        self.lamb = np.zeros(self.N)
        self.Qrb = D.zeros(self.prob.nred, self.N)

    # ---- objectives (:702-760) ----------------------------------------------------------------------
    def _aggregate_weights(self, rho, mode):
        lam = np.asarray(self.lam)
        if mode == "exp":
            eta = np.exp(-rho * (lam - np.min(lam)))
            a = b = None
        else:
            a = np.tanh(rho * (lam - 0.0))
            b = np.tanh(rho * (lam - 50.0))
            eta = a - b
        return eta / np.sum(eta), a, b

    def get_eigenvector_aggregate(self, rho, node, mode="tanh"):
        """h = sum_i eta_i Q[node, i]^2 (:702-724); as in the reference ``node`` indexes the FULL dof vector."""
        eta, _, _ = self._aggregate_weights(rho, mode)
        qn = self._dof_values(node)
        return float(np.sum(eta * qn * qn))

    def _dof_values(self, dof):
        f2r = np.full(self.nvars, -1, dtype=np.int64)
        f2r[self.reduced] = np.arange(len(self.reduced))
        r = int(f2r[dof])
        self._dof_row = r
        return to_host(self.Qr[r]) if r >= 0 else np.zeros(self.N)

    def add_eigenvector_aggregate_derivative(self, hb, rho, node, mode="tanh"):
        """Seeds of h = sum_i eta_i Q[node, i]^2 (:726-760): Qrb[row(node), i] += 2 hb eta_i Q[node, i] and
        lamb_i -= hb rho eta_i (a_i + b_i) (Q[node, i]^2 - h)."""
        eta, a, b = self._aggregate_weights(rho, mode)
        qn = self._dof_values(node)
        h = float(np.sum(eta * qn * qn))
        if self._dof_row >= 0:
            row = self.Qrb[self._dof_row]
            row += small_to_dev(2.0 * hb * eta * qn)
        if mode == "exp":
            self.lamb -= hb * rho * eta * (qn * qn - h)
        else:
            self.lamb -= hb * rho * eta * (a + b) * (qn * qn - h)
        return h

    def eval_ks_buckling(self, ks_rho=160.0):
        """KS maximum of mu_i = 1 / BLF_i (:641-646)."""
        mu = 1.0 / np.asarray(self.BLF)
        c = np.max(mu)
        return float(c + np.log(np.sum(np.exp(ks_rho * (mu - c)))) / ks_rho)

    def eval_ks_buckling_derivative(self, ks_rho=160.0):
        """Design gradient of ``eval_ks_buckling`` (:648-700, tensor form): eigenvalue sensitivities only (no eigenvector
        adjoint), with the fundamental-path adjoint K_r a_r = -(dG/du)_r.  Everything stays in HBM; returns the
        gradient in the flavour of ``self.x``."""
        t0 = _now()
        pr = self.prob
        mu = 1.0 / np.asarray(self.BLF)
        eta = np.exp(ks_rho * (mu - np.max(mu)))
        eta /= np.sum(eta)
        Q = self.Qr
        etaQ = Q.clone()
        D.col_scale(etaQ, small_to_dev(eta), mode=0)
        etamuQ = Q.clone()
        D.col_scale(etamuQ, small_to_dev(eta * mu), mode=0)
        dKdx = pr.dKdx.device_call(etamuQ, Q)                               # per element
        dGdu = pr.dGdu.device_call(etaQ, Q)                                 # full dof vector
        adj_r = self.Kfact.solve_dev(pr.reduce_vector(dGdu))
        adj = pr.full_vector(adj_r)                                         # = -adjoint of the reference (:689-690)
        dGdx = pr.dGdx.device_call(etaQ, Q)
        dfde = D.axpby(-1.0, dGdx, -1.0, dKdx)                              # -(dGdx + dKdx) ...
        D.axpby(1.0, dfde, 1.0, pr.dK_single(adj, self.u_d), out=dfde)      # ... - dK(adj_ref, u) = + dK(adj, u)
        dfdrho = pr.scatter_to_nodes(dfde)
        g = self.fltr.apply_gradient(dfdrho, self.x_d)
        self.profile["total derivative time"] = self.profile.get("total derivative time", 0.0) + (_now() - t0)
        return like_input(g, self.x)

    # ---- reverse (:866-982) -------------------------------------------------------------------------
    def _eigenvector_seeds(self):
        return self.Qrb

    def _total_derivative(self, psir, corr_data):
        self.psir = psir
        pr = self.prob
        # d/du of the eigen-terms: dfdu0 = sum_i w_i^T (dG/du) phi_i  (dB/du = 0: K does not depend on u)
        dfdu0 = D.zeros(self.nvars)
        self.eig_solver.add_total_derivative(self.lamb, self.Qrb, psir, pr.dGdu, None, dfdu0, adj_corr_data=corr_data,
                                             deriv_type=self.deriv_type)
        # explicit design dependence of G and K
        self.eig_solver.add_total_derivative(self.lamb, self.Qrb, psir, pr.dGdx, pr.dKdx, self.rhoEb,
                                             adj_corr_data=corr_data, deriv_type=self.deriv_type)
        # adjoint of the fundamental path: K_r psi_u = -dfdu0_r, rhob += psi_u^T (dK/drho) u   (:974-979)
        psiu_r = self.Kfact.solve_dev(pr.reduce_vector(dfdu0))
        psiu = pr.full_vector(psiu_r)
        D.axpby(1.0, self.rhoEb, -1.0, pr.dK_single(psiu, self.u_d), out=self.rhoEb)
        self.rhob = pr.scatter_to_nodes(self.rhoEb)
        g = self.fltr.apply_gradient(self.rhob, self.x_d)
        D.axpby(1.0, self.xb, 1.0, g, out=self.xb)


def domain_compressed_column(nx=64, ny=128, Lx=1.0, Ly=2.0, shear_force=False):
    """examples/buckling.py ``domain_compressed_column`` (:1300-1369), vectorised: mesh, left-right symmetry map
    of the design variables, clamped bottom edge, compressive (or shear) load on the top edge."""
    conn, X = fe.grid_mesh(nx, ny, Lx, Ly)
    nodes = np.arange((nx + 1) * (ny + 1), dtype=np.int64).reshape(nx + 1, ny + 1)
    dvmap = np.zeros((nx + 1, ny + 1), dtype=np.int64)
    index = 0
    for i in range(nx // 2 + 1):                      # same visiting order as the reference (:1336-1341)
        dvmap[i, :] = index + np.arange(ny + 1)
        dvmap[nx - i, :] = dvmap[i, :]
        index += ny + 1
    bcs = {int(nodes[i, 0]): [0, 1] for i in range(nx + 1)}
    P = 1e-3
    forces = {}
    if shear_force:
        for i in range(nx + 1):
            forces[int(nodes[i, ny])] = [P / (nx + 1), 0]
    else:
        offset = int(np.ceil(nx / 30))
        for i in range(offset):
            forces[int(nodes[nx // 2 - i - 1, ny])] = [0, -P / (2 * offset + 1)]
            forces[int(nodes[nx // 2 + i + 1, ny])] = [0, -P / (2 * offset + 1)]
        forces[int(nodes[nx // 2, ny])] = [0, -P / (2 * offset + 1)]
    return conn, X, dvmap.flatten(), index, bcs, forces


def make_buckling_model(nx=64, ny=128, Lx=1.0, Ly=2.0, rfact=4.0, N=10, shear_force=False, **kwargs):
    """examples/buckling.py ``make_model`` (:1372-1409)."""
    conn, X, dvmap, ndv, bcs, forces = domain_compressed_column(nx=nx, ny=ny, Lx=Lx, Ly=Ly, shear_force=shear_force)
    fltr = fe.NodeFilter(conn, X, r0=rfact * (Lx / nx), dvmap=dvmap, num_design_vars=ndv)
    return BucklingTopologyAnalysis(fltr, conn, X, bcs=bcs, forces=forces, N=N, **kwargs)


class BucklingTopology3DAnalysis(BucklingTopologyAnalysis):
    """The linearised buckling problem of ``BucklingTopologyAnalysis`` on a 3-D solid of trilinear hexahedra
    (``fe.BucklingH8Problem``), with the same forward and reverse pipeline and objectives.

    Each design keeps two factors on one symbolic analysis, K_r (for the fundamental-path adjoint) and K_r + sigma G_r.
    With resident fronts (the default) each keeps its own front workspace; the previous design's factors, and the
    eigensolver that references them, are dropped before the next design is factored, so the peak is two front
    workspaces rather than three.  With ``fronts="pooled"`` neither keeps fronts: both factorisations borrow one
    lifetime-ordered pool in turn."""

    def _make_problem(self, bcs, forces, **material):
        return fe.BucklingH8Problem(self.conn, self.X, bcs, forces, **material)

    def solve_eigenvalue_problem(self, store=False):
        self.factor = self.Kfact = self.eig_solver = None
        return super().solve_eigenvalue_problem(store)


def domain_compressed_column_3d(nx, ny, nz, Lx, Ly, Lz):
    """Column along z on ``fe.hex_mesh(nx, ny, nz, Lx, Ly, Lz)``, the 3-D counterpart of ``domain_compressed_column``:
    base face (z = 0) clamped, a compressive load P = 3e-4 in -z spread evenly over a central patch of the top face of
    (2 ceil(nx / 30) + 1) x (2 ceil(ny / 30) + 1) nodes.  Returns conn, X, bcs {node: [0, 1, 2]} and forces
    {node: [0, 0, -P / patch nodes]}."""
    conn, X = fe.hex_mesh(nx, ny, nz, Lx, Ly, Lz)
    nodes = np.arange((nx + 1) * (ny + 1) * (nz + 1), dtype=np.int64).reshape(nx + 1, ny + 1, nz + 1)
    bcs = {int(v): [0, 1, 2] for v in nodes[:, :, 0].ravel()}
    P = 3e-4
    ox, oy = int(np.ceil(nx / 30)), int(np.ceil(ny / 30))
    patch = nodes[nx // 2 - ox:nx // 2 + ox + 1, ny // 2 - oy:ny // 2 + oy + 1, nz].ravel()
    forces = {int(v): [0.0, 0.0, -P / len(patch)] for v in patch}
    return conn, X, bcs, forces


def make_buckling_3d_model(nx=32, ny=24, nz=128, Lx=1.0, Ly=0.75, Lz=4.0, rfact=4.0, N=10, **kwargs):
    """``domain_compressed_column_3d`` with one design variable per node and a conic filter of radius rfact * Lx / nx.
    The default cross-section is rectangular: a square column has pairs of equal buckling loads, where eigenvector
    derivatives are undefined.  The load makes the first load factors O(1): on a coarse 4 x 3 x 16 mesh at x = 0.5 the
    Euler modes about the weak and strong axes are at about 2.4 and 4.0; finer meshes add modes near the loaded patch
    from about 2.5 up (32 x 24 x 128, x ~ U(0.3, 0.7): 8 load factors below 3).  The default sigma = 3 lies inside
    the spectrum, so K_r + sigma G_r is indefinite.  As in the 2-D driver the eigensolver returns the N load factors
    nearest sigma in the buckling shift-invert transform, which ranks a lambda < sigma below every lambda > sigma
    when lambda < sigma / 2.  At 32 x 24 x 128 each factor's resident fronts take 44 GB (DESIGN.md section 8b);
    ``fronts="pooled"`` (forwarded through ``kwargs``) replaces them by one shared pool."""
    conn, X, bcs, forces = domain_compressed_column_3d(nx, ny, nz, Lx, Ly, Lz)
    fltr = fe.NodeFilter(conn, X, r0=rfact * (Lx / nx))
    return BucklingTopology3DAnalysis(fltr, conn, X, bcs=bcs, forces=forces, N=N, **kwargs)
