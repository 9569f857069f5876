"""B200-native mirror of reference ``eigd/eigenvector_derivatives.py`` (smdogroup/eigd).

Same public names, argument meaning and error behaviour as the reference (file:line cited on
every routine); every floating-point operation on n-length data is one of the hand-written
sm_100a kernels of ``libeigd_b200.so`` reached through ``eigd_b200.device``.  numpy arrays in
give numpy arrays out (the reference's convention); CUDA torch tensors / ``device.CsrDevice``
in give device tensors out and skip the host<->device copies.  The only host arithmetic is the
reference's own "small" algebra: m x m ``eigh`` of the projected operator, (j+1) x j least
squares of the Krylov solvers, N x N adjoint-correction scalars.  There is no CPU fallback.

Structural differences from the reference (results are the same):
  * ``SpLuOperator`` is a supernodal multifrontal LDL^T of the (symmetric) shifted matrix on the
    GPU instead of SuperLU's LU; ``factor(X)`` solves all columns of X at once.
  * ``sibk`` / ``pcpg`` / ``pgmres`` run the N per-mode Krylov processes in lock step (one
    N-column solve and SpMM per iteration).  With ``update_guess=False`` the modes are
    uncoupled (reference :1189-1217), so every mode sees exactly the reference's recurrence.
  * ``IRAM`` uses the thick-restart Lanczos of ``eigd_b200.arpack`` (see there).
"""
import warnings

import numpy as np
import torch

from . import device as D
from ._hostdev import XFER, as_csr_device, is_dev, like_input, small_to_dev, to_dev, to_host
from .arpack import eigsh_mod

__all__ = ["SpLuOperator", "add_eig_total_derivative", "eval_adjoint_residual_norm", "are_eigenvalues_repeated",
           "generate_adjoint_correction", "laa", "dl", "pcpg", "pgmres", "sibk", "BasicLanczos", "IRAM"]

_SYMBOLIC_CACHE = {}


def _public(fn):
    """Public entry point: uploads issued straight from the caller's page-locked arrays are awaited before control
    returns to the caller (device.drain_uploads), whatever path the call takes."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        try:
            return fn(*args, **kwargs)
        finally:
            D.drain_uploads()
    return wrapper


def _is_complex_host(M):
    """scipy sparse matrix with complex values (a complex-step operand); device matrices are always real"""
    d = getattr(M, "data", None)
    return isinstance(d, np.ndarray) and np.iscomplexobj(d)


def _check_symmetric_sampled(mat, nsample=64):
    """The reference's ``splu`` takes any square matrix; the LDL^T here needs a symmetric one, and a CSC operand is
    read as the CSR arrays of its transpose.  A full symmetry test costs more than the factorisation's upload, so
    compare ``nsample`` rows / columns entry by entry (structure and values) and refuse anything else."""
    if mat.format not in ("csr", "csc") or mat.shape[0] != mat.shape[1] or mat.nnz == 0:
        return
    n = mat.shape[0]
    if not mat.has_sorted_indices:
        mat.sort_indices()
    ptr, idx, val = mat.indptr, mat.indices, mat.data
    major = np.unique(np.linspace(0, n - 1, min(nsample, n)).astype(np.int64))
    cnt = np.minimum(ptr[major + 1] - ptr[major], 16).astype(np.int64)
    j = np.repeat(major, cnt)                                           # sampled entries (i, j) of the compressed axis
    pos = np.repeat(ptr[major].astype(np.int64) - np.concatenate([[0], np.cumsum(cnt)[:-1]]), cnt) + np.arange(int(cnt.sum()))
    i, v = idx[pos].astype(np.int64), val[pos]
    lo, hi = ptr[i].astype(np.int64), ptr[i + 1].astype(np.int64)        # vectorised bisection for j in segment i
    for _ in range(int(np.ceil(np.log2(max(int((hi - lo).max()), 2)))) + 1):
        mid = (lo + hi) // 2
        less = (mid < hi) & (idx[np.minimum(mid, len(idx) - 1)] < j)
        lo, hi = np.where(less, mid + 1, lo), np.where(less, hi, mid)
    q = np.minimum(lo, len(idx) - 1)
    # assembled FE matrices are symmetric only up to the rounding of their COO sums (K + sigma G of
    # examples/buckling.py differs by ~1e-10 of its largest entry across the diagonal): reject real asymmetry only
    scale = max(float(np.abs(v).max()), float(np.abs(val[::97]).max())) or 1.0
    found = (lo < ptr[i + 1]) & (idx[q] == j)          # scipy's sparse sums prune exact zeros: a missing mirror entry is 0.0
    bad = np.abs(np.where(found, val[q], 0.0) - v) > 1e-6 * scale
    if bad.any():
        k = int(np.argmax(bad))
        raise ValueError("SpLuOperator: the matrix is not symmetric (entry (%d, %d)); the GPU factorisation is an "
                         "LDL^T of a symmetric shifted matrix" % (i[k], j[k]))


def _check_mode(mode):
    if mode not in ("normal", "buckling"):
        raise ValueError(f"Unknown mode {mode!r}")


# ------------------------------------------------------------------------------------------
# factor wrapper -- reference eigd/eigenvector_derivatives.py:11-23
# ------------------------------------------------------------------------------------------
class SpLuOperator:
    """``(A - sigma B)^{-1}`` (or ``(B + sigma A)^{-1}``) as a GPU LDL^T factorisation.

    Reference: ``SpLuOperator`` (:11-23) wraps ``scipy.sparse.linalg.splu``; attributes ``lu``,
    ``shape``, ``dtype`` and the per-column solve counter ``count`` (:16-22) are kept.  ``mat``
    must be structurally and numerically symmetric (it is ``K - sigma*M`` / ``Kr + sigma*Gr`` in
    every caller: examples/natural_frequency.py:338-340, examples/buckling.py:582-584); a scipy
    CSC or CSR matrix, or a ``device.CsrDevice`` whose values already live in HBM.

    Extra keyword arguments (not in the reference): ``coords`` / ``dof_per_node`` enable geometric
    nested dissection, ``symbolic`` reuses an analysis, ``refine`` sets the number of iterative
    refinement steps per solve (default: 1 if the factorisation met negative or perturbed pivots),
    ``pivoting`` chooses the pivot strategy of the LDL^T: ``"static"`` (default: no pivot search, a pivot below
    1e-11 max|A| is perturbed to +-that threshold and the solves are refined) or ``"bunch-kaufman"`` (restricted
    Bunch-Kaufman 1x1 / 2x2 pivoting inside every 32-column pivot block: for indefinite shifts with zero or tiny
    diagonal entries, e.g. saddle-point operators or a shift close to an eigenvalue).  ``info`` reports the pivot
    statistics either way; the probe / refinement policy is the same for both.  ``fronts`` chooses the memory of the
    factorisation's dense fronts (``device.Factor``): ``"resident"`` (default) keeps them in the factor,
    ``"pooled"`` borrows a much smaller lifetime-ordered pool for each factorisation only; the factor is the same.
    """

    @_public
    def __init__(self, mat, coords=None, dof_per_node=1, symbolic=None, refine=None, max_rhs=32, pivoting="static",
                 fronts="resident"):
        if pivoting not in D.PIVOTING_MODES:
            raise ValueError("SpLuOperator: pivoting must be one of %s, not %r" % (D.PIVOTING_MODES, pivoting))
        D.check_fronts(fronts, "SpLuOperator: fronts")
        self.tangent = None
        if isinstance(mat, D.CsrDevice):
            csr = mat
        else:
            if not hasattr(mat, "tocsr"):
                raise TypeError("SpLuOperator needs a scipy sparse matrix or a device.CsrDevice")
            self.tangent = None
            if np.iscomplexobj(mat.data):
                # complex-step operand: factor the real part, keep the imaginary part as the tangent matrix (dual.py)
                from . import dual
                csr, self.tangent = dual.split_csr(mat, symmetric=True)
                XFER["h2d"] += 2 * csr.uploaded_bytes
            else:
                _check_symmetric_sampled(mat)
                csr = D.CsrDevice.from_scipy(mat, symmetric=True)   # symmetric: CSC arrays of mat are CSR arrays of mat
                XFER["h2d"] += csr.uploaded_bytes
        if csr.shape[0] != csr.shape[1]:
            raise ValueError("expected square matrix")
        self.shape = csr.shape
        self.dtype = np.dtype(np.complex128 if self.tangent is not None else np.float64)
        self.count = 0
        self.mat = csr
        n = csr.shape[0]
        if symbolic is None:
            extra = "geo%d" % dof_per_node if coords is not None else "graph"
            pid = getattr(csr, "pattern_id", None)
            host = getattr(csr, "pattern_host", None)
            if host is None:
                host = (to_host(csr.indptr), to_host(csr.indices))
            key = (pid, extra) if pid is not None else D.pattern_key(host[0], host[1], extra.encode())
            cached = _SYMBOLIC_CACHE.get(key)
            if cached is None:
                sym = D.Symbolic(host[0], host[1], n, coords=coords, dof_per_node=dof_per_node)
                amap = sym.assembly_map_device(csr.indptr, csr.indices)
                if len(_SYMBOLIC_CACHE) > 8:
                    _SYMBOLIC_CACHE.clear()
                _SYMBOLIC_CACHE[key] = cached = (sym, amap)
            symbolic = cached
        elif isinstance(symbolic, D.Symbolic):
            symbolic = (symbolic, symbolic.assembly_map_device(csr.indptr, csr.indices))
        self.symbolic, self._amap = symbolic
        self.lu = D.Factor(self.symbolic, max_rhs=max_rhs, pivoting=pivoting, fronts=fronts).numeric(csr.data, self._amap)
        # The factorisation is now queued on the device.  Its pivot statistics (inertia, perturbed pivots) and the choice
        # of the refinement depth need a read-back, i.e. a wait for the whole factorisation: that is deferred to the first
        # use (``info`` / ``refine`` / the first solve), so that the caller's next host-side steps -- typically the
        # upload and verification of K and M in ``solve`` -- overlap with it instead of idling behind it.
        self._refine_request = refine
        self._state = None

    def _finish(self):
        if self._state is not None:
            return
        self._state = {"info": None, "probe": None, "probe_refined": None}
        st = self._state
        st["info"] = info = self.lu.info()
        if info["non_finite"]:
            raise RuntimeError("SpLuOperator: non-finite pivots in the LDL^T factorisation (singular shifted matrix?)")
        refine = self._refine_request
        if refine is None:
            if info["perturbed_pivots"]:
                refine = 1
            elif info["negative_pivots"]:
                # indefinite but unperturbed (e.g. K + sigma G above the first buckling load): LDL^T without
                # pivoting may or may not have lost accuracy -- measure it once on a probe right-hand side and keep
                # the refinement step unless the plain solve is already at rounding level.  (Measured at C3: probe
                # 3e-11; dropping the refinement inside the adjoint Krylov solvers alone moved the gradient norm by
                # 5e-4 relative -- the modes next to the shift amplify the operator error -- so it stays.)
                st["probe"] = self._probe_residual()
                refine = 0 if st["probe"] < 1e-13 else 1
            else:
                refine = 0
        self.lu.set_refinement(refine, self.mat)
        if self.lu.refine and (info["perturbed_pivots"] or info["negative_pivots"]):
            # static pivoting is only as good as the refined solve it leaves behind: measure that, iterate the
            # refinement to tolerance if one step is not enough, and say so loudly if it cannot be reached
            # (a shift that sits on an eigenvalue; the reference's partially pivoted LU would lose accuracy there too)
            st["probe_refined"] = self._probe_residual(refined=True)
            while st["probe_refined"] > 1e-10 and self.lu.refine < 4:
                self.lu.set_refinement(self.lu.refine + 1, self.mat)
                st["probe_refined"] = self._probe_residual(refined=True)
            if not st["probe_refined"] <= 1e-8:
                warnings.warn("SpLuOperator: the LDL^T factorisation of the shifted matrix is inaccurate (relative residual "
                              "%.1e after %d refinement steps, %d perturbed and %d negative pivots); move the shift away "
                              "from the spectrum" % (st["probe_refined"], self.lu.refine, info["perturbed_pivots"],
                                                     info["negative_pivots"]))

    @property
    def info(self):
        self._finish()
        return self._state["info"]

    @property
    def refine(self):
        self._finish()
        return self.lu.refine

    @refine.setter
    def refine(self, value):
        self._finish()
        self.lu.set_refinement(value, self.mat)

    @property
    def probe(self):
        self._finish()
        return self._state["probe"]

    @property
    def probe_refined(self):
        self._finish()
        return self._state["probe_refined"]

    def _probe_residual(self, refined=False):
        """max |b - mat x| / max |b| of one solve (plain LDL^T sweep, or the refined solve every caller gets) with a
        fixed pseudo-random right-hand side."""
        n = self.shape[0]
        g = torch.Generator(device=D.dev())
        g.manual_seed(12345)
        b = torch.rand(n, dtype=D.F64, device=D.dev(), generator=g) - 0.5
        if refined:
            c0 = self.count
            x = self.solve_dev(b)
            self.count = c0
        else:
            x = self.lu.solve(b)
        r = self.mat.spmm(x)
        D.axpby(1.0, b, -1.0, r, out=r)
        return float((r.abs().max() / b.abs().max()).item())

    # -- device entry point used by every solver in this package --------------------------------
    def solve_dev(self, Bd, out=None):
        """X = mat^{-1} B for a device (n,) or (n, k) tensor; counts k solves (reference :19-22)."""
        self._finish()                               # settles the refinement depth the factor applies
        self.count += 1 if Bd.dim() == 1 else Bd.shape[1]
        return self.lu.solve(Bd, out=out, refined=True)

    @_public
    def _apply(self, x):
        if is_dev(x):
            return self.solve_dev(x)
        x = np.asarray(x)
        if x.shape[0] != self.shape[0] or x.ndim > 2:
            raise ValueError("dimension mismatch")
        if self.tangent is not None or np.iscomplexobj(x):
            # dual solve: A y = b, A dy = db - dA y (the imaginary parts are forward derivatives, dual.py)
            xr = to_dev(np.ascontiguousarray(x.real))
            yr = self.solve_dev(xr)
            rhs = to_dev(np.ascontiguousarray(x.imag)) if np.iscomplexobj(x) else D.zeros(*x.shape)
            if self.tangent is not None:
                t = self.tangent.spmm(yr)
                D.axpby(1.0, _contig(rhs).reshape(-1), -1.0, t.reshape(-1), out=t.reshape(-1))
                rhs = t
            self.count -= 1 if x.ndim == 1 else x.shape[1]
            return to_host(yr) + 1j * to_host(self.solve_dev(rhs))
        return to_host(self.solve_dev(to_dev(x)))

    __call__ = _apply
    matvec = _apply
    matmat = _apply
    dot = _apply
    __matmul__ = _apply

    def solve(self, x):
        return self._apply(x)


def _project(U, V, X):
    """X <- X - U (V^T X), device tensors (reference ``_project`` :26-30)."""
    return D.project(U, V, X)


def _apply_L(Ad, Bd, lam_d, X, mode, out=None):
    """L X with L_i = A - lam_i B (normal) or B + lam_i A (buckling); reference :262-265."""
    if mode == "normal":
        R = Ad.spmm(X, out=out)
        T = Bd.spmm(X)
        D.col_axpy(R, lam_d, T, sign=-1.0)
    else:
        R = Bd.spmm(X, out=out)
        T = Ad.spmm(X)
        D.col_axpy(R, lam_d, T, sign=1.0)
    return R


def _neg_sum(Phib, LX):
    """-Phib - LX (flat, both (n, N) row-major contiguous)."""
    out = torch.empty_like(LX)
    D.axpby(-1.0, Phib.reshape(-1), -1.0, LX.reshape(-1), out=out.reshape(-1))
    return out


def _contig(t):
    return t if t.is_contiguous() else t.contiguous()


def _col_norms(X):
    return np.sqrt(to_host(D.col_dot(X, X)))


# ------------------------------------------------------------------------------------------
# total derivative -- reference :33-182
# ------------------------------------------------------------------------------------------
def _corr_matrices(N, adj_corr_data):
    Cxi, Ceta = np.zeros((N, N)), np.zeros((N, N))
    for i, items in (adj_corr_data or {}).items():
        for j, xi, eta in items:
            Cxi[j, i] += xi
            Ceta[j, i] += eta
    return Cxi, Ceta


def _total_derivative_weights(lam, Phi_d, lamb, Phib_d, psi_d, adj_corr_data, mode):
    """Device (n, N) weights of the tensor form (reference :135-180).  Returns WA, WB, signB."""
    N = Phi_d.shape[1]
    lam = np.asarray(lam, dtype=float)
    lamb = np.asarray(lamb, dtype=float)
    beta = 0.5 * to_host(D.col_dot(Phi_d, Phib_d))
    Cxi, Ceta = _corr_matrices(N, adj_corr_data)
    if mode == "normal":
        # WA_i = lamb_i phi_i + psi_i + sum xi phi_j ; WB_i = (beta_i + lam_i lamb_i) phi_i + lam_i psi_i + sum eta phi_j
        SA = np.diag(lamb) + Cxi
        SB = np.diag(beta + lam * lamb) + Ceta
        WA = psi_d.clone()
        WB = psi_d.clone()
        D.col_scale(WB, small_to_dev(lam), mode=0)
        signB = -1.0
    else:
        # WA_i = lam_i (lamb_i phi_i + psi_i) + sum eta phi_j ; WB_i = (lamb_i - beta_i) phi_i + psi_i + sum xi phi_j
        SA = np.diag(lam * lamb) + Ceta
        SB = np.diag(lamb - beta) + Cxi
        WA = psi_d.clone()
        D.col_scale(WA, small_to_dev(lam), mode=0)
        WB = psi_d.clone()
        signB = 1.0
    D.gemm_nn(Phi_d, small_to_dev(SA), WA, alpha=1.0, beta=1.0)
    D.gemm_nn(Phi_d, small_to_dev(SB), WB, alpha=1.0, beta=1.0)
    return WA, WB, signB


def _call_deriv(fn, W_d, V_d, host):
    """Invoke a dAdx / dBdx callback.  Device operators (``device_call``) take HBM tensors."""
    if hasattr(fn, "device_call"):
        return fn.device_call(W_d, V_d)
    return fn(to_host(W_d), to_host(V_d))


@_public
def add_eig_total_derivative(lam, Phi, lamb, Phib, psi, dAdx, dBdx, dfdx, adj_corr_data={}, mode="normal",
                             deriv_type="vector"):
    """Reference ``add_eig_total_derivative`` (:33-182): dfdx += sum_i w_i^T (dA/dx) phi_i -/+ ...

    ``dAdx`` / ``dBdx`` are the reference's callbacks ``f(w, v)`` (either may be None).  Objects with
    a ``device_call(W, V)`` method (``eigd_b200.fe``) are evaluated in HBM without copying W and
    Phi back; plain Python callbacks receive numpy arrays as in the reference.  If both callbacks
    are the two halves of one ``fe`` sensitivity object they are evaluated by a single fused kernel.
    """
    n, N = Phi.shape[0], Phi.shape[1]
    _check_mode(mode)
    if len(lam) != N:
        raise ValueError(f"Eigenvalues must be of length {N}")
    if tuple(psi.shape) != (n, N):
        raise ValueError(f"Eigenvectors must have the shape ({n},{N})")
    if tuple(Phi.shape) != (n, N):
        raise ValueError(f"Eigenvectors must have the shape ({n},{N})")
    if tuple(Phib.shape) != (n, N):
        raise ValueError(f"Right-hand-side must have the shape ({n},{N})")
    if deriv_type not in ("vector", "tensor"):
        raise ValueError(f"Unknown deriv_type {deriv_type!r}")
    lam_h = to_host(lam) if is_dev(lam) else np.asarray(lam, dtype=float)
    lamb_h = to_host(lamb) if is_dev(lamb) else np.asarray(lamb, dtype=float)
    Phi_d, Phib_d, psi_d = to_dev(Phi), to_dev(Phib), to_dev(psi)
    WA, WB, signB = _total_derivative_weights(lam_h, Phi_d, lamb_h, Phib_d, psi_d, adj_corr_data, mode)

    def accumulate(val, sign):
        if is_dev(dfdx):
            v = val if is_dev(val) else to_dev(val)
            D.axpby(1.0, dfdx.reshape(-1), sign, _contig(v).reshape(-1), out=dfdx.reshape(-1))
        else:
            v = to_host(val) if is_dev(val) else val
            if sign > 0:
                dfdx[...] += v
            else:
                dfdx[...] -= v

    fused = getattr(dAdx, "fused_with", None)
    if deriv_type == "tensor" and fused is not None and fused is dBdx and dAdx is not None:
        accumulate(dAdx.parent.device_call_fused(WA, WB, Phi_d, 1.0, signB), 1.0)
        return dfdx
    if deriv_type == "tensor":
        if dAdx is not None:
            accumulate(_call_deriv(dAdx, WA, Phi_d, not is_dev(dfdx)), 1.0)
        if dBdx is not None:
            accumulate(_call_deriv(dBdx, WB, Phi_d, not is_dev(dfdx)), signB)
    else:
        for i in range(N):
            if dAdx is not None:
                accumulate(_call_deriv(dAdx, _contig(WA[:, i]), _contig(Phi_d[:, i]), True), 1.0)
            if dBdx is not None:
                accumulate(_call_deriv(dBdx, _contig(WB[:, i]), _contig(Phi_d[:, i]), True), signB)
    return dfdx


# ------------------------------------------------------------------------------------------
# residual check -- reference :185-275
# ------------------------------------------------------------------------------------------
@_public
def eval_adjoint_residual_norm(A, B, lam, Phi, Phib, psi, mode="normal", b_ortho=False):
    """Reference :185-275: ||L_i psi_i - b_i||_2 and the B-orthogonality defect, per mode."""
    n, N = A.shape[1], Phi.shape[1]
    if len(lam) != N:
        raise ValueError(f"Eigenvalues must be of length {N}")
    if A.shape != (n, n):
        raise ValueError(f"A must have dimensions ({n},{n})")
    if B.shape != (n, n):
        raise ValueError(f"B must have dimensions ({n},{n})")
    if tuple(psi.shape) != (n, N):
        raise ValueError(f"Eigenvectors must have the shape ({n},{N})")
    if tuple(Phi.shape) != (n, N):
        raise ValueError(f"Eigenvectors must have the shape ({n},{N})")
    if tuple(Phib.shape) != (n, N):
        raise ValueError(f"Right-hand-side must have the shape ({n},{N})")
    _check_mode(mode)
    Ad, Bd = as_csr_device(A), as_csr_device(B)
    Phi_d, Phib_d, psi_d = to_dev(Phi), to_dev(Phib), to_dev(psi)
    lam_d = small_to_dev(to_host(lam) if is_dev(lam) else lam)
    BPhi = Bd.spmm(Phi_d)
    # r = L psi + Phib - BPhi_i (phi_i . Phib_i)
    R = _apply_L(Ad, Bd, lam_d, psi_d, mode)
    D.axpby(1.0, R.reshape(-1), 1.0, _contig(Phib_d).reshape(-1), out=R.reshape(-1))
    c = D.col_dot(Phi_d, Phib_d)
    D.col_axpy(R, c, BPhi, sign=-1.0)
    if b_ortho:
        _project(BPhi, Phi_d, R)
        ortho = np.abs(to_host(D.gemm_tn(BPhi, psi_d))).max(axis=0)
    else:
        ortho = np.abs(to_host(D.col_dot(BPhi, psi_d)))
    return _col_norms(R), ortho


def _is_close(a, b, atol=1e-5):
    return bool(np.fabs(a - b) < atol)


def are_eigenvalues_repeated(lam, atol=1e-5):
    """Reference :284-300 (expects ascending eigenvalues)."""
    lam = to_host(lam) if is_dev(lam) else np.asarray(lam)
    return any(_is_close(lam[i], lam[i + 1], atol=atol) for i in range(len(lam) - 1))


# ------------------------------------------------------------------------------------------
# adjoint correction -- reference :303-391
# ------------------------------------------------------------------------------------------
def _correction_coeffs(lam, G, eig_atol, mode):
    """N x N coefficient matrix C (psi += Phi C) and the repeated-pair data (reference :362-391)."""
    N = len(lam)
    G0 = G if mode == "normal" else np.diag(lam) @ G
    C = np.zeros((N, N))
    data = {}
    for i in range(N):
        for j in range(i):
            dlam = lam[j] - lam[i]
            if _is_close(lam[i], lam[j], eig_atol):
                with np.errstate(divide="ignore", invalid="ignore"):
                    xi = 0.5 * (G0[j, i] - G0[i, j]) / dlam
                    eta = 0.5 * (lam[i] * G0[j, i] - lam[j] * G0[i, j]) / dlam
                data.setdefault(i, []).append((j, xi, eta))
                data.setdefault(j, []).append((i, xi, eta))
            else:
                C[j, i] += G0[j, i] / dlam           # psi_i += G0[j,i]/(lam_j - lam_i) phi_j
                C[i, j] += G0[i, j] / (-dlam)        # psi_j += G0[i,j]/(lam_i - lam_j) phi_i
    return C, data


def _apply_correction_dev(lam, Phi_d, psi_d, G, eig_atol, mode):
    C, data = _correction_coeffs(np.asarray(lam, dtype=float), np.asarray(G, dtype=float), eig_atol, mode)
    if np.any(C):
        D.gemm_nn(Phi_d, small_to_dev(C), psi_d, alpha=1.0, beta=1.0)
    return data


@_public
def generate_adjoint_correction(lam, Phi, psi, G=None, Phib=None, eig_atol=1e-5, mode="normal"):
    """Reference :303-391.  ``psi`` is corrected in place; returns the repeated-eigenvalue data."""
    _check_mode(mode)
    n, N = Phi.shape[0], len(lam)
    if G is None:
        if tuple(Phi.shape) != (n, N):
            raise ValueError(f"Eigenvectors must have the shape ({n},{N})")
        if Phib is None or tuple(Phib.shape) != (n, N):
            raise ValueError(f"Right-hand-side must have the shape ({n},{N})")
        if tuple(psi.shape) != (n, N):
            raise ValueError(f"Eigenvector adjoint must have the shape ({n},{N})")
    else:
        if tuple(G.shape) != (N, N):
            raise ValueError(f"G must have dimensions ({N},{N})")
        if tuple(Phi.shape) != (n, N):
            raise ValueError(f"Phi must have dimensions ({n},{N})")
    lam_h = to_host(lam) if is_dev(lam) else np.asarray(lam, dtype=float)
    Phi_d = to_dev(Phi)
    if G is None:
        G = -to_host(D.gemm_tn(Phi_d, to_dev(Phib)))
    elif is_dev(G):
        G = to_host(G)
    psi_d = to_dev(psi)
    data = _apply_correction_dev(lam_h, Phi_d, psi_d, G, eig_atol, mode)
    if not is_dev(psi):
        psi[...] = to_host(psi_d)
    return data


# ------------------------------------------------------------------------------------------
# Lanczos adjoint approximation -- reference :394-523
# ------------------------------------------------------------------------------------------
def _basis_dev(V):
    """Krylov basis as a logical (n, m) device tensor (vector-major storage kept if given)."""
    if is_dev(V):
        return V
    return to_dev(np.ascontiguousarray(np.asarray(V).T)).T


def _laa_dev(Phib_d, Bd, factor, sigma, lam, V_d, Y, theta, indices, b_ortho, mode, cols=None, Nfull=None):
    """``cols`` / ``Nfull``: Phib_d and lam hold only the modes ``cols`` out of ``Nfull`` (mode sharding)."""
    m, N = len(theta), Phib_d.shape[1]
    Yb = to_host(D.gemm_tn(V_d, Phib_d))                      # (m, N) = V^T Phib   (:502)
    Dm = np.zeros((m, N))
    Nfull = N if Nfull is None else Nfull
    first = indices[:Nfull] if cols is None else indices[np.asarray(cols)]
    if cols is not None and not b_ortho:
        raise NotImplementedError("column subsets are only used with b_ortho=True")
    if b_ortho:
        rest = indices[Nfull:]
        Dm[rest, :] = (Y[:, rest].T @ Yb) / (theta[first][None, :] - theta[rest][:, None])   # (:503-508)
    else:
        for j in range(N):
            for i in range(m):
                ii, jj = indices[i], indices[j]
                if ii != jj:
                    Dm[ii, j] = (Y[:, ii] @ Yb[:, j]) / (theta[jj] - theta[ii])
    S = Y @ (Dm / (np.asarray(lam) - sigma))
    S *= -1.0 if mode == "normal" else -sigma                 # (:519-521)
    X = D.empty(Phib_d.shape[0], N)
    D.gemm_nn(V_d, small_to_dev(S), X, alpha=1.0, beta=0.0)
    return factor.solve_dev(Bd.spmm(X))


@_public
def laa(Phib, B, factor, sigma, lam, V, Y, theta, indices, D0=None, b_ortho=False, mode="normal"):
    """Reference ``laa`` (:394-523): Galerkin solution of the adjoint equations in span(V)."""
    _check_mode(mode)
    n, N, m = Phib.shape[0], Phib.shape[1], len(theta)
    if len(lam) != N:
        raise ValueError(f"Eigenvalues must be of length {N}")
    if tuple(Phib.shape) != (n, N):
        raise ValueError(f"Right-hand-side must have the shape ({n},{N})")
    if B.shape != (n, n):
        raise ValueError(f"B must have dimensions ({n},{n})")
    if factor.shape != (n, n):
        raise ValueError(f"Factorized operator must have dimensions ({n},{n})")
    if len(indices) != m:
        raise ValueError(f"Length of indices array must be (m = {m})")
    if tuple(V.shape) != (n, m):
        raise ValueError(f"Dimension of the Lanczos subspace must be ({n},{m})")
    if D0 is not None:
        raise NotImplementedError("the D0 branch of the reference (:492-500) uses D before assignment and cannot run")
    lam_h = to_host(lam) if is_dev(lam) else np.asarray(lam, dtype=float)
    psi = _laa_dev(to_dev(Phib), as_csr_device(B), factor, sigma, lam_h, _basis_dev(V), np.asarray(Y),
                   np.asarray(theta), np.asarray(indices), b_ortho, mode)
    return like_input(psi, Phib)


# ------------------------------------------------------------------------------------------
# differentiated Lanczos -- reference :526-696
# ------------------------------------------------------------------------------------------
def _dl_dev(Phib_d, Bd, factor, sigma, lam, Phi_d, indices, V_d, T, Y, theta, eig_atol, mode):
    n, N, m = Phib_d.shape[0], Phib_d.shape[1], len(theta)
    repeated = are_eigenvalues_repeated(lam, eig_atol)
    first = indices[:N]
    G = BPhi = None
    R = Phib_d
    if repeated:
        BPhi = Bd.spmm(Phi_d)
        G = -to_host(D.gemm_tn(Phi_d, Phib_d))
        R = Phib_d.clone()
        D.gemm_nn(BPhi, small_to_dev(G), R, alpha=1.0, beta=1.0)
    # Vb stored vector-major (m, n): row j is the reverse-mode seed of Lanczos vector j
    Vbt = D.empty(m, n)
    Vb = Vbt.T
    D.gemm_nn(R, small_to_dev(np.ascontiguousarray(Y[:, first].T)), Vb, alpha=1.0, beta=0.0)    # Vb = R Y0^T (:616)
    Yb = to_host(D.gemm_tn(V_d, R))
    Dm = np.zeros((m, m))
    for i in range(m):
        for j in range(N):
            ii, jj = indices[i], indices[j]
            if ii == jj or (i < N and _is_close(lam[i], lam[j], eig_atol)):
                continue
            Dm[ii, jj] = (Y[:, ii] @ Yb[:, j]) / (theta[jj] - theta[ii])
    Tb = Y @ (Dm @ Y.T)
    col = lambda M, j: M[:, j]                                           # noqa: E731  logical column views
    one = lambda v: small_to_dev(np.atleast_1d(v))                       # noqa: E731
    t = Bd.spmm(factor.solve_dev(Bd.spmm(_contig(col(V_d, m - 1)))))
    D.gemm_nn(t.unsqueeze(1), small_to_dev(Tb[:m, m - 1][None, :]), Vb, alpha=1.0, beta=1.0)      # Vb[:, j] += Tb[j, m-1] t
    x = D.empty(n)
    D.gemm_nn(V_d, small_to_dev(Tb[:, m - 1][:, None]), x, alpha=1.0, beta=0.0)
    u = factor.solve_dev(Bd.spmm(x))
    D.col_axpy(Vbt[m - 1], one(1.0), Bd.spmm(u))
    for i in range(m - 2, -1, -1):
        lo = max(i - 1, 0)
        D.gemm_nn(V_d[:, lo:i + 2], small_to_dev(T[lo:i + 2, i][:, None]), x, alpha=1.0, beta=0.0)
        t = Bd.spmm(x)
        c0 = float(to_host(D.col_dot(_contig(col(V_d, i + 1)), Vbt[i + 1]))[0]) - T[i + 1, i] * Tb[i + 1, i]
        sb = Vbt[i + 1].clone()
        D.col_axpy(sb, one(c0), Bd.spmm(_contig(col(V_d, i + 1))), sign=-1.0)
        D.col_scale(sb, one(T[i + 1, i]), mode=1)
        if i > 0:
            D.col_axpy(Vbt[i - 1], one(T[i - 1, i]), sb, sign=-1.0)
        D.col_axpy(Vbt[i], one(T[i, i]), sb, sign=-1.0)
        hb = to_host(D.gemm_tn(V_d[:, :i + 1], sb)).ravel() - Tb[:i + 1, i]
        D.gemm_nn(t.unsqueeze(1), small_to_dev(hb[None, :]), Vb[:, :i + 1], alpha=-1.0, beta=1.0)
        D.gemm_nn(V_d[:, :i + 1], small_to_dev(hb[:, None]), x, alpha=1.0, beta=0.0)
        D.col_axpy(sb, one(1.0), Bd.spmm(x), sign=-1.0)
        Vbt[i + 1].copy_(u)
        u = factor.solve_dev(sb)
        D.col_axpy(Vbt[i], one(1.0), Bd.spmm(u))
    Vbt[0].copy_(u)
    S = Y[:, first] / (np.asarray(lam) - sigma)
    S *= -1.0 if mode == "normal" else -sigma
    psi = D.empty(n, N)
    D.gemm_nn(Vb, small_to_dev(S), psi, alpha=1.0, beta=0.0)
    data = {}
    if repeated:
        _project(Phi_d, BPhi, psi)
        data = _apply_correction_dev(lam, Phi_d, psi, G, eig_atol, mode)
    return psi, data


@_public
def dl(Phib, B, factor, sigma, lam, Phi, indices, V, T, Y, theta, eig_atol=1e-5, mode="normal"):
    """Reference ``dl`` (:526-696): reverse-mode differentiation of the un-restarted Lanczos recurrence."""
    _check_mode(mode)
    n, N, m = Phib.shape[0], Phib.shape[1], len(theta)
    if len(lam) != N:
        raise ValueError(f"Eigenvalues must be of length {N}")
    if tuple(Phib.shape) != (n, N):
        raise ValueError(f"Right-hand-side must have the shape ({n},{N})")
    if B.shape != (n, n):
        raise ValueError(f"B must have dimensions ({n},{n})")
    if factor.shape != (n, n):
        raise ValueError(f"Factorized operator must have dimensions ({n},{n})")
    if len(indices) != m:
        raise ValueError(f"Length of indices array must be (m = {m})")
    if tuple(V.shape) != (n, m):
        raise ValueError(f"Dimension of the Lanczos subspace must be ({n},{m})")
    lam_h = to_host(lam) if is_dev(lam) else np.asarray(lam, dtype=float)
    psi, data = _dl_dev(to_dev(Phib), as_csr_device(B), factor, sigma, lam_h, to_dev(Phi), np.asarray(indices),
                        _basis_dev(V), np.asarray(T), np.asarray(Y), np.asarray(theta), eig_atol, mode)
    return like_input(psi, Phib), data


# ------------------------------------------------------------------------------------------
# lock-step per-mode Krylov solvers -- reference pcpg :699-869, pgmres :872-1040, sibk :1052-1328
# ------------------------------------------------------------------------------------------
def _check_krylov_args(Phib, A, B, lam, Phi, psi, mode):
    _check_mode(mode)
    n, N = Phib.shape[0], Phib.shape[1]
    if len(lam) != N:
        raise ValueError(f"Eigenvalues must be of length {N}")
    if A.shape != (n, n):
        raise ValueError(f"A must have dimensions ({n},{n})")
    if B.shape != (n, n):
        raise ValueError(f"B must have dimensions ({n},{n})")
    if psi is not None and tuple(psi.shape) != (n, N):
        raise ValueError(f"Initial guess must have the shape ({n},{N})")
    if tuple(Phi.shape) != (n, N):
        raise ValueError(f"Eigenvectors must have the shape ({n},{N})")
    if tuple(Phib.shape) != (n, N):
        raise ValueError(f"Right-hand-side must have the shape ({n},{N})")
    return n, N


def _default_factor(A, B, sigma, mode, factor, lam=None):
    if factor is not None:
        if not hasattr(factor, "solve_dev"):
            raise TypeError("factor must be an eigd_b200.SpLuOperator (there is no CPU solve to fall back on)")
        return factor
    if sigma is None:
        sigma = 0.9 * float(lam[0])                   # reference :784-785, :1161-1162
    Ad, Bd = as_csr_device(A), as_csr_device(B)       # reference :786-790 builds A - sigma B / B + sigma A
    if mode == "normal":
        vals = D.axpby(1.0, Ad.data, -float(sigma), Bd.data)
    else:
        vals = D.axpby(1.0, Bd.data, float(sigma), Ad.data)
    return SpLuOperator(Ad.with_values(vals))


def _return_psi(psi_d, psi_in, Phib):
    """The reference updates a caller-supplied initial guess in place and returns it (:792-795, :1182-1186)."""
    if is_dev(Phib):
        return psi_d
    if psi_in is not None and not is_dev(psi_in):
        psi_in[...] = to_host(psi_d)
        return psi_in
    return to_host(psi_d)


def _replay(callback, hist):
    if callback is not None:
        for per_mode in hist:
            for r in per_mode:
                callback(float(r))


_PINNED = {}


def _pinned(shape):
    """Cached page-locked host buffer (cudaHostAlloc is too slow to repeat per call)."""
    t = _PINNED.get(shape)
    if t is None:
        if len(_PINNED) > 16:
            _PINNED.clear()
        t = _PINNED[shape] = torch.empty(shape, dtype=torch.float64, pin_memory=True)
    return t


def _masked_inverse(vals, active):
    out = np.zeros_like(vals)
    ok = active & (vals > 0.0)
    out[ok] = 1.0 / vals[ok]
    return out


def _sibk_dev(Phib_d, Ad, Bd, lam, Phi_d, mode, psi_d, sigma, factor, rtol, atol, maxiter, rnorm0=None):
    n, N = Phib_d.shape
    lam = np.asarray(lam, dtype=float)
    lam_d = small_to_dev(lam)
    # Everything up to the first Krylov vector is queued before the first read-back, so the device runs through the
    # set-up once instead of draining at four small device -> host copies (the second projection and its norms are
    # wasted only when every mode is already converged).
    rn_d = D.col_dot(Phib_d, Phib_d) if rnorm0 is None else None                 # :1170 (max over ALL modes)
    BPhi = Bd.spmm(Phi_d)                                                        # :1173
    G_d = D.gemm_tn(Phi_d, Phib_d)                                               # :1180
    R = _neg_sum(_contig(Phib_d), _apply_L(Ad, Bd, lam_d, psi_d, mode))          # :1189-1193
    _project(BPhi, Phi_d, R)
    beta0_d = D.col_dot(R, R)
    # first Krylov vector: w0 = P R / ||P R||   (:1227-1234 with bs = 1)
    W = [R]
    _project(BPhi, Phi_d, W[0])
    r0_d = D.col_dot(W[0], W[0])
    if rn_d is not None:
        rnorm0 = float(np.sqrt(np.max(to_host(rn_d))))
    G = -to_host(G_d)
    beta0 = np.sqrt(to_host(beta0_d))
    hist = [[b] for b in beta0]
    active = ~((beta0 < rtol * rnorm0) | (beta0 < atol))
    info = [0] * N
    if not active.any():
        return G, info, hist
    r0 = np.sqrt(to_host(r0_d))
    D.col_scale(W[0], small_to_dev(_masked_inverse(r0, active)), mode=0)
    Z = []
    alpha = (lam - sigma) if mode == "normal" else -(lam - sigma)                 # :1262-1266
    opmat = Bd if mode == "normal" else Ad
    H = np.zeros((N, maxiter + 1, maxiter))
    Ycoef = np.zeros((maxiter, N))
    hdev = D.zeros(maxiter + 2, N)
    done = ~active
    # The Hessenberg column of iteration j is copied to pinned host memory asynchronously and the small
    # least-squares problems (:1043-1049) are solved on the host WHILE the device already runs iteration
    # j + 1 (its work does not depend on them; only the decision to stop does).  The price is one
    # speculative iteration at the end, the gain is that the device never waits for the host.
    hpin = _pinned((2, maxiter + 2, N))
    events = [torch.cuda.Event(), torch.cuda.Event()]

    def host_step(j):
        events[j & 1].synchronize()
        XFER["d2h"] += (j + 1) * N * 8
        hcol = hpin[j & 1, : j + 1].numpy().copy()
        hcol[j] = np.sqrt(hcol[j])
        H[:, : j + 1, j - 1] = hcol.T
        for i in np.nonzero(~done)[0]:
            Hi = np.eye(j + 1, j) - alpha[i] * H[i, : j + 1, :j]
            rhs = np.zeros(j + 1)
            rhs[0] = r0[i]
            y = np.linalg.lstsq(Hi, rhs, rcond=None)[0]                           # :1043-1049
            res = float(np.linalg.norm(Hi @ y - rhs))
            hist[i].append(res)
            ok = res < rtol * rnorm0 or res < atol
            if ok or j == maxiter:
                Ycoef[:j, i] = y
                info[i] = j if ok else -1
                done[i] = True

    for j in range(1, maxiter + 1):
        Z.append(factor.solve_dev(W[j - 1]))                                      # :1248
        w = opmat.spmm(Z[j - 1])                                                  # :1250-1252
        _project(BPhi, Phi_d, w)
        ks = range(j - 1, -1, -1)                                                 # modified Gram-Schmidt, descending (:1254-1257)
        D.mgs_sweep(w, [W[k] for k in ks], [hdev[k] for k in ks])
        _project(BPhi, Phi_d, w)                                                  # :1258
        D.col_dot(w, w, out=hdev[j])
        D.col_scale(w, hdev[j], mode=3)                                           # :1259-1260
        W.append(w)
        hpin[j & 1, : j + 1].copy_(hdev[: j + 1], non_blocking=True)
        events[j & 1].record()
        if j > 1:
            host_step(j - 1)
            if done.all():
                factor.count -= N             # the speculative solve of iteration j is not part of the result
                Z.pop()
                break
    else:
        j = maxiter + 1
    if not done.all():
        host_step(j - 1 if j > maxiter else j)
    for jj, Zj in enumerate(Z):                                                   # psi_i += Z y  (:1275-1277)
        if np.any(Ycoef[jj]):
            D.col_axpy(psi_d, small_to_dev(Ycoef[jj]), Zj, sign=1.0)
    return G, info, hist


def _sibk_seq_dev(Phib_d, Ad, Bd, lam, Phi_d, mode, psi_d, sigma, factor, rtol, atol, maxiter, bs_target, update_guess,
                  nrestart, callback):
    """The reference's coupled variants of sibk (:1195-1321): modes are visited in order, ``bs_target`` of them share
    one block Arnoldi process, and with ``update_guess`` the finished Krylov space is recycled to improve the guesses
    and residuals of the modes still to come (:1279-1305).  Inherently sequential (one single-column solve per
    Arnoldi step), so it runs vector by vector on the device; the Krylov bases are vector-major so that the
    orthogonalisation uses the same basis kernels as the Lanczos recurrence (classical Gram-Schmidt, two passes,
    instead of the reference's modified Gram-Schmidt: same space, same converged solution)."""
    n, N = Phib_d.shape
    lam = np.asarray(lam, dtype=float)
    lam_d = small_to_dev(lam)
    rnorm0 = float(np.sqrt(np.max(to_host(D.col_dot(Phib_d, Phib_d)))))           # :1170
    BPhi = Bd.spmm(Phi_d)
    G = -to_host(D.gemm_tn(Phi_d, Phib_d))
    R = _neg_sum(_contig(Phib_d), _apply_L(Ad, Bd, lam_d, psi_d, mode))           # :1189-1193
    _project(BPhi, Phi_d, R)
    opmat = Bd if mode == "normal" else Ad
    Wt = D.empty(maxiter + bs_target, n)          # Krylov vectors, one per row
    Zt = D.empty(maxiter, n)
    hbuf = D.zeros(maxiter + bs_target + 1)
    info = []

    def alpha_of(k):
        return (lam[k] - sigma) if mode == "normal" else -(lam[k] - sigma)

    def lstsq(alpha, H0, rhs):                                                      # :1043-1049
        Hi = np.eye(H0.shape[0], H0.shape[1]) - alpha * H0
        y = np.linalg.lstsq(Hi, rhs, rcond=None)[0]
        return y, float(np.linalg.norm(Hi @ y - rhs))

    def norm(v):
        return float(np.sqrt(to_host(D.col_dot(v, v))[0]))

    def orth(w, j):
        """w -= W[:, :j] (W[:, :j]^T w), two classical passes; returns the summed coefficients"""
        h = np.zeros(j)
        if j == 0:
            return h
        for _ in range(2):
            D.gemm_tn(Wt[:j].T, w, out=hbuf[:j].unsqueeze(1))
            D.gemm_nn(Wt[:j].T, hbuf[:j].unsqueeze(1), w, alpha=-1.0, beta=1.0)
            h += to_host(hbuf[:j])
        return h

    i, restart = 0, 0
    while i < N:
        r = np.zeros((maxiter + bs_target, bs_target))
        bs = 0
        while i + bs < N and bs < bs_target:
            k = i + bs
            w = Wt[bs]
            if update_guess:                                                        # :1203-1215
                pk = _contig(psi_d[:, k])
                _project(Phi_d, BPhi, pk)
                psi_d[:, k].copy_(pk)
                Lp = _apply_L(Ad, Bd, lam_d[k:k + 1], pk.unsqueeze(1), mode).reshape(-1)
                D.axpby(-1.0, _contig(Phib_d[:, k]), -1.0, Lp, out=w)
                _project(BPhi, Phi_d, w)
            else:
                w.copy_(R[:, k])                                                    # :1217
            beta0 = norm(w)
            if callback is not None:
                callback(beta0)
            if beta0 < rtol * rnorm0 or beta0 < atol:
                info.append(0)
                break
            r[:bs, bs] = orth(w, bs)                                                # :1228-1230
            _project(BPhi, Phi_d, w)
            r[bs, bs] = norm(w)
            w.mul_(1.0 / r[bs, bs])
            bs += 1
        if bs == 0:
            i += 1
            continue
        H = np.zeros((maxiter + bs, maxiter))
        y = np.zeros((maxiter, bs))
        for j in range(bs, maxiter + bs):
            kp = j - bs
            factor.solve_dev(Wt[kp], out=Zt[kp])                                    # :1248
            w = Wt[j]
            opmat.spmm(Zt[kp], out=w)
            _project(BPhi, Phi_d, w)
            H[:j, kp] = orth(w, j)                                                  # :1254-1257
            _project(BPhi, Phi_d, w)
            H[j, kp] = norm(w)
            w.mul_(1.0 / H[j, kp])
            res = 0.0
            H0 = H[: j + 1, : j + 1 - bs]
            for k in range(bs):
                y[: kp + 1, k], res0 = lstsq(alpha_of(i + k), H0, r[: j + 1, k])
                res = max(res, res0)
            if callback is not None:
                callback(res)
            converged = res < rtol * rnorm0 or res < atol
            if converged or j == maxiter + bs - 1:
                nz = kp + 1
                D.gemm_nn(Zt[:nz].T, small_to_dev(y[:nz, :]), psi_d[:, i:i + bs], alpha=1.0, beta=1.0)   # :1276 / :1310
            if converged:
                info.append(j)
                if update_guess and i + bs < N:                                     # :1279-1305
                    rest = N - (i + bs)
                    r0 = to_host(D.gemm_tn(Wt[: j + 1].T, R[:, i + bs:]))
                    y0 = np.zeros((j + 1 - bs, rest))
                    t0 = np.zeros((j + 1, rest))
                    for c in range(rest):
                        a_k = alpha_of(i + bs + c)
                        yk, _ = lstsq(a_k, H0, r0[:, c])
                        y0[:, c] = yk
                        t0[:, c] = -a_k * (H0 @ yk)
                        t0[: j + 1 - bs, c] += yk
                    D.gemm_nn(Zt[: j + 1 - bs].T, small_to_dev(y0), psi_d[:, i + bs:], alpha=1.0, beta=1.0)
                    D.gemm_nn(Wt[: j + 1].T, small_to_dev(t0), R[:, i + bs:], alpha=-1.0, beta=1.0)
                i += bs
                restart = 0
                break
            if j == maxiter + bs - 1:
                if restart >= nrestart:
                    restart = 0
                    i += bs
                    break
                restart += 1
    return G, info


@_public
def sibk(Phib, A, B, lam, Phi, mode="normal", psi=None, sigma=None, factor=None, rtol=1e-10, atol=1e-30,
         eig_atol=1e-5, maxiter=50, bs_target=1, update_guess=False, callback=None, nrestart=2):
    """Reference ``sibk`` (:1052-1328), shift-and-invert block Krylov, with the N per-mode Arnoldi
    processes advanced in lock step (default settings of every reference example).  ``bs_target > 1`` and
    ``update_guess=True`` (the reference's coupled block / recycling variants, :1195-1321) run the sequential
    form ``_sibk_seq_dev``."""
    n, N = _check_krylov_args(Phib, A, B, lam, Phi, psi, mode)
    lam_h = to_host(lam) if is_dev(lam) else np.asarray(lam, dtype=float)
    if sigma is None:
        if factor is not None:
            raise ValueError("sibk needs the shift sigma that the factorisation was built with")
        sigma = 0.9 * float(lam_h[0])                                              # :1161-1162
    factor = _default_factor(A, B, sigma, mode, factor, lam_h)
    Ad, Bd = as_csr_device(A), as_csr_device(B)
    Phi_d, Phib_d = to_dev(Phi), to_dev(Phib)
    psi_d = D.zeros(n, N) if psi is None else to_dev(psi, copy=True)
    if bs_target != 1 or update_guess:
        G, info = _sibk_seq_dev(Phib_d, Ad, Bd, lam_h, Phi_d, mode, psi_d, float(sigma), factor, rtol, atol, maxiter,
                                int(bs_target), bool(update_guess), nrestart, callback)
        data = _apply_correction_dev(lam_h, Phi_d, psi_d, G, eig_atol, mode)
        return _return_psi(psi_d, psi, Phib), data, info
    G, info, hist = _sibk_dev(Phib_d, Ad, Bd, lam_h, Phi_d, mode, psi_d, float(sigma), factor, rtol, atol, maxiter)
    _replay(callback, hist)
    data = _apply_correction_dev(lam_h, Phi_d, psi_d, G, eig_atol, mode)          # :1324
    return _return_psi(psi_d, psi, Phib), data, info


def _pcpg_dev(Phib_d, Ad, Bd, lam, Phi_d, mode, psi_d, factor, rtol, atol, maxiter, reset, rnorm0=None):
    n, N = Phib_d.shape
    lam = np.asarray(lam, dtype=float)
    lam_d = small_to_dev(lam)
    if rnorm0 is None:
        rnorm0 = float(np.sqrt(np.max(to_host(D.col_dot(Phib_d, Phib_d)))))
    BPhi = Bd.spmm(Phi_d)
    R = _neg_sum(_contig(Phib_d), _apply_L(Ad, Bd, lam_d, psi_d, mode))           # :806
    # G[:, i] = Phi^T R_i ; R_i -= BPhi G[:, i]   (:807-811)
    Gd = D.gemm_tn(Phi_d, R)
    D.gemm_nn(BPhi, Gd, R, alpha=-1.0, beta=1.0)
    G = to_host(Gd)
    P = D.zeros(n, N)
    prev = np.ones(N)
    done = np.zeros(N, dtype=bool)
    info = [False] * N
    hist = [[] for _ in range(N)]
    for k in range(maxiter):
        res = _col_norms(R)
        for i in np.nonzero(~done)[0]:
            hist[i].append(res[i])
            if res[i] < rtol * rnorm0 or res[i] < atol:
                done[i] = True
                info[i] = True
        if done.all():
            break
        Zt = R.clone()
        _project(BPhi, Phi_d, Zt)
        Zt = factor.solve_dev(Zt)
        _project(Phi_d, BPhi, Zt)                                                 # :829-830
        zr = to_host(D.col_dot(Zt, R))
        bcoef = np.zeros(N) if k % reset == 0 else zr / prev                      # :832-840
        bcoef[done] = 0.0
        prev = np.where(done, prev, zr)
        D.col_scale(P, small_to_dev(bcoef), mode=0)
        D.axpby(1.0, P.reshape(-1), 1.0, Zt.reshape(-1), out=P.reshape(-1))
        LP = _apply_L(Ad, Bd, lam_d, P, mode)
        pLp = to_host(D.col_dot(LP, P))
        a = np.where(done, 0.0, zr / np.where(pLp == 0.0, 1.0, pLp))              # :842-857
        a_d = small_to_dev(a)
        D.col_axpy(psi_d, a_d, P, sign=1.0)
        D.col_axpy(R, a_d, LP, sign=-1.0)
    return G, info, hist


@_public
def pcpg(Phib, A, B, lam, Phi, mode="normal", psi=None, sigma=None, factor=None, rtol=1e-10, atol=1e-30,
         eig_atol=1e-5, maxiter=100, reset=25, callback=None):
    """Reference ``pcpg`` (:699-869): projected preconditioned conjugate gradients, all modes in lock step."""
    n, N = _check_krylov_args(Phib, A, B, lam, Phi, psi, mode)
    lam_h = to_host(lam) if is_dev(lam) else np.asarray(lam, dtype=float)
    factor = _default_factor(A, B, sigma, mode, factor, lam_h)
    Ad, Bd = as_csr_device(A), as_csr_device(B)
    Phi_d, Phib_d = to_dev(Phi), to_dev(Phib)
    psi_d = D.zeros(n, N) if psi is None else to_dev(psi, copy=True)
    G, info, hist = _pcpg_dev(Phib_d, Ad, Bd, lam_h, Phi_d, mode, psi_d, factor, rtol, atol, maxiter, reset)
    _replay(callback, hist)
    data = _apply_correction_dev(lam_h, Phi_d, psi_d, G, eig_atol, mode)
    return _return_psi(psi_d, psi, Phib), data, info


def _pgmres_dev(Phib_d, Ad, Bd, lam, Phi_d, mode, psi_d, factor, rtol, atol, maxiter, rnorm0=None):
    n, N = Phib_d.shape
    lam = np.asarray(lam, dtype=float)
    lam_d = small_to_dev(lam)
    if rnorm0 is None:
        rnorm0 = float(np.sqrt(np.max(to_host(D.col_dot(Phib_d, Phib_d)))))
    BPhi = Bd.spmm(Phi_d)
    R = _neg_sum(_contig(Phib_d), _apply_L(Ad, Bd, lam_d, psi_d, mode))           # :985
    Gd = D.gemm_tn(Phi_d, R)
    D.gemm_nn(BPhi, Gd, R, alpha=-1.0, beta=1.0)                                  # :986-990
    G = to_host(Gd)
    beta = _col_norms(R)
    hist = [[b] for b in beta]
    active = ~((beta < rtol * rnorm0) | (beta < atol))
    info = [0] * N
    if not active.any():
        return G, info, hist
    W = [R]
    D.col_scale(W[0], small_to_dev(_masked_inverse(beta, active)), mode=0)
    Z = []
    H = np.zeros((N, maxiter + 1, maxiter))
    Ycoef = np.zeros((maxiter, N))
    hdev = D.zeros(maxiter + 2, N)
    done = ~active
    for j in range(maxiter):
        t = W[j].clone()
        _project(BPhi, Phi_d, t)
        Z.append(factor.solve_dev(t))                                             # :1003
        w = _apply_L(Ad, Bd, lam_d, Z[j], mode)
        _project(BPhi, Phi_d, w)                                                  # :1004-1010
        D.mgs_sweep(w, W[: j + 1], [hdev[k] for k in range(j + 1)])               # MGS ascending (:1012-1014)
        D.col_dot(w, w, out=hdev[j + 1])
        D.col_scale(w, hdev[j + 1], mode=3)
        W.append(w)
        hcol = to_host(hdev[: j + 2])
        hcol[j + 1] = np.sqrt(hcol[j + 1])
        H[:, : j + 2, j] = hcol.T
        for i in np.nonzero(~done)[0]:
            Hi = H[i, : j + 2, : j + 1]
            rhs = np.zeros(j + 2)
            rhs[0] = beta[i]
            y = np.linalg.lstsq(Hi, rhs, rcond=None)[0]                           # :1019-1022
            res = float(np.linalg.norm(Hi @ y - rhs))
            hist[i].append(res)
            ok = res < rtol * rnorm0 or res < atol
            if ok or j == maxiter - 1:
                Ycoef[: j + 1, i] = y
                info[i] = j if ok else -1
                done[i] = True
        if done.all():
            break
    for jj, Zj in enumerate(Z):
        if np.any(Ycoef[jj]):
            D.col_axpy(psi_d, small_to_dev(Ycoef[jj]), Zj, sign=1.0)
    return G, info, hist


@_public
def pgmres(Phib, A, B, lam, Phi, mode="normal", psi=None, sigma=None, factor=None, rtol=1e-10, atol=1e-30,
           eig_atol=1e-5, maxiter=50, callback=None):
    """Reference ``pgmres`` (:872-1040): right-preconditioned projected GMRES, all modes in lock step."""
    n, N = _check_krylov_args(Phib, A, B, lam, Phi, psi, mode)
    lam_h = to_host(lam) if is_dev(lam) else np.asarray(lam, dtype=float)
    factor = _default_factor(A, B, sigma, mode, factor, lam_h)
    Ad, Bd = as_csr_device(A), as_csr_device(B)
    Phi_d, Phib_d = to_dev(Phi), to_dev(Phib)
    psi_d = D.zeros(n, N) if psi is None else to_dev(psi, copy=True)
    G, info, hist = _pgmres_dev(Phib_d, Ad, Bd, lam_h, Phi_d, mode, psi_d, factor, rtol, atol, maxiter)
    _replay(callback, hist)
    data = _apply_correction_dev(lam_h, Phi_d, psi_d, G, eig_atol, mode)
    return _return_psi(psi_d, psi, Phib), data, info


# ------------------------------------------------------------------------------------------
# eigensolver classes
# ------------------------------------------------------------------------------------------
class _SolverBase:
    """State shared by IRAM and BasicLanczos between solve / solve_adjoint / add_total_derivative
    (the reference keeps the same attributes on the solver object, SURVEY.md section 5)."""

    def _common_solve_checks(self, A, B, factor):
        n = A.shape[1]
        if A.shape != (n, n):
            raise ValueError(f"A must have dimensions ({n},{n})")
        if B.shape != (n, n):
            raise ValueError(f"B must have dimensions ({n},{n})")
        if factor.shape != (n, n):
            raise ValueError(f"Factorized operator must have dimensions ({n},{n})")
        if not hasattr(factor, "solve_dev"):
            raise TypeError("factor must be an eigd_b200.SpLuOperator (device LDL^T); there is no CPU fallback")
        return n

    def _publish_phi(self, Phi_d, A):
        """numpy callers get a host copy of the eigenvectors (reference convention); callers that handed
        in device matrices keep them in HBM."""
        if isinstance(A, D.CsrDevice):
            self.Phi = Phi_d
        else:
            self.Phi = to_host(Phi_d)

    def _phi_dev(self):
        """Device copy of the eigenvectors.  When ``solve`` returned a host array, that array is authoritative: the
        callers slice it and edit it in place (sign flips, examples/natural_frequency.py:383-390), and nothing short
        of reading all of it can tell whether they did -- so it is uploaded again at every entry point (20 MB at C2:
        0.4 ms of DMA from the page-locked block ``solve`` returned it in).  No fingerprints, no reuse."""
        if is_dev(self.Phi):
            return self.Phi
        self._Phi_d = to_dev(self.Phi)
        return self._Phi_d

    def _phib_dev(self, Phib):
        """Device copy of the adjoint right-hand sides: uploaded on every call (the caller owns the array and may
        refill it between ``solve_adjoint`` and ``add_total_derivative``)."""
        return to_dev(Phib)

    def _adjoint(self, lam, Phib, method, psi, rtol, atol, lanczos_guess, kwargs):
        n = self.A.shape[1]
        if method not in ("pcpg", "pgmres", "sibk", "laa", "dl"):
            raise ValueError(f"Unknown method {method!r}")
        if psi is not None and tuple(psi.shape) != (n, self.N):
            raise ValueError(f"Initial guess must have the shape ({n},{self.N})")
        if tuple(Phib.shape) != (n, self.N):
            raise ValueError(f"Right-hand-side must have the shape ({n},{self.N})")
        if method == "dl":
            lanczos_guess = False
        Phib_d = self._phib_dev(Phib)
        Phi_d = self._phi_dev()
        lam = np.asarray(lam, dtype=float)
        callback = kwargs.pop("callback", None)
        N = self.N
        shard = getattr(self, "sharding", None)
        if shard is not None and (shard.world == 1 or method == "dl"):
            shard = None                      # dl is one sequential sweep over the Lanczos vectors: replicated
        if shard is None:
            cols, Phib_s, lam_s = None, Phib_d, lam
        else:                                 # per-mode shard: this rank owns modes rank, rank+world, ...
            cols = shard.my_cols(N)
            lam_s = lam[cols]
            Phib_s = D.empty(n, len(cols))
            if len(cols):
                D.copy2d(Phib_d[:, shard.rank::shard.world], Phib_s)
        Ns = Phib_s.shape[1]
        if (lanczos_guess or method == "laa") and Ns:
            psi_s = _laa_dev(Phib_s, self._Bd, self.factor, self.sigma, lam_s, self._V_d, self.Y, self.theta,
                             self.indices, True, self.mode, cols=cols, Nfull=N)
        else:
            psi_s = D.zeros(n, Ns)
        if method == "dl":
            psi_d, data = _dl_dev(Phib_d, self._Bd, self.factor, self.sigma, lam, Phi_d, self.indices, self._V_d,
                                  self.T, self.Y, self.theta, self.eig_atol, self.mode)
            return like_input(psi_d, Phib), data
        G, info, hist = None, [], []
        rn0 = None if shard is None else float(np.sqrt(np.max(to_host(D.col_dot(Phib_d, Phib_d)))))
        if method != "laa" and Ns:
            if method == "sibk":
                bs_target, update_guess = int(kwargs.pop("bs_target", 1)), bool(kwargs.pop("update_guess", False))
                nrestart = kwargs.pop("nrestart", 2)
                if bs_target != 1 or update_guess:
                    # coupled block / recycling variants (:1195-1321): sequential over the modes, not sharded
                    if shard is not None:
                        raise NotImplementedError("sibk with bs_target > 1 or update_guess=True couples the modes and "
                                                  "cannot be sharded per mode")
                    G, info = _sibk_seq_dev(Phib_s, self._Ad, self._Bd, lam_s, Phi_d, self.mode, psi_s, float(self.sigma),
                                            self.factor, rtol, atol, kwargs.pop("maxiter", 50), bs_target, update_guess,
                                            nrestart, callback)
                    callback = None
                else:
                    G, info, hist = _sibk_dev(Phib_s, self._Ad, self._Bd, lam_s, Phi_d, self.mode, psi_s,
                                              float(self.sigma), self.factor, rtol, atol, kwargs.pop("maxiter", 50),
                                              rnorm0=rn0)
            elif method == "pcpg":
                G, info, hist = _pcpg_dev(Phib_s, self._Ad, self._Bd, lam_s, Phi_d, self.mode, psi_s, self.factor, rtol,
                                          atol, kwargs.pop("maxiter", 100), kwargs.pop("reset", 25), rnorm0=rn0)
            else:
                G, info, hist = _pgmres_dev(Phib_s, self._Ad, self._Bd, lam_s, Phi_d, self.mode, psi_s, self.factor,
                                            rtol, atol, kwargs.pop("maxiter", 50), rnorm0=rn0)
            if kwargs:
                raise TypeError("unexpected keyword arguments %r" % sorted(kwargs))
        if shard is None:
            psi_d = psi_s
        elif method == "laa":
            psi_d = shard.allgather_cols(psi_s, N, transpose=D.copy2d)
        else:                                 # ONE packed all-gather: psi columns + per-mode scalars (dist.py)
            packed = shard.pack_mode_scalars(N, G if G is not None else np.zeros((N, 0)), info, hist)
            psi_d, extras = shard.allgather_cols(psi_s, N, transpose=D.copy2d, extra=packed)
            G, info, hist = shard.unpack_mode_scalars(N, extras, info_type=bool if method == "pcpg" else int)
        if method == "laa":
            G = -to_host(D.gemm_tn(Phi_d, Phib_d))
        self.adjoint_info = info
        _replay(callback, hist)
        data = _apply_correction_dev(lam, Phi_d, psi_d, G, self.eig_atol, self.mode)
        return like_input(psi_d, Phib), data


class BasicLanczos(_SolverBase):
    """Reference ``BasicLanczos`` (:1331-1870): un-restarted shift-and-invert Lanczos with full
    B-orthogonalisation (modified Gram-Schmidt, descending order) and a fixed seeded start vector.
    ``ortho_type="selective"`` (:1553-1605) orthogonalises against the two previous vectors and the nearly converged
    Ritz vectors only.  Complex (complex-step) operands are not on the device path."""

    def __init__(self, N=10, m=60, tol=1e-14, Ntarget=None, eig_atol=1e-5, mode="normal", ortho_type="full"):
        if Ntarget is not None and not isinstance(Ntarget, (int, np.integer)):
            raise ValueError("Ntarget must be an integer or None")
        if ortho_type not in ("full", "selective"):
            raise ValueError(f"Unknown ortho_type {ortho_type!r}")
        _check_mode(mode)
        self.N, self.m_max, self.tol, self.Ntarget = N, m, tol, Ntarget
        self.eig_atol, self.mode, self.ortho_type = eig_atol, mode, ortho_type
        self.m = m
        self._Phi_d = None

    def _solve_reduced_problem(self, alpha, beta, sigma, m):
        T = np.diag(alpha[:m]) + np.diag(beta[: m - 1], 1) + np.diag(beta[: m - 1], -1)     # :1416-1439
        theta, Y = np.linalg.eigh(T)
        if self.mode == "normal":
            lam = 1.0 / theta + sigma
            indices = np.argsort(lam)
        else:
            lam = sigma * theta / (theta - 1.0)
            indices = np.argsort(-1.0 / lam)
        return theta, Y, T, lam, indices

    def _solve_dual(self, A, B, factor, sigma):
        """Complex-step operands (reference :1483-1493 dtype switch): the recurrence in dual numbers (dual.py)."""
        from . import dual
        if self.ortho_type != "full":
            raise NotImplementedError("complex-step operands are implemented for ortho_type='full'")
        if getattr(factor, "tangent", None) is None:
            raise ValueError("complex A, B need a SpLuOperator built from the complex shifted matrix")
        def z(M):
            if isinstance(M, tuple):                     # (value, tangent) CsrDevice pair prepared on the device (topo drivers)
                return M
            if dual.is_complex_matrix(M):
                return dual.split_csr(M)
            Md = as_csr_device(M)
            return Md, Md.with_values(D.zeros(Md.nnz))
        (Ar, At), (Br, Bt) = z(A), z(B)
        self.A, self.B, self.factor, self.sigma = A, B, factor, sigma
        self._Ad, self._Bd = Ar, Br
        res = dual.basic_lanczos(Ar, At, Br, Bt, factor, sigma, self.N, self.m_max, self.tol, self.Ntarget, self.mode)
        m = self.m = res["m"]
        self.alpha, self.beta = res["alpha"], res["beta"]
        self.theta, self.Y, self.T, self.lam, self.indices = res["theta"], res["Y"], res["T"], res["lam"], res["indices"]
        if self.Ntarget is not None:
            self.N = self.Ntarget
            while self.N < m and _is_close(self.lam[self.indices[self.N - 1]].real, self.lam[self.indices[self.N]].real,
                                           self.eig_atol):
                self.N += 1
        self.lam0 = self.lam[self.indices[: self.N]]
        self.Y0 = self.Y[:, self.indices[: self.N]]
        self.eig_res = np.abs(self.beta[m - 1].real * self.Y0[m - 1, :].real)
        self.fail = bool(np.any(self.eig_res >= max(self.tol, 1e-8)))
        self.Phi = dual.ritz_vectors(res, self.indices[: self.N])
        self._Phi_d = None
        self._dual = res
        self._V_host = np.stack([to_host(v.r) + 1j * to_host(v.t) for v in res["V"]], axis=1)
        return self.lam0, self.Phi

    @_public
    def solve(self, A, B, factor, sigma):
        if _is_complex_host(A) or _is_complex_host(B) or isinstance(A, tuple) or isinstance(B, tuple):
            return self._solve_dual(A, B, factor, sigma)
        n = self._common_solve_checks(A, B, factor)
        self.A, self.B, self.factor, self.sigma = A, B, factor, sigma
        self._Ad, self._Bd = as_csr_device(A), as_csr_device(B)
        Bd = self._Bd
        m_max = self.m_max
        alpha, beta = np.zeros(m_max), np.zeros(m_max)
        Vt = D.empty(m_max + 1, n)                   # vector-major basis
        BVt = D.empty(m_max + 1, n)
        v0 = np.random.default_rng(12345).uniform(size=n, low=-1.0, high=1.0)               # :1514-1515
        Vt[0].copy_(to_dev(v0))
        Bd.spmm(Vt[0], out=BVt[0])
        nrm2 = D.col_dot(Vt[0], BVt[0])
        D.col_scale(Vt[0], nrm2, mode=2)
        D.col_scale(BVt[0], nrm2, mode=2)
        hdev = D.zeros(m_max + 2)
        w = D.empty(n)
        bw = D.empty(n)
        self.m = m_max
        Nc = self.N if self.Ntarget is None else self.Ntarget
        S_d = BS_d = None                            # selective orthogonalisation: Ritz vectors and their B-images
        for i in range(1, m_max + 1):
            factor.solve_dev(BVt[i - 1], out=w)                                             # :1500
            if i > 1:
                D.col_axpy(w, small_to_dev([beta[i - 2]]), Vt[i - 2], sign=-1.0)
            # full: B-MGS against every previous vector, descending (:1522-1538); selective: only against the two
            # previous vectors (:1560-1567), then against the nearly converged Ritz vectors S (:1569-1573)
            jlo = -1 if self.ortho_type == "full" else max(-1, i - 3)
            for j in range(i - 1, jlo, -1):
                D.col_dot(w, BVt[j], out=hdev[j: j + 1])
                D.col_axpy(w, hdev[j: j + 1], Vt[j], sign=-1.0)
            if S_d is not None:
                hs = D.gemm_tn(BS_d, w.unsqueeze(1))
                D.gemm_nn(S_d, hs, w.unsqueeze(1), alpha=-1.0, beta=1.0)
            Bd.spmm(w, out=bw)
            D.col_dot(w, bw, out=hdev[i: i + 1])
            Vt[i].copy_(w)
            BVt[i].copy_(bw)
            D.col_scale(Vt[i], hdev[i: i + 1], mode=2)
            D.col_scale(BVt[i], hdev[i: i + 1], mode=2)
            hh = to_host(hdev[i - 1: i + 1])
            alpha[i - 1], beta[i - 1] = hh[0], np.sqrt(hh[1])
            if i >= 2:
                theta, Y, T, lam, idx = self._solve_reduced_problem(alpha, beta, sigma, i)
                err = np.abs(beta[i - 1] * Y[i - 1, idx])                                   # :1441-1451
                bad = np.nonzero(err >= self.tol)[0]
                if (len(err) if len(bad) == 0 else bad[0]) >= Nc:
                    self.m = i
                    break
                if self.ortho_type == "selective":                                          # :1591-1602
                    conv = np.nonzero(err < np.sqrt(self.tol))[0]
                    S_d = BS_d = None
                    if len(conv):
                        S_d = D.empty(n, len(conv))
                        D.gemm_nn(Vt[:i].T, small_to_dev(np.ascontiguousarray(Y[:, idx][:, conv])), S_d, alpha=1.0, beta=0.0)
                        BS_d = Bd.spmm(S_d)
        m = self.m
        self.alpha, self.beta = alpha, beta
        self.theta, self.Y, self.T, self.lam, self.indices = self._solve_reduced_problem(alpha, beta, sigma, m)
        if self.Ntarget is not None:                                                        # :1615-1625
            self.N = self.Ntarget
            while self.N < m and _is_close(self.lam[self.indices[self.N - 1]], self.lam[self.indices[self.N]], self.eig_atol):
                self.N += 1
        if self.N < m and _is_close(self.lam[self.indices[self.N - 1]], self.lam[self.indices[self.N]], self.eig_atol):
            warnings.warn(f"BasicLanczos: Ritz values {self.N} and {self.N+1} are numerically repeated.")   # :1632
        self.lam0 = self.lam[self.indices[: self.N]]
        self.Y0 = self.Y[:, self.indices[: self.N]]
        self.eig_res = np.abs(beta[m - 1] * self.Y0[m - 1, :])
        self.fail = bool(np.any(self.eig_res >= max(self.tol, 1e-8)))
        self._Vt = Vt
        self._V_d = Vt[:m].T
        Phi_d = D.empty(n, self.N)
        D.gemm_nn(self._V_d, small_to_dev(self.Y0), Phi_d, alpha=1.0, beta=0.0)            # :1648
        self._Phi_d = Phi_d
        self._V_host = None
        self._publish_phi(Phi_d, A)
        return self.lam0, self.Phi

    @property
    def V(self):
        """(n, m_max + 1) Lanczos basis as a numpy array (copied from HBM on first access)."""
        if self._V_host is None:
            self._V_host = to_host(self._Vt).T.copy()
        return self._V_host

    @_public
    def solve_adjoint(self, Phib, method="sibk", psi=None, rtol=1e-10, atol=1e-30, lanczos_guess=True, **kwargs):
        """Reference :1652-1797."""
        return self._adjoint(self.lam0, Phib, method, psi, rtol, atol, lanczos_guess, dict(kwargs))

    @_public
    def eval_adjoint_residual_norm(self, Phib, psi, b_ortho=False):
        """Reference :1799-1828."""
        return eval_adjoint_residual_norm(self._Ad, self._Bd, self.lam0, self._phi_dev(), self._phib_dev(Phib), to_dev(psi),
                                          mode=self.mode, b_ortho=b_ortho)

    @_public
    def add_total_derivative(self, lamb, Phib, psi, dAdx, dBdx, dfdx, adj_corr_data={}, deriv_type="vector"):
        """Reference :1830-1870."""
        return add_eig_total_derivative(self.lam0, self._phi_dev(), lamb, self._phib_dev(Phib), to_dev(psi), dAdx, dBdx, dfdx,
                                        adj_corr_data=adj_corr_data, mode=self.mode, deriv_type=deriv_type)


class IRAM(_SolverBase):
    """Reference ``IRAM`` (:1873-2207): restarted shift-and-invert Lanczos + adjoint solvers."""

    def __init__(self, N=10, m=None, eig_atol=1e-5, tol=0.0, mode="normal"):
        self.N = N
        self.m = max(20, 2 * N + 1) if m is None else max(20, 2 * N + 1, m)                 # :1896-1900
        self.eig_atol, self.tol = eig_atol, tol
        _check_mode(mode)
        self.mode = mode
        self.seed = None          # start-vector seed (scipy >= 1.15 draws it at random; None keeps that)
        self.block_size = None    # Lanczos block size (None: arpack.BLOCK_SIZE; 1: single-vector recurrence)
        # The reference pairs the returned eigenvectors with ``indices[:N]``, the N first Ritz values in its sorted order
        # (:1960-1965).  When the shift lies inside the wanted spectrum (buckling, sigma above the first load factors)
        # that is NOT the set the eigensolver returned (the N largest |theta|): the Lanczos-adjoint guess then carries
        # components along Phi and the reference's gradient is wrong (BASELINE configs[2]: -11.90 against the finite-
        # difference value -3.654, tests/test_fullsize_golden_gpu.py).  Default here: ``indices`` lists the returned
        # pairs first (identical to the reference whenever the two sets coincide); True reproduces the reference.
        self.reference_pairing = False
        self._Phi_d = None

    @_public
    def solve(self, A, B, factor, sigma):
        n = self._common_solve_checks(A, B, factor)
        self.factor, self.A, self.B, self.sigma = factor, A, B, sigma
        self._Ad, self._Bd = as_csr_device(A), as_csr_device(B)
        A0 = self._Ad if self.mode == "normal" else self._Bd                                # :1938-1942
        seed = self.seed
        shard = getattr(self, "sharding", None)
        if seed is None and shard is not None and shard.world > 1:
            # replicated eigensolve: every rank must build the SAME basis (signs, rotations inside clusters), or
            # the adjoint columns gathered from the other ranks belong to different eigenvectors
            seed = 0
        lam, _, T, _, st = eigsh_mod(A0, M=self._Bd, OPinv=factor, k=self.N, sigma=sigma, which="LM", mode=self.mode,
                                     tol=self.tol, ncv=self.m, return_state=True, seed=seed, block=self.block_size)
        self.lam, self.T = lam, T
        self.lanczos_state = st
        self._V_d = st.Vt.T
        self._V_host = None
        # eigh(T) (:1958): the restart loop has just computed it for this very T (same LAPACK call, same input)
        self.theta, self.Y = (st.eigh_T[0].copy(), st.eigh_T[1].copy()) if getattr(st, "eigh_T", None) is not None \
            else np.linalg.eigh(self.T)
        if self.mode == "normal":
            eigs = 1.0 / self.theta + sigma
            self.indices = np.argsort(eigs)
        else:
            eigs = sigma * self.theta / (self.theta - 1.0)
            self.indices = np.argsort(-1.0 / eigs)
        sel = set(int(i) for i in st.sel)
        if not self.reference_pairing and set(int(i) for i in self.indices[: self.N]) != sel:
            # the returned pairs first (in the sorted order), then the remaining Ritz pairs (see __init__)
            self.indices = np.array([i for i in self.indices if int(i) in sel] + [i for i in self.indices if int(i) not in sel])
        if _is_close(eigs[self.indices[self.N - 1]], eigs[self.indices[self.N]], self.eig_atol):
            warnings.warn(f"IRAM: Ritz values {self.N} and {self.N+1} are numerically repeated.")   # :1967-1974
        # modal-assurance sign alignment of Y against the returned eigenvectors (:1978-1984):
        # sign(phi_i . V y_i) = sign((V^T B phi_i) . y_i) up to the positive-definite metric; evaluate it
        # in the reduced space through Q = V Y0 on the device
        if getattr(st, "eigh_T", None) is not None and np.array_equal(self.indices[: self.N], st.sel):
            pass      # the returned eigenvectors ARE V Y[:, indices[:N]] with this Y: every sign already agrees
        else:
            Q = D.empty(n, self.N)
            D.gemm_nn(self._V_d, small_to_dev(self.Y[:, self.indices[: self.N]]), Q, alpha=1.0, beta=0.0)
            mac = to_host(D.col_dot(Q, st.Z))
            for i in range(self.N):
                if mac[i] < 0.0:
                    self.Y[:, self.indices[i]] *= -1.0
        self._Phi_d = st.Z
        self._publish_phi(st.Z, A)
        return self.lam, self.Phi

    @property
    def V(self):
        if self._V_host is None:
            self._V_host = to_host(self.lanczos_state.Vt).T.copy()
        return self._V_host

    @_public
    def solve_adjoint(self, Phib, method="sibk", psi=None, rtol=1e-10, atol=1e-30, lanczos_guess=True, **kwargs):
        """Reference :1988-2134."""
        if method == "dl":
            warnings.warn("IRAM: the dl method requires the Lanczos three-term recurrence and gives wrong "
                          "results with a restarted basis; use BasicLanczos.")                # :2039-2043
        return self._adjoint(self.lam, Phib, method, psi, rtol, atol, lanczos_guess, dict(kwargs))

    @_public
    def eval_adjoint_residual_norm(self, Phib, psi, b_ortho=False):
        """Reference :2136-2165."""
        return eval_adjoint_residual_norm(self._Ad, self._Bd, self.lam, self._phi_dev(), self._phib_dev(Phib), to_dev(psi),
                                          mode=self.mode, b_ortho=b_ortho)

    @_public
    def add_total_derivative(self, lamb, Phib, psi, dAdx, dBdx, dfdx, adj_corr_data={}, deriv_type="vector"):
        """Reference :2167-2207."""
        return add_eig_total_derivative(self.lam, self._phi_dev(), lamb, self._phib_dev(Phib), to_dev(psi), dAdx, dBdx, dfdx,
                                        adj_corr_data=adj_corr_data, mode=self.mode, deriv_type=deriv_type)
