"""Thin device layer: torch owns HBM buffers and streams, every arithmetic op is one of the
hand-written kernels in libeigd_b200.so reached through the C-ABI (include/eigd_b200.h).

All dense operands are 2-D torch CUDA fp64 tensors of *logical* shape (n, k); their strides
are passed through unchanged, so a Krylov basis stored one vector per row is simply used as
``Vt.T``.  Nothing here falls back to the CPU: without the library or without a CUDA device
every call raises.
"""
import ctypes
import hashlib
import time
import warnings

import numpy as np

from . import _lib
from ._lib import check

try:
    import torch
except Exception as exc:  # pragma: no cover
    raise ImportError("eigd_b200 needs torch for device buffers") from exc


F64 = torch.float64


class _State:
    device = None
    work = None
    ready = False
    stream = None      # cudaStream_t the native library is currently bound to


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class Timeline:
    """Optional per-call CUDA-event timing of the heavy entry points (used by bench.py for the live
    roofline numbers).  Events are recorded on the stream the kernels are launched on (torch's
    current stream, see ``init``) and only resolved in ``summary`` after a synchronize."""
    enabled = False
    records = {}

    @classmethod
    def begin(cls, cat):
        if not cls.enabled:
            return None
        e0 = torch.cuda.Event(enable_timing=True)
        e0.record()
        return (cat, e0)

    @classmethod
    def end(cls, tok, nbytes=0, launches=0):
        if tok is None:
            return
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        cls.records.setdefault(tok[0], []).append((tok[1], e1, nbytes, launches))

    @classmethod
    def reset(cls):
        cls.records = {}

    @classmethod
    def summary(cls):
        torch.cuda.synchronize()
        out = {}
        for cat, recs in cls.records.items():
            ms = sum(a.elapsed_time(b) for a, b, _, _ in recs)
            out[cat] = {"calls": len(recs), "ms": ms, "bytes": float(sum(r[2] for r in recs)),
                        "launches": int(sum(r[3] for r in recs))}
        return out


def init(device=None):
    """Select the CUDA device and allocate the reduction workspace."""
    lib = _lib.load()
    if not torch.cuda.is_available():
        raise _lib.EigdNativeError("eigd_b200: no CUDA device visible (there is no CPU fallback)")
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device())
    device = torch.device(device)
    if _State.ready and _State.device == device:
        return device
    torch.cuda.set_device(device)
    _State.device = device
    _State.stream = None
    nwork = lib.eigd_gemm_tn_workspace(32, 32)
    _State.work = torch.empty(int(nwork), dtype=F64, device=device)
    _State.ready = True
    _bind_stream()
    return device


def _bind_stream():
    """The native kernels launch on the stream bound with eigd_set_stream; the torch ops interleaved with them
    (copies, clones, event records, NCCL) follow torch's CURRENT stream.  Re-bind whenever the two differ, so that a
    caller working under ``torch.cuda.stream(s)`` gets one consistent order instead of a race."""
    cur = torch.cuda.current_stream(_State.device).cuda_stream
    if cur != _State.stream:
        check(_lib.load().eigd_set_stream(ctypes.c_void_p(cur)), "set_stream")
        _State.stream = cur


def dev():
    """The selected device; every device-side helper of the package passes through here (or through ``empty`` /
    ``zeros`` / ``to_device``) before it launches, which keeps the native stream bound to torch's current one."""
    if not _State.ready:
        init()
    else:
        _bind_stream()
    return _State.device


def solve_timing_begin():
    check(_lib.load().eigd_solve_timing_begin(), "solve_timing_begin")


def solve_timing_end():
    """-> {k: (calls, total ms)} for every solve launch since solve_timing_begin (CUDA events, native side)."""
    calls = (ctypes.c_int64 * 33)()
    ms = (ctypes.c_double * 33)()
    check(_lib.load().eigd_solve_timing_end(ctypes.cast(calls, ctypes.c_void_p), ctypes.cast(ms, ctypes.c_void_p)),
          "solve_timing_end")
    return {k: (int(calls[k]), float(ms[k])) for k in range(33) if calls[k]}


_DMMA_PEAK = {}


def dmma_peak_tflops():
    """Measured FP64 tensor-pipe peak (TFLOP/s) of the current device (eigd_dmma_peak; cached per device)."""
    d = dev()
    if d not in _DMMA_PEAK:
        out = ctypes.c_double(0.0)
        check(_lib.load().eigd_dmma_peak(4096, 3, ctypes.byref(out)), "dmma_peak")
        _DMMA_PEAK[d] = float(out.value)
    return _DMMA_PEAK[d]


def launch_count():
    return int(_lib.load().eigd_launch_count())


# Host <-> device copies of the numpy API.  Arrays of a megabyte or more travel through page-locked memory:
# uploads are staged (host copy into a block of torch's caching pinned allocator -- or not at all
# when the caller's array already is page-locked, see ``pinned_empty``) and issued on a copy stream, so that they
# overlap kernels already queued on the compute stream (the factorisation while K and M upload); downloads land
# in a pinned block that the returned numpy array views directly (no second host copy).
_BIG_COPY = 1 << 20


class _Copy:
    stream = None
    pending = []        # events of uploads issued straight from the caller's page-locked arrays (see drain_uploads)


def _copy_stream():
    if _Copy.stream is None:
        _Copy.stream = torch.cuda.Stream(device=dev())
    return _Copy.stream


def pinned_empty(shape, dtype=np.float64):
    """numpy array in page-locked host memory (uploads from it skip the staging copy)."""
    dev()
    t = torch.empty(tuple(int(v) for v in np.atleast_1d(shape)), dtype=torch.from_numpy(np.empty(0, dtype=dtype)).dtype,
                    pin_memory=True)
    return t.numpy()


COPY_STATS = {}     # developer counters: piece -> [calls, seconds, bytes] (tools/prof_e2e.py prints them)


def _stat(key, t0, nbytes):
    c = COPY_STATS.setdefault(key, [0, 0.0, 0])
    c[0] += 1
    c[1] += time.perf_counter() - t0
    c[2] += nbytes


def h2d(a):
    """contiguous numpy array -> CUDA tensor of the same dtype, ordered before later work on the current stream."""
    d = dev()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")            # read-only numpy arrays: we only read
        if a.nbytes < _BIG_COPY:
            return torch.as_tensor(a, device=d)
        src = torch.from_numpy(a)
    own = src.is_pinned()
    if own:
        stage = src
    else:
        t0 = time.perf_counter()
        stage = torch.empty(src.shape, dtype=src.dtype, pin_memory=True)
        _stat("h2d pinned block", t0, 0)
        t0 = time.perf_counter()
        # single-threaded on purpose: inside a gradient step this host copies cold data at about 10 GB/s whatever
        # the thread count (4 Python threads: 9.5 vs 9.1 ms per 96 MB), and torch's OpenMP copy_ fell to 2.6-6 GB/s
        # there (104 GB/s in a cache-warm microbenchmark, tools/time_copies.py)
        np.copyto(stage.numpy(), a)
        _stat("h2d staging copy", t0, a.nbytes)
    t0 = time.perf_counter()
    cs, main = _copy_stream(), torch.cuda.current_stream(d)
    with torch.cuda.stream(cs):
        out = stage.to(d, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(cs)
    main.wait_event(ev)
    out.record_stream(main)
    _stat("h2d issue", t0, a.nbytes)
    if own:
        # the DMA reads the caller's own page-locked array: it must have finished before control returns to the
        # caller (who may overwrite the array) -- not before this function returns.  The public entry points drain
        # the list on their way out (drain_uploads), so the host keeps enqueueing kernels meanwhile.
        _Copy.pending.append(ev)
    return out


def drain_uploads():
    """Wait for the uploads that read the caller's page-locked arrays directly (called by every public entry point
    before it returns; a no-op when nothing is pending)."""
    if _Copy.pending:
        t0 = time.perf_counter()
        for ev in _Copy.pending:
            ev.synchronize()
        _stat("h2d wait (caller's pinned arrays, at API exit)", t0, 0)
        _Copy.pending.clear()


def d2h(t):
    """CUDA tensor -> numpy array (same strides for dense tensors, as ``Tensor.cpu``)."""
    t = t.detach()
    if not t.is_cuda or t.numel() * t.element_size() < _BIG_COPY:
        t0 = time.perf_counter()
        out = t.cpu().numpy()
        _stat("d2h small (.cpu, includes waiting for the GPU)", t0, out.nbytes)
        if t.is_cuda:
            _Copy.pending.clear()       # the compute stream waited for every earlier upload and has just been drained
        return out
    t0 = time.perf_counter()
    stage = torch.empty_like(t, device="cpu", pin_memory=True)
    _stat("d2h pinned block", t0, 0)
    t0 = time.perf_counter()
    stage.copy_(t, non_blocking=True)
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(t.device))
    _stat("d2h issue", t0, 0)
    t0 = time.perf_counter()
    ev.synchronize()
    _stat("d2h wait (includes waiting for the GPU)", t0, stage.numel() * stage.element_size())
    _Copy.pending.clear()               # (as above)
    return stage.numpy()


def to_device(x, dtype=F64):
    """numpy / torch -> CUDA tensor (no copy if already there)."""
    d = dev()
    if isinstance(x, torch.Tensor):
        return x.to(device=d, dtype=dtype)
    return h2d(np.ascontiguousarray(x)).to(dtype)


def empty(*shape):
    return torch.empty(*shape, dtype=F64, device=dev())


def zeros(*shape):
    return torch.zeros(*shape, dtype=F64, device=dev())


def _as2d(x):
    if x.dim() == 1:
        return x.unsqueeze(1)
    if x.dim() != 2:
        raise ValueError("expected a 1-D or 2-D tensor")
    return x


def _chk(x, name="operand"):
    if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == F64):
        raise TypeError("%s must be a CUDA float64 tensor" % name)
    return x


# ------------------------------------------------------------------------------------------
# sparse matrices
# ------------------------------------------------------------------------------------------
class CsrDevice:
    """CSR matrix resident in HBM (int32 structure, fp64 values)."""

    def __init__(self, indptr, indices, data, shape):
        d = dev()
        self.shape = tuple(int(s) for s in shape)
        self.indptr = torch.as_tensor(np.ascontiguousarray(indptr, dtype=np.int32), device=d) \
            if not isinstance(indptr, torch.Tensor) else indptr.to(device=d, dtype=torch.int32)
        self.indices = torch.as_tensor(np.ascontiguousarray(indices, dtype=np.int32), device=d) \
            if not isinstance(indices, torch.Tensor) else indices.to(device=d, dtype=torch.int32)
        self.data = to_device(data)
        self.nnz = int(self.indices.numel())
        self.dtype = np.dtype(np.float64)

    @classmethod
    def from_scipy(cls, A, symmetric=False):
        """scipy sparse -> device CSR.  The int32 structure goes through PatternCache (uploaded once per
        pattern).  symmetric=True: a CSC matrix is taken as the CSR of its transpose (= itself)."""
        import scipy.sparse as sp
        if not (sp.issparse(A) and (A.format == "csr" or (symmetric and A.format == "csc"))):
            A = sp.csr_matrix(A)
        if not A.has_sorted_indices:
            A = A.sorted_indices()
        indptr = np.ascontiguousarray(A.indptr, dtype=np.int32)
        indices = np.ascontiguousarray(A.indices, dtype=np.int32)
        eid, ip_d, ix_d, fresh = PatternCache.get(indptr, indices)
        out = cls(ip_d, ix_d, A.data, A.shape)
        out.pattern_id = eid
        out.pattern_host = (indptr, indices)
        out.uploaded_bytes = A.nnz * 8 + ((A.nnz * 4 + (A.shape[0] + 1) * 4) if fresh else 0)
        return out

    def with_values(self, data):
        out = object.__new__(CsrDevice)
        out.shape, out.indptr, out.indices, out.nnz, out.dtype = self.shape, self.indptr, self.indices, self.nnz, self.dtype
        out.data = _chk(data, "values")
        out.pattern_id = getattr(self, "pattern_id", None)
        out.pattern_host = getattr(self, "pattern_host", None)
        return out

    def spmm(self, X, out=None, alpha=1.0, beta=0.0):
        """out = alpha * A @ X + beta * out"""
        X2 = _as2d(_chk(X, "X"))
        n, k = self.shape[0], X2.shape[1]
        if X2.shape[0] != self.shape[1]:
            raise ValueError("dimension mismatch in spmm")
        if out is None:
            out = empty(n, k) if X.dim() == 2 else empty(n)
            beta = 0.0
        Y2 = _as2d(_chk(out, "out"))
        tok = Timeline.begin("spmm")
        check(_lib.load().eigd_csr_spmm(n, _ptr(self.indptr), _ptr(self.indices), _ptr(self.data),
                                        _ptr(X2), X2.stride(0), X2.stride(1), _ptr(Y2), Y2.stride(0), Y2.stride(1),
                                        k, float(alpha), float(beta)), "csr_spmm")
        # algorithmic bytes (SURVEY.md 8d): nnz*12 + (n+1)*4 + 2*n*k*8
        Timeline.end(tok, self.nnz * 12 + (n + 1) * 4 + 2 * n * k * 8, 1)
        return out

    def __matmul__(self, X):
        return self.spmm(X)

    def to_scipy(self):
        import scipy.sparse as sp
        return sp.csr_matrix((self.data.cpu().numpy(), self.indices.cpu().numpy(), self.indptr.cpu().numpy()), shape=self.shape)


def axpby(a, x, b, y, out=None):
    """out = a*x + b*y on flat value arrays (shifted-matrix values)."""
    if out is None:
        out = torch.empty_like(x)
    check(_lib.load().eigd_axpby(x.numel(), float(a), _ptr(x), float(b), _ptr(y) if y is not None else None, _ptr(out)), "axpby")
    return out


# ------------------------------------------------------------------------------------------
# tall-skinny dense ops
# ------------------------------------------------------------------------------------------
def gemm_tn(X, Y, out=None):
    """C = X^T Y  (k1 x k2)"""
    X2, Y2 = _as2d(_chk(X)), _as2d(_chk(Y))
    n, k1, k2 = X2.shape[0], X2.shape[1], Y2.shape[1]
    if Y2.shape[0] != n:
        raise ValueError("dimension mismatch in gemm_tn")
    if out is None:
        out = empty(k1, k2)
    check(_lib.load().eigd_gemm_tn(n, k1, k2, _ptr(X2), X2.stride(0), X2.stride(1), _ptr(Y2), Y2.stride(0), Y2.stride(1),
                                   _ptr(out), out.stride(0), _ptr(_State.work)), "gemm_tn")
    return out


def gemm_nn(X, S, Y, alpha=1.0, beta=0.0):
    """Y = beta*Y + alpha * X @ S, S a small (k1 x k2) device matrix"""
    X2, Y2 = _as2d(_chk(X)), _as2d(_chk(Y))
    S2 = _as2d(_chk(S))
    n, k1, k2 = X2.shape[0], X2.shape[1], Y2.shape[1]
    if S2.shape != (k1, k2) or Y2.shape[0] != n:
        raise ValueError("dimension mismatch in gemm_nn: X %s S %s Y %s" % (tuple(X2.shape), tuple(S2.shape), tuple(Y2.shape)))
    if S2.stride(1) != 1 and S2.shape[1] != 1:
        S2 = S2.contiguous()
    lds = S2.stride(0) if S2.shape[0] > 1 else max(k2, 1)
    check(_lib.load().eigd_gemm_nn(n, k1, k2, float(alpha), _ptr(X2), X2.stride(0), X2.stride(1), _ptr(S2), lds,
                                   float(beta), _ptr(Y2), Y2.stride(0), Y2.stride(1)), "gemm_nn")
    return Y


def col_dot(X, Y, out=None):
    X2, Y2 = _as2d(_chk(X)), _as2d(_chk(Y))
    n, k = X2.shape
    if out is None:
        out = empty(k)
    check(_lib.load().eigd_col_dot(n, k, _ptr(X2), X2.stride(0), X2.stride(1), _ptr(Y2), Y2.stride(0), Y2.stride(1),
                                   _ptr(out), _ptr(_State.work)), "col_dot")
    return out


def mgs_sweep(w, Ws, Hs):
    """Modified Gram-Schmidt of the columns of w (n, k) against the blocks Ws in the order given, coefficients of
    block t into Hs[t] (k doubles): one cooperative launch instead of a dot / axpy pair per block."""
    j = len(Ws)
    if j == 0:
        return w
    n, k = w.shape
    flat = k <= 64 and w.is_contiguous() and all(tuple(W.shape) == (n, k) and W.is_contiguous() for W in Ws) \
        and all(h.numel() == k and h.is_contiguous() for h in Hs)
    if not flat:
        for W, h in zip(Ws, Hs):
            col_dot(w, W, out=h)
            col_axpy(w, h, W, sign=-1.0)
        return w
    _chk(w)
    Wp = (ctypes.c_void_p * j)(*[_chk(W).data_ptr() for W in Ws])
    Hp = (ctypes.c_void_p * j)(*[_chk(h).data_ptr() for h in Hs])
    check(_lib.load().eigd_mgs_sweep(n, k, j, ctypes.cast(Wp, ctypes.c_void_p), ctypes.cast(Hp, ctypes.c_void_p),
                                     _ptr(w), _ptr(_State.work)), "mgs_sweep")
    return w


def col_axpy(Y, s, X, sign=1.0):
    """Y[:, c] += sign * s[c] * X[:, c]"""
    X2, Y2 = _as2d(_chk(X)), _as2d(_chk(Y))
    n, k = Y2.shape
    check(_lib.load().eigd_col_axpy(n, k, float(sign), _ptr(_chk(s, "s")), _ptr(X2), X2.stride(0), X2.stride(1),
                                    _ptr(Y2), Y2.stride(0), Y2.stride(1)), "col_axpy")
    return Y


def col_scale(X, s, mode=0):
    """mode 0: X *= s ; 1: X /= s ; 2: X /= sqrt(s)   (per column, s on device)"""
    X2 = _as2d(_chk(X))
    n, k = X2.shape
    check(_lib.load().eigd_col_scale(n, k, int(mode), _ptr(_chk(s, "s")), _ptr(X2), X2.stride(0), X2.stride(1)), "col_scale")
    return X


def copy2d(src, dst):
    S2, D2 = _as2d(_chk(src)), _as2d(_chk(dst))
    if S2.shape != D2.shape:
        raise ValueError("shape mismatch in copy2d")
    n, k = S2.shape
    check(_lib.load().eigd_copy2d(n, k, _ptr(S2), S2.stride(0), S2.stride(1), _ptr(D2), D2.stride(0), D2.stride(1)), "copy2d")
    return dst


def project(U, V, X):
    """Oblique projection X <- X - U (V^T X)   (reference _project, eigenvector_derivatives.py:26-30).
    (A single cooperative launch for the whole projection was measured slower than these two products -- 68 vs
    52 us at C2 -- and removed; profiles/r1_sibk_step_kernels_ab.txt.)"""
    t = gemm_tn(V, X)
    gemm_nn(U, t, X, alpha=-1.0, beta=1.0)
    return X


# ------------------------------------------------------------------------------------------
# symbolic analysis + numeric factorisation
# ------------------------------------------------------------------------------------------
_SYM_NAMES = ["perm", "parent", "sn_first", "sn_rowptr", "sn_rows", "sn_parent", "sn_level",
              "front_off", "rel", "colcount", "level_ptr", "level_sn"]
_QUERY = {"n": 0, "nsuper": 1, "nlevels": 2, "nnzL": 3, "front_doubles": 4, "sum_front": 5,
          "max_front": 6, "max_cols": 7, "flops": 8, "exact_nnzL": 9}
_QUERY_MORE = {"pool_doubles": 10}      # answered by ``query``, not listed by ``stats``


class Symbolic:
    """Host-side symbolic analysis of a symmetric CSR pattern (works without a GPU)."""

    def __init__(self, indptr, indices, n, coords=None, dof_per_node=1, opts=None):
        lib = _lib.load()
        self.n = int(n)
        self._indptr = np.ascontiguousarray(indptr, dtype=np.int32)
        self._indices = np.ascontiguousarray(indices, dtype=np.int32)
        h = ctypes.c_void_p()
        cptr, dim = None, 0
        if coords is not None:
            coords = np.ascontiguousarray(coords, dtype=np.float64)
            dim = coords.shape[1]
            cptr = coords.ctypes.data_as(ctypes.c_void_p)
        optr = None
        if opts is not None:
            o = list(opts) + [0] * (8 - len(opts))
            oarr = (ctypes.c_int * 8)(*o)
            optr = ctypes.cast(oarr, ctypes.c_void_p)
        check(lib.eigd_symbolic_create(self.n, self._indptr.ctypes.data_as(ctypes.c_void_p),
                                       self._indices.ctypes.data_as(ctypes.c_void_p), cptr, dim, int(dof_per_node),
                                       optr, ctypes.byref(h)), "symbolic_create")
        self.handle = h
        self._dmap_cache = {}

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                _lib.load().eigd_symbolic_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def query(self, name):
        return int(_lib.load().eigd_symbolic_query(self.handle, _QUERY[name] if name in _QUERY else _QUERY_MORE[name]))

    def stats(self):
        return {k: self.query(k) for k in _QUERY}

    def get(self, name):
        lib = _lib.load()
        which = _SYM_NAMES.index(name)
        cnt = lib.eigd_symbolic_get(self.handle, which, None, 0)
        out = np.zeros(cnt, dtype=np.int64)
        lib.eigd_symbolic_get(self.handle, which, out.ctypes.data_as(ctypes.c_void_p), cnt)
        return out

    def arrays(self):
        return {nm: self.get(nm) for nm in _SYM_NAMES}

    def pool_offsets(self):
        """Offset (doubles) of every front in the pooled front workspace of ``query("pool_doubles")`` doubles."""
        lib = _lib.load()
        cnt = lib.eigd_symbolic_get(self.handle, 12, None, 0)
        out = np.zeros(cnt, dtype=np.int64)
        lib.eigd_symbolic_get(self.handle, 12, out.ctypes.data_as(ctypes.c_void_p), cnt)
        return out

    def pool_scatter(self, d_map):
        """The entry lists of the pooled factorisation (eigd_factor_numeric_pool) for the assembly map ``d_map``: (seg,
        ent), ent an (m, 2) int32 device tensor of (CSR index, slot inside its front) grouped by front and sorted by slot,
        seg the int64 start of every front's group.  Built once per map and kept with it."""
        cached = getattr(self, "_pool_scatter", None)
        if cached is not None and cached[0] is d_map:
            return cached[1], cached[2]
        d = dev()
        slots, idx = torch.sort(d_map)
        keep = slots >= 0                                  # -1: the strict upper triangle of the CSR
        slots, idx = slots[keep], idx[keep]
        if not hasattr(self, "_front_off_d"):
            self._front_off_d = torch.as_tensor(self.get("front_off"), device=d)
        fo = self._front_off_d
        seg = torch.searchsorted(slots, fo)
        front = torch.searchsorted(fo, slots, right=True) - 1
        ent = torch.stack([idx.to(torch.int32), (slots - fo[front]).to(torch.int32)], dim=1).contiguous()
        self._pool_scatter = (d_map, seg, ent)
        return seg, ent

    def assembly_map_host(self, indptr=None, indices=None):
        ip = self._indptr if indptr is None else np.ascontiguousarray(indptr, dtype=np.int32)
        ix = self._indices if indices is None else np.ascontiguousarray(indices, dtype=np.int32)
        out = np.zeros(len(ix), dtype=np.int64)
        check(_lib.load().eigd_symbolic_assembly_map_host(self.handle, self.n, ip.ctypes.data_as(ctypes.c_void_p),
                                                          ix.ctypes.data_as(ctypes.c_void_p),
                                                          out.ctypes.data_as(ctypes.c_void_p)), "assembly_map_host")
        return out

    def assembly_map_device(self, d_indptr, d_indices):
        """CSR nz -> front slot, computed by the CUDA integer kernel."""
        out = torch.empty(d_indices.numel(), dtype=torch.int64, device=dev())
        check(_lib.load().eigd_symbolic_assembly_map_device(self.handle, self.n, _ptr(d_indptr), _ptr(d_indices), _ptr(out)),
              "assembly_map_device")
        return out


def pattern_key(indptr, indices, extra=b""):
    h = hashlib.blake2b(digest_size=16)
    h.update(np.ascontiguousarray(indptr).view(np.uint8))
    h.update(np.ascontiguousarray(indices).view(np.uint8))
    h.update(extra)
    return h.hexdigest()


def _same_ints(a, b):
    """Full element-wise equality of two contiguous int32 arrays (torch's vectorised compare: about a third of the
    time of numpy.array_equal at 9 MB, no temporary)."""
    if a.shape != b.shape:
        return False
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")            # read-only numpy arrays: we only read
        return bool(torch.equal(torch.from_numpy(a), torch.from_numpy(b)))


class PatternCache:
    """Device copies of CSR structures (indptr, indices), shared by every matrix with that pattern.

    K, M and K - sigma*M of one design -- and of every later design on the same mesh -- have identical
    patterns (examples/natural_frequency.py:94-104,157,233), so the int32 structure is uploaded once and
    only the fp64 values travel per matrix.  Look-up: a cheap fingerprint (sizes + strided sums) selects the
    candidates, a FULL comparison against the cached host copy confirms the hit -- always: a sampled fingerprint
    or the identity of the caller's array objects proves nothing about arrays that may have been edited in place.
    Entry ids come from a counter (never from ``id()``: CPython recycles addresses of dead arrays)."""
    _entries = {}
    _next_id = 0

    @staticmethod
    def _fingerprint(indptr, indices):
        return (len(indptr), len(indices), int(indptr[::61].sum()), int(indices[::127].sum()),
                int(indices[: 64].sum()), int(indices[-64:].sum()))

    @classmethod
    def get(cls, indptr, indices):
        """-> (entry id, device indptr, device indices, fresh); arrays must be int32, contiguous, sorted rows."""
        fp = cls._fingerprint(indptr, indices)
        for ent in cls._entries.get(fp, []):
            if _same_ints(ent[1], indptr) and _same_ints(ent[2], indices):
                return ent[0], ent[3], ent[4], False
        if sum(len(v) for v in cls._entries.values()) > 16:
            cls._entries.clear()
        cls._next_id += 1
        eid = "p%d" % cls._next_id
        ent = (eid, indptr.copy(), indices.copy(), h2d(indptr), h2d(indices))
        cls._entries.setdefault(fp, []).append(ent)
        return eid, ent[3], ent[4], True


PIVOTING_MODES = ("static", "bunch-kaufman")
FRONTS_MODES = ("resident", "pooled")


def check_fronts(fronts, who="fronts"):
    if fronts not in FRONTS_MODES:
        raise ValueError("%s must be one of %s, not %r" % (who, FRONTS_MODES, fronts))
    return fronts


class Factor:
    """Numeric LDL^T on the device for a fixed symbolic analysis.

    pivoting: "static" (no pivot search; a pivot below 1e-11 max|A| is perturbed to +-that threshold) or
    "bunch-kaufman" (restricted Bunch-Kaufman 1x1 / 2x2 pivoting inside every 32-column pivot block, for indefinite
    matrices with tiny or zero diagonal entries; pivots that are still tiny are perturbed and counted as well).

    fronts: "resident" (one dense front per supernode kept in the factor's workspace for its whole life) or "pooled"
    (the workspace holds no fronts; ``numeric`` borrows a pool of ``symbolic.query("pool_doubles")`` doubles from
    torch's caching allocator for the duration of the call, laid out by front lifetimes, so it is many times smaller
    and factors of one pattern take turns on it).  Both give the same factor bit for bit; "pooled" launches the
    inverse and panel kernels once per tree level instead of once, which costs time on small models."""

    def __init__(self, symbolic, max_rhs=32, pivoting="static", fronts="resident"):
        if pivoting not in PIVOTING_MODES:
            raise ValueError("pivoting must be one of %s, not %r" % (PIVOTING_MODES, pivoting))
        check_fronts(fronts)
        dev()
        self.sym = symbolic
        self.n = symbolic.n
        h = ctypes.c_void_p()
        lib = _lib.load()
        mode = FRONTS_MODES.index(fronts)
        nbytes = int(lib.eigd_factor_workspace_bytes_fronts(symbolic.handle, int(max_rhs), mode))
        if nbytes < 0:
            check(1, "factor_workspace_bytes")
        # torch owns the memory: the caching allocator recycles it when this factor is dropped
        self._workspace = torch.empty(nbytes, dtype=torch.uint8, device=dev())
        check(lib.eigd_factor_create_in_fronts(symbolic.handle, int(max_rhs), mode, _ptr(self._workspace), nbytes,
                                               ctypes.byref(h)), "factor_create_in")
        self.handle = h
        self.fronts = fronts
        self.max_rhs = int(max_rhs)
        self.pivoting = pivoting
        self.refine, self._refine_mat, self._refine_work, self._refine_cols = 0, None, None, 0
        if pivoting != "static":
            check(lib.eigd_factor_set_pivoting(h, PIVOTING_MODES.index(pivoting)), "factor_set_pivoting")

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                _lib.load().eigd_factor_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def numeric(self, d_vals, d_map):
        tok = Timeline.begin("factor")
        l0 = launch_count()
        if self.fronts == "resident":
            check(_lib.load().eigd_factor_numeric(self.handle, d_vals.numel(), _ptr(_chk(d_vals)), _ptr(d_map)), "factor_numeric")
        else:
            seg, ent = self.sym.pool_scatter(d_map)
            pool = torch.empty(self.pool_bytes(), dtype=torch.uint8, device=dev())
            check(_lib.load().eigd_factor_numeric_pool(self.handle, d_vals.numel(), _ptr(_chk(d_vals)), _ptr(seg), _ptr(ent),
                                                       _ptr(pool), pool.numel()), "factor_numeric_pool")
            del pool            # back to the caching allocator, stream-ordered after the kernels just queued
        Timeline.end(tok, 0, launch_count() - l0)
        return self

    def pool_bytes(self):
        """Bytes of the front pool a pooled ``numeric`` borrows (0 for resident fronts)."""
        return 8 * self.sym.query("pool_doubles") if self.fronts == "pooled" else 0

    def solve_bytes(self, k):
        """Algorithmic bytes of one forward+backward sweep with k right-hand sides (SURVEY.md 8d):
        2*(nnz(L)*8 + idx(L)) + n*8 + 4*n*k*8, idx(L) = the supernodal row lists (int32)."""
        if not hasattr(self, "_sb"):
            self._sb = (self.sym.query("nnzL"), self.sym.query("sum_front") - self.n)
        nnzL, nidx = self._sb
        return 2 * (nnzL * 8 + nidx * 4) + self.n * 8 + 4 * self.n * k * 8

    def info(self):
        out = (ctypes.c_int64 * 3)()
        lib = _lib.load()
        check(lib.eigd_factor_info(self.handle, ctypes.cast(out, ctypes.c_void_p)), "factor_info")
        pc = (ctypes.c_int64 * 2)()
        check(lib.eigd_factor_pivot_counts(self.handle, ctypes.cast(pc, ctypes.c_void_p)), "factor_pivot_counts")
        return {"negative_pivots": int(out[0]), "perturbed_pivots": int(out[1]), "non_finite": int(out[2]),
                "two_by_two_pivots": int(pc[0]), "interchanges": int(pc[1])}

    def nbytes(self):
        return int(_lib.load().eigd_factor_bytes(self.handle))

    def set_refinement(self, steps, mat, k=1):
        """The refined solves (``solve(refined=True)``, the Lanczos extends) add ``steps`` rounds of iterative refinement
        x += F(b - mat x), ``mat`` the CsrDevice this factor factorised; the scratch they need, 2 n k doubles owned
        here, grows to the widest k asked for."""
        if steps and k > self._refine_cols:
            self._refine_work, self._refine_cols = torch.empty(2 * self.n * k, dtype=F64, device=dev()), k
        self.refine, self._refine_mat = int(steps), mat
        check(_lib.load().eigd_factor_set_refinement(self.handle, self.refine, _ptr(mat.indptr), _ptr(mat.indices),
                                                     _ptr(mat.data), _ptr(self._refine_work), self._refine_cols),
              "factor_set_refinement")

    def solve(self, B, out=None, refined=False):
        """out = (L D L^T)^{-1} B for a (n,) or (n, k) device tensor; out may alias B.  refined: followed by the
        refinement steps of ``set_refinement``."""
        B2 = _as2d(_chk(B, "B"))
        if B2.shape[0] != self.n:
            raise ValueError("dimension mismatch in solve")
        if out is None:
            out = torch.empty_like(B)
        X2 = _as2d(_chk(out, "out"))
        k = B2.shape[1]
        steps = self.refine if refined else 0
        if steps and k > self._refine_cols:
            self.set_refinement(steps, self._refine_mat, k)
        name = "eigd_factor_apply" if refined else "eigd_factor_solve"
        tok = Timeline.begin("solve")
        l0 = launch_count() if tok else 0
        check(getattr(_lib.load(), name)(self.handle, _ptr(B2), B2.stride(0), B2.stride(1), _ptr(X2), X2.stride(0),
                                         X2.stride(1), k), name)
        if tok:                             # steps + 1 sweeps and steps SpMMs with the factorised matrix (as CsrDevice.spmm)
            spmm = self._refine_mat.nnz * 12 + (self.n + 1) * 4 + 2 * self.n * k * 8 if steps else 0
            Timeline.end(tok, (steps + 1) * self.solve_bytes(k) + steps * spmm, launch_count() - l0)
        return out


def lanczos_extend(op, Bip, Vt, BVt, j0, j1, w, h, g, ab):
    """Steps j0 .. j1-1 of the shift-and-invert Lanczos recurrence on the device (csrc/krylov.cu).

    op: SpLuOperator (its factor applies the refinement it registered); Bip: CsrDevice of the inner product;
    Vt, BVt: (ncv + 1, n) row-major bases; w: (n,); h, g: (ncv + 1,); ab: (2, ncv + 1) [alpha; beta^2]."""
    n = Vt.shape[1]
    for t in (Vt, BVt, w, h, g, ab):
        _chk(t)
    if not (Vt.is_contiguous() and BVt.is_contiguous() and ab.is_contiguous() and w.is_contiguous()):
        raise ValueError("lanczos_extend needs contiguous row-major bases")
    op.lu.set_refinement(op.refine, op.mat, 1)    # reading op.refine settles the depth; scratch for one column
    tok = Timeline.begin("lanczos")
    l0 = launch_count() if tok else 0
    check(_lib.load().eigd_lanczos_extend(op.lu.handle, n, _ptr(Bip.indptr), _ptr(Bip.indices), _ptr(Bip.data), _ptr(Vt),
                                          _ptr(BVt), Vt.stride(0), int(j0), int(j1), _ptr(w), _ptr(h), _ptr(g), _ptr(ab),
                                          ab.stride(0), _ptr(_State.work)), "lanczos_extend")
    nsteps = int(j1) - int(j0)
    op.count += nsteps                      # one operator application per step, as SpLuOperator counts them
    if tok:
        Timeline.end(tok, 0, launch_count() - l0)


def block_lanczos_start(Bip, Vt, BVt, P, scratch):
    """B-orthonormalise the P start vectors Vt[:P] in place, BVt[:P] = B Vt[:P] (csrc/block_krylov.cu)."""
    n = Vt.shape[1]
    check(_lib.load().eigd_block_lanczos_start(n, int(P), _ptr(Bip.indptr), _ptr(Bip.indices), _ptr(Bip.data), _ptr(Vt), _ptr(BVt),
                                               Vt.stride(0), _ptr(scratch), _ptr(_State.work)), "block_lanczos_start")


def block_lanczos_extend(op, Bip, Vt, BVt, P, j0, m0, ncv, Ablk, Rblk, H1, H2, scratch):
    """Block steps j0, j0 + P, ... < ncv of the shift-and-invert block Lanczos recurrence on the device.

    op: SpLuOperator; Bip: CsrDevice of the inner product; Vt, BVt: (ncv + P, n) row-major bases holding m0 vectors;
    Ablk, Rblk: (nsteps, P, P) device outputs (diagonal / sub-diagonal blocks of the projected operator)."""
    n = Vt.shape[1]
    for t in (Vt, BVt, Ablk, Rblk, H1, H2, scratch):
        _chk(t)
    if not (Vt.is_contiguous() and BVt.is_contiguous()):
        raise ValueError("block_lanczos_extend needs contiguous row-major bases")
    op.lu.set_refinement(op.refine, op.mat, P)    # reading op.refine settles the depth; scratch for P columns
    tok = Timeline.begin("lanczos")
    l0 = launch_count() if tok else 0
    check(_lib.load().eigd_block_lanczos_extend(op.lu.handle, n, int(P), _ptr(Bip.indptr), _ptr(Bip.indices), _ptr(Bip.data),
                                                _ptr(Vt), _ptr(BVt), Vt.stride(0), int(j0), int(m0), int(ncv), _ptr(Ablk), _ptr(Rblk),
                                                _ptr(H1), _ptr(H2), _ptr(scratch), _ptr(_State.work)), "block_lanczos_extend")
    op.count += int(ncv) - int(j0)          # one operator application per new basis vector, as SpLuOperator counts columns
    if tok:
        Timeline.end(tok, 0, launch_count() - l0)


# ------------------------------------------------------------------------------------------
# element kernels
# ------------------------------------------------------------------------------------------
def q4_quadforms(kind, conn, xy, cmat6, WA, WB, V, dk, dm, sA, sB, out):
    nelems = conn.shape[0]
    N = V.shape[1]
    ldw = V.stride(0)
    for t in (WA, WB):
        if t is not None and (t.stride(0) != ldw or t.stride(1) != 1):
            raise ValueError("WA/WB/V must share one row-major layout")
    if V.stride(1) != 1:
        raise ValueError("V must be row-major")
    check(_lib.load().eigd_q4_quadforms(int(kind), nelems, _ptr(conn), _ptr(xy), _ptr(cmat6), _ptr(WA), _ptr(WB), _ptr(V),
                                        N, ldw, _ptr(dk), _ptr(dm), float(sA), float(sB), _ptr(out)), "q4_quadforms")
    return out


def q4_assemble(kind, conn, xy, ks, ms, cmat6, src_ptr, src, nnz, Kvals, Mvals):
    check(_lib.load().eigd_q4_assemble(int(kind), conn.shape[0], _ptr(conn), _ptr(xy), _ptr(ks), _ptr(ms), _ptr(cmat6),
                                       _ptr(src_ptr), _ptr(src), int(nnz), _ptr(Kvals), _ptr(Mvals)), "q4_assemble")


def element_material(law, par, rho, conn=None, rhoE=None, ks=None, ms=None, dk=None, dm=None):
    """Penalised material factors ks, ms and their derivatives dk, dm of law 0 / 1 / 2 with the four parameters ``par``
    (eigd_q4_material), of the element densities: the mean of the nodal ``rho`` over the element's nodes (``conn``
    (nelems, npe), mean written to ``rhoE``) or, without ``conn``, ``rho`` itself.  Outputs left None are not written."""
    nelems, npe = (conn.shape[0], conn.shape[1]) if conn is not None else (rho.numel(), 4)     # npe unread without conn
    par4 = (ctypes.c_double * 4)(*[float(v) for v in par])
    check(_lib.load().eigd_q4_material(int(law), nelems, npe, _ptr(conn), _ptr(rho), par4, _ptr(rhoE), _ptr(ks), _ptr(ms),
                                       _ptr(dk), _ptr(dm)), "q4_material")


def node_gather(nptr, nelem, evals, scale, out):
    check(_lib.load().eigd_node_gather(out.numel(), _ptr(nptr), _ptr(nelem), _ptr(evals), float(scale), _ptr(out)), "node_gather")
    return out


def dof_gather(nptr, nelem, nlocal, due, out):
    """out[c v + i] = sum over the elements e around node v of due[e, c nlocal + i]: the element terms due (nelems,
    npe * c) gathered to the c = out.numel() / nnodes components of every node."""
    nnodes = nptr.numel() - 1
    ncomp = out.numel() // nnodes
    check(_lib.load().eigd_dof_gather(nnodes, ncomp, due.shape[1] // ncomp, _ptr(nptr), _ptr(nelem), _ptr(nlocal), _ptr(due),
                                      _ptr(out)), "dof_gather")
    return out


def filter_project(rho, beta, eta, g=None):
    """tanh projection of the filtered density ``rho``, or with ``g`` the gradient g * d(projection)/d(rho)."""
    out = empty(rho.shape[0])
    check(_lib.load().eigd_filter_project(rho.shape[0], float(beta), float(eta), _ptr(rho), _ptr(g), _ptr(out)),
          "filter_project")
    return out


# ------------------------------------------------------------------------------------------
# stored unit element matrices (csrc/stored_fe.cu, csrc/h8.cu, csrc/t10.cu)
# ------------------------------------------------------------------------------------------
def h8_element_matrices(conn, X, E, nu, density, K0, M0):
    """Unit stiffness and mass matrices K0, M0 (nelems * 576 each) of the H8 elements ``conn`` (nelems, 8)."""
    check(_lib.load().eigd_h8_element_matrices(conn.shape[0], _ptr(conn), _ptr(X), float(E), float(nu), float(density),
                                               _ptr(K0), _ptr(M0)), "h8_element_matrices")


def h8_thermal_element_matrices(conn, X, K0, M0):
    """Unit conductivity and capacity matrices K0, M0 (nelems * 64 each) of the scalar H8 elements ``conn`` (nelems, 8)."""
    check(_lib.load().eigd_h8_thermal_element_matrices(conn.shape[0], _ptr(conn), _ptr(X), _ptr(K0), _ptr(M0)),
          "h8_thermal_element_matrices")


def t10_element_matrices(conn, X, E, nu, density, K0, M0):
    """Unit stiffness and mass matrices K0, M0 (nelems * 900 each) of the T10 elements ``conn`` (nelems, 10)."""
    check(_lib.load().eigd_t10_element_matrices(conn.shape[0], _ptr(conn), _ptr(X), float(E), float(nu), float(density),
                                                _ptr(K0), _ptr(M0)), "t10_element_matrices")


def t10_thermal_element_matrices(conn, X, K0, M0):
    """Unit conductivity and capacity matrices K0, M0 (nelems * 100 each) of the scalar T10 elements ``conn``
    (nelems, 10)."""
    check(_lib.load().eigd_t10_thermal_element_matrices(conn.shape[0], _ptr(conn), _ptr(X), _ptr(K0), _ptr(M0)),
          "t10_thermal_element_matrices")


def stored_assemble(src_ptr, src, ne, E1, c1, vals, E3=None, c3=None, F1=None, d1=None, vals2=None, F3=None, d3=None):
    """vals = CSR values of the elements c1[e] E1_e (+ c3[e] E3_e) through the (element, a, b) source lists; with
    ``vals2``, the second matrix d1[e] F1_e (+ d3[e] F3_e) on the same pattern in the same pass."""
    check(_lib.load().eigd_stored_assemble(src_ptr.numel() - 1, _ptr(src_ptr), _ptr(src), int(ne), _ptr(E1), _ptr(E3), _ptr(c1),
                                           _ptr(c3), _ptr(vals), _ptr(F1), _ptr(F3), _ptr(d1), _ptr(d3), _ptr(vals2)),
          "stored_assemble")
    return vals


def stored_quadform(dofmap, E1, c1, W, V, out, E3=None, c3=None, F1=None, d1=None, W2=None, s1=1.0, s2=1.0):
    """out[e] = sum_k W_k^T (c1[e] E1_e + c3[e] E3_e) V_k over the element dofs ``dofmap`` (nelems, ne); with the second
    term, s1 * that + s2 * sum_k W2_k^T (d1[e] F1_e) V_k (eigd_stored_quadform).  W, W2, V: (n, N) row-major."""
    ld = V.stride(0)
    for t in (W, W2):
        if t is not None and (t.shape != V.shape or t.stride(0) != ld or t.stride(1) != 1):
            raise ValueError("W / W2 must have the shape and row-major layout of V")
    if V.stride(1) != 1:
        raise ValueError("V must be row-major")
    check(_lib.load().eigd_stored_quadform(dofmap.shape[0], dofmap.shape[1], _ptr(dofmap), _ptr(E1), _ptr(E3), _ptr(c1), _ptr(c3),
                                           _ptr(W), _ptr(V), V.shape[1], ld, _ptr(out), _ptr(F1), _ptr(d1), _ptr(W2), float(s1),
                                           float(s2)), "stored_quadform")
    return out


def segment_sum(seg_ptr, perm, x, scale, out):
    """out[c] = scale * sum of x[perm[i]] over the segment [seg_ptr[c], seg_ptr[c + 1])."""
    check(_lib.load().eigd_segment_sum(seg_ptr.numel() - 1, _ptr(seg_ptr), _ptr(perm), _ptr(x), float(scale), _ptr(out)),
          "segment_sum")
    return out


# ------------------------------------------------------------------------------------------
# linearised buckling (csrc/buckling.cu)
# ------------------------------------------------------------------------------------------
def q4_stress(conn, xy, cmat6, ks, u, sdet):
    check(_lib.load().eigd_q4_stress(conn.shape[0], _ptr(conn), _ptr(xy), _ptr(cmat6), _ptr(ks), _ptr(u), _ptr(sdet)),
          "q4_stress")
    return sdet


def q4_assemble_geometric(conn, xy, sdet, src_ptr, src, nnz, Gvals):
    check(_lib.load().eigd_q4_assemble_geometric(conn.shape[0], _ptr(conn), _ptr(xy), _ptr(sdet), _ptr(src_ptr), _ptr(src),
                                                 int(nnz), _ptr(Gvals)), "q4_assemble_geometric")
    return Gvals


def q4_gderiv(conn, xy, cmat6, W, V, ks, dks, u, sx, out_rho=None, due=None):
    """Fused sensitivities of sum_k w_k^T G(u, x) v_k (W, V: full-dof (2 nnodes, N) row-major)."""
    if W.stride(1) != 1 or V.stride(1) != 1 or W.stride(0) != V.stride(0):
        raise ValueError("W and V must share one row-major layout")
    check(_lib.load().eigd_q4_gderiv(conn.shape[0], _ptr(conn), _ptr(xy), _ptr(cmat6), _ptr(W), _ptr(V), V.shape[1],
                                     V.stride(0), _ptr(ks), _ptr(dks), _ptr(u), float(sx), _ptr(out_rho), _ptr(due)),
          "q4_gderiv")


def h8_stress_stiffness(conn, X, E, nu, kg, dofmap, u, stress, G0):
    """Element stresses kg C B_q u_e (``stress`` (nelems, 8, 6) or None) and the unit stress stiffness G0 (nelems * 576)
    of the H8 solid; ``u`` is read through ``dofmap`` (nelems, 24), -1 = constrained."""
    check(_lib.load().eigd_h8_stress_stiffness(conn.shape[0], _ptr(conn), _ptr(X), float(E), float(nu), _ptr(kg), _ptr(dofmap),
                                               _ptr(u), _ptr(stress), _ptr(G0)), "h8_stress_stiffness")
    return G0


def h8_gderiv_u(conn, X, E, nu, kg, dofmap, W, V, due):
    """due (nelems, 24): the element terms of d/du sum_k w_k^T G(u) v_k (W, V: (n, N) row-major, read through dofmap)."""
    if W.stride(1) != 1 or V.stride(1) != 1 or W.stride(0) != V.stride(0) or W.shape != V.shape:
        raise ValueError("W and V must share one row-major layout")
    check(_lib.load().eigd_h8_gderiv_u(conn.shape[0], _ptr(conn), _ptr(X), float(E), float(nu), _ptr(kg), _ptr(dofmap), _ptr(W),
                                       _ptr(V), V.shape[1], V.stride(0), _ptr(due)), "h8_gderiv_u")
    return due


def expand_rows(idx, red, nfull):
    """full[idx[i], :] = red[i, :], zeros elsewhere (examples/buckling.py full_vector)."""
    r2 = _as2d(red)
    k = r2.shape[1]
    r2 = r2 if r2.is_contiguous() else r2.contiguous()
    full = zeros(nfull, k)
    check(_lib.load().eigd_expand_rows(idx.numel(), k, _ptr(idx), _ptr(r2), _ptr(full)), "expand_rows")
    return full if red.dim() == 2 else full.reshape(-1)


def reduce_rows(idx, full):
    """red[i, :] = full[idx[i], :] (examples/buckling.py reduce_vector)."""
    f2 = _as2d(full)
    k = f2.shape[1]
    f2 = f2 if f2.is_contiguous() else f2.contiguous()
    red = empty(idx.numel(), k)
    check(_lib.load().eigd_reduce_rows(idx.numel(), k, _ptr(idx), _ptr(f2), _ptr(red)), "reduce_rows")
    return red if full.dim() == 2 else red.reshape(-1)
