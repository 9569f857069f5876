"""Developer timing of the triangular solve alone at benchmark size (CUDA events, L2 flushed)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from eigd_b200 import device as D, topo as T
D.init()
nx = int(sys.argv[1]) if len(sys.argv) > 1 else 500
model = T.make_thermal_model(nx=nx, ny=nx, N=10, m=60, sigma=-0.1, adjoint_options={"lanczos_guess": True}, seed=0)
rng = np.random.default_rng(0)
x_d = D.to_device(rng.uniform(0.3, 1.0, model.nnodes))
model.x_d = x_d
model.rho = model.fltr.apply(x_d); model.prob.set_density(rho=model.rho)
K, M = model.prob.assemble()
import eigd_b200 as E
vals = D.axpby(1.0, K.data, 0.1, M.data)
f = E.SpLuOperator(K.with_values(vals), coords=model.X, dof_per_node=1)
n = K.shape[0]
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
Kh = K.with_values(vals).to_scipy()
for k in (1, 2, 4, 10, 16, 20):
    B = torch.randn(n, k, dtype=torch.float64, device="cuda") if k > 1 else torch.randn(n, dtype=torch.float64, device="cuda")
    X = f.lu.solve(B)
    r = Kh @ X.cpu().numpy() - B.cpu().numpy()
    err = np.abs(r).max() / np.abs(B.cpu().numpy()).max()
    ts = []
    for it in range(8):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); f.lu.solve(B, out=X); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts2 = []
    for it in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10): f.lu.solve(B, out=X)
        e1.record(); torch.cuda.synchronize()
        ts2.append(e0.elapsed_time(e1) / 10)
    by = f.lu.solve_bytes(k)
    print("k=%2d  cold %.1f us  warm %.1f us  resid %.1e  alg GB/s cold %.0f warm %.0f" % (k, min(ts) * 1e3, min(ts2) * 1e3, err, by / min(ts) / 1e6, by / min(ts2) / 1e6))
# per-phase profile (CTA 0 timestamps)
import ctypes
from eigd_b200 import _lib
lib = _lib.load()
nph = lib.eigd_solve_num_phases(f.lu.handle)
buf = torch.zeros(nph + 1, dtype=torch.int64, device="cuda")
for k in (1, 2, 4, 10):
    B = torch.randn(n, k, dtype=torch.float64, device="cuda")
    X = torch.empty_like(B)
    lib.eigd_solve_set_phase_times(ctypes.c_void_p(buf.data_ptr()))
    acc = np.zeros(nph)
    for it in range(5):
        f.lu.solve(B, out=X); torch.cuda.synchronize()
        t = buf.cpu().numpy()[: nph + 1]
        if it: acc += np.diff(t) / 4.0
    lib.eigd_solve_set_phase_times(None)
    print("k=%d phase us:" % k, " ".join("%.1f" % (v / 1e3) for v in acc), " total %.1f" % (acc.sum() / 1e3))
# per-tile trace of CTA 0 / warp 0 (clock64 deltas in ns at the SM clock reported by nvidia-smi)
tr = torch.zeros(16 * nph, dtype=torch.int64, device="cuda")
B = torch.randn(n, dtype=torch.float64, device="cuda")
X = torch.empty_like(B)
lib.eigd_solve_set_trace(ctypes.c_void_p(tr.data_ptr()))
for it in range(3):
    f.lu.solve(B, out=X); torch.cuda.synchronize()
lib.eigd_solve_set_trace(None)
t = tr.cpu().numpy().reshape(nph, 16)
print("trace (cycles): phase: wait (of which panel copy) | product | reduce | store | signal | bookkeeping || start-to-start")
prev = 0
for p in range(nph):
    if t[p, 0]:
        print("  %2d: %6d (%5d) %6d %6d %6d %6d %6d   total %6d || %6d" % (
            p, t[p, 1] - t[p, 0], max(t[p, 6] - t[p, 0], 0) if t[p, 6] else 0, t[p, 2] - t[p, 1], t[p, 3] - t[p, 2], t[p, 4] - t[p, 3],
            t[p, 5] - t[p, 4], max(t[p, 7] - t[p, 5], 0) if t[p, 7] else 0, t[p, 5] - t[p, 0], t[p, 0] - prev if prev else 0),
            "| loop top -> dispatch %5d -> tile start %5d" % (t[p, 9] - t[p, 8], t[p, 0] - t[p, 9]) if t[p, 8] and t[p, 9] else "")
        prev = t[p, 0]
# skew of the dependency chain across CTAs (pipelined level kernel, k = 1): %globaltimer of every CTA's first tile per phase
nsm = torch.cuda.get_device_properties(0).multi_processor_count
sk = torch.zeros(nph * nsm * 4, dtype=torch.int64, device="cuda")
lib.eigd_solve_set_skew(ctypes.c_void_p(sk.data_ptr()))
for it in range(3):
    sk.zero_()
    f.lu.solve(B, out=X); torch.cuda.synchronize()
lib.eigd_solve_set_skew(None)
s_ = sk.cpu().numpy().reshape(nph, nsm, 4).astype(np.float64)
print("skew (ns, all CTAs with a tile in the phase): CTAs | dependencies complete: spread (max - min) | signalled - deps complete: min / median / max |"
      " last signal -> first deps complete of the next phase")
prev_last = None
for p in range(nph):
    m = s_[p, :, 3] > 0
    if not m.any():
        prev_last = None
        continue
    dep, sig = s_[p, m, 2], s_[p, m, 3]
    work = sig - dep
    hop = (dep.min() - prev_last) if prev_last else float("nan")
    print("  %2d: %3d | %6.0f | %6.0f %6.0f %6.0f | %6.0f   phase %6.0f" % (p, m.sum(), dep.max() - dep.min(), work.min(), np.median(work),
                                                                  work.max(), hop, sig.max() - dep.min()))
    prev_last = sig.max()
