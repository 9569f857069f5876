"""Developer timing of the block-Lanczos step at benchmark size (C2: thermal 500 x 500, P = 2, ncv = 60), CUDA events.

Times one restart cycle of block_lanczos_extend (30 block steps, m = 2 .. 58) and the P-column solve alone; the
difference per step is the Gram-Schmidt / B W / Cholesky-QR work after the solve.  Then single-step calls at several
m (each is the first step after a "restart", so its local pass runs against the whole basis: two full passes).
Bytes are what the algorithm has to move per step: the full pass reads V[0:m] and BV[0:m], the local pass V[lo:m]
and BV[lo:m] (2 P rows), B W reads B and the new block, and V[m:m+P], BV[m:m+P] are stored."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from eigd_b200 import device as D, topo as T
D.init()
import eigd_b200 as E

nx = int(sys.argv[1]) if len(sys.argv) > 1 else 500
P, ncv = 2, 60
model = T.make_thermal_model(nx=nx, ny=nx, N=10, m=ncv, sigma=-0.1, adjoint_options={"lanczos_guess": True}, seed=0)
rng = np.random.default_rng(0)
x_d = D.to_device(rng.uniform(0.3, 1.0, model.nnodes))
model.x_d = x_d
model.rho = model.fltr.apply(x_d); model.prob.set_density(rho=model.rho)
K, M = model.prob.assemble()
f = E.SpLuOperator(K.with_values(D.axpby(1.0, K.data, 0.1, M.data)), coords=model.X, dof_per_node=1)
f.refine                                         # finish the factorisation (and its refinement decision) first
n = K.shape[0]
nnz = int(M.data.numel())
print("n = %d, nnz(B) = %d, P = %d, ncv = %d, refine = %d" % (n, nnz, P, ncv, f.refine))
print(torch.cuda.get_device_name(), flush=True)

Vt, BVt = D.empty(ncv + P, n), D.empty(ncv + P, n)
nsteps = ncv // P
blocks = D.zeros(2, nsteps + 1, P, P)
H1, H2, scratch = D.zeros((ncv + P) * P), D.zeros((ncv + P) * P), D.zeros(3 * P * P)
W0 = D.to_device(rng.uniform(-1.0, 1.0, (P, n)))


def start():
    Vt[:P].copy_(W0)
    D.block_lanczos_start(M, Vt, BVt, P, scratch)


def ev():
    return torch.cuda.Event(enable_timing=True)


def step_bytes(m, lo):
    return 8 * n * (2 * m + 2 * (m - lo) + 2 * P + P) + 12 * nnz + 4 * (n + 1)


# one cycle from the start block: steps j = 0, 2, ..., ncv - 2 (m = j + P)
start()
D.block_lanczos_extend(f, M, Vt, BVt, P, 0, P, ncv, blocks[0], blocks[1], H1, H2, scratch)   # warm-up
cyc = []
for it in range(5):
    start()
    torch.cuda.synchronize()
    e0, e1 = ev(), ev()
    e0.record()
    D.block_lanczos_extend(f, M, Vt, BVt, P, 0, P, ncv, blocks[0], blocks[1], H1, H2, scratch)
    e1.record(); torch.cuda.synchronize()
    cyc.append(e0.elapsed_time(e1))
# the P-column solve alone (column-major operands here, rows of the basis inside the cycle)
Bc = BVt[:P].T.contiguous()
Xc = torch.empty(n, P, dtype=torch.float64, device="cuda")
sol = []
for it in range(5):
    e0, e1 = ev(), ev()
    e0.record()
    for _ in range(nsteps):
        f.lu.solve(Bc, out=Xc)
    e1.record(); torch.cuda.synchronize()
    sol.append(e0.elapsed_time(e1) / nsteps)
tc, ts = min(cyc), min(sol)
per = (tc - nsteps * ts) / nsteps
alg = sum(step_bytes(j + P, 0 if j == 0 else j - P) for j in range(0, ncv, P))
print("cycle (%d steps): %.3f ms (min of %d; all %s)" % (nsteps, tc, len(cyc), " ".join("%.3f" % t for t in cyc)))
print("k = %d solve: %.1f us" % (P, ts * 1e3))
print("non-solve per step: %.1f us; algorithmic bytes per cycle %.2f GB -> %.2f TB/s over the non-solve time"
      % (per * 1e3, alg / 1e9, alg / (tc - nsteps * ts) / 1e9))
# single steps against m (first step after a restart: the local pass is a full pass too)
print("single step at m (local pass = full pass): total us, non-solve us, alg bytes MB, TB/s")
for m in (4, 10, 20, 30, 40, 50, 60):
    j = m - P
    start()
    D.block_lanczos_extend(f, M, Vt, BVt, P, 0, P, m - P, blocks[0], blocks[1], H1, H2, scratch)   # fill V[0:m]
    ts_ = []
    for it in range(5):
        e0, e1 = ev(), ev()
        e0.record()
        D.block_lanczos_extend(f, M, Vt, BVt, P, j, m, m, blocks[0], blocks[1], H1, H2, scratch)
        e1.record(); torch.cuda.synchronize()
        ts_.append(e0.elapsed_time(e1))
    t = min(ts_)
    b = step_bytes(m, 0)
    print("  m = %2d: %7.1f %7.1f %7.1f %6.2f" % (m, t * 1e3, (t - ts) * 1e3, b / 1e6, b / ((t - ts) * 1e-3) / 1e12))
