"""Developer timing of the numeric factorisation at benchmark size (CUDA events).

    python tools/time_factor.py [nx] [resident|pooled]      (front memory of the factor, default resident)"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from eigd_b200 import device as D, topo as T
import eigd_b200 as E
D.init()
nx = int(sys.argv[1]) if len(sys.argv) > 1 else 500
fronts = sys.argv[2] if len(sys.argv) > 2 else "resident"
model = T.make_thermal_model(nx=nx, ny=nx, N=10, m=60, sigma=-0.1, seed=0)
rng = np.random.default_rng(0)
model.x_d = D.to_device(rng.uniform(0.3, 1.0, model.nnodes))
model.prob.set_density(rho=model.fltr.apply(model.x_d))
K, M = model.prob.assemble()
vals = D.axpby(1.0, K.data, 0.1, M.data)
torch.cuda.reset_peak_memory_stats()
f = E.SpLuOperator(K.with_values(vals), coords=model.X, dof_per_node=1, fronts=fronts)
ts = []
for it in range(6):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); f.lu.numeric(vals, f._amap); e1.record(); torch.cuda.synchronize()
    ts.append(e0.elapsed_time(e1))
st = f.symbolic.stats()
print("fronts %s: pool %.3f GB, factor %.3f GB, peak allocated %.3f GB" % (fronts, f.lu.pool_bytes() / 1e9, f.lu.nbytes() / 1e9,
                                                                      torch.cuda.max_memory_allocated() / 1e9))
print("factor: best %.3f ms  median %.3f ms  flops %.2f GF -> %.2f TF/s" % (min(ts), sorted(ts)[len(ts) // 2], st["flops"] / 1e9, st["flops"] / min(ts) / 1e9))
B = torch.randn(K.shape[0], 3, dtype=torch.float64, device="cuda")
X = f.lu.solve(B)
A = K.with_values(vals).to_scipy()
print("resid", np.abs(A @ X.cpu().numpy() - B.cpu().numpy()).max())
