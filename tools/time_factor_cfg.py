"""Developer timing of the numeric factorisation per launch kind (EIGD_FACTOR_PROF=1) on the bench configurations.

    python tools/time_factor_cfg.py [c2|c3|c4] [resident|pooled]      (front memory of the factor, default resident)"""
import os, sys, warnings
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from eigd_b200 import device as D, topo as T, shell as S
D.init()
which = sys.argv[1] if len(sys.argv) > 1 else "c2"
fronts = sys.argv[2] if len(sys.argv) > 2 else "resident"
if which == "c2":
    m = T.make_thermal_model(nx=500, ny=500, N=10, m=60, sigma=-0.1, seed=0, fronts=fronts)
    m.x = np.random.default_rng(0).uniform(0.3, 1.0, m.nnodes)
elif which == "c3":
    m = T.make_buckling_model(nx=352, ny=704, N=20, m=60, sigma=3.0, solver_type="IRAM", fronts=fronts)
else:
    m = S.make_shell_model(nx=408, ny=408, ncx=20, ncy=20, N=20, m=60, fronts=fronts)
with warnings.catch_warnings():
    warnings.simplefilter("ignore")
    m.initialize()
f = m.factor
for it in range(3):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); f.lu.numeric(f.mat.data, f._amap); e1.record(); torch.cuda.synchronize()
    st = f.symbolic.stats()
    print("%s fronts %s: factor %.3f ms  flops %.2f GF -> %.2f TF/s" % (which, fronts, e0.elapsed_time(e1), st["flops"] / 1e9, st["flops"] / e0.elapsed_time(e1) / 1e9), flush=True)
b = torch.randn(f.shape[0], 3, dtype=torch.float64, device="cuda")
x = f.lu.solve(b)
r = f.mat.spmm(x) - b
print("solve residual %.2e" % float(r.abs().max() / b.abs().max()))
