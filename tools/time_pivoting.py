"""C3 (buckling, 497k DOF, sigma = 3) with the static and the restricted Bunch-Kaufman pivoting of the shifted factor
K_r + sigma G_r, alternating in one process after a warm-up of each:

    python tools/time_pivoting.py [--reps 3] [--out FILE]

Per mode: factorisation time (CUDA events around Factor.numeric, best / median of --factor-reps), its split by launch
kind (EIGD_FACTOR_PROF=1, measured in a child process because that switch synchronises after every launch), pivot
counts, probe residuals and the refinement depth SpLuOperator chose, eigensolve / adjoint / time-to-gradient of each
repetition, and the gradient xb against tests/golden/fullsize_c3_noguess.npz.  Prints the card name and power limit of
the same run and one JSON document."""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
MODES = ("static", "bunch-kaufman")


def golden():
    return dict(np.load(os.path.join(ROOT, "tests", "golden", "fullsize_c3_noguess.npz"), allow_pickle=False))


def make_model(g, pivoting):
    from eigd_b200 import topo as T
    return T.make_buckling_model(nx=int(g["nx"]), ny=int(g["ny"]), N=int(g["N"]), m=int(g["m"]), sigma=float(g["sigma"]),
                                 solver_type="IRAM", adjoint_method="sibk", adjoint_options={"lanczos_guess": True},
                                 rtol=1e-12, deriv_type="tensor", pivoting=pivoting)


def gradient(model, g):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.initialize()
    model.initialize_adjoint()
    model.add_eigenvector_aggregate_derivative(1.0, 100.0, int(g["node"]), mode="tanh")
    model.finalize_adjoint()
    torch.cuda.synchronize()
    p = model.profile
    return {"wall_s": time.perf_counter() - t0, "eig_s": p["eigenvalue solve time"], "adjoint_s": p["adjoint solution time"],
            "time_to_gradient_s": model.time_to_gradient(), "eig_solves": p["solve preconditioner count"],
            "adjoint_solves": p["adjoint preconditioner count"]}


def shifted_values(model):
    from eigd_b200 import device as D
    return D.axpby(1.0, model.Kr.data, float(model.sigma), model.Gr.data)


def factor_times(model, reps):
    import torch
    f = model.factor
    vals = shifted_values(model)
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        f.lu.numeric(vals, f._amap)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return ts


def card():
    import torch
    out = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        out["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["nvidia_smi"] = "unavailable: %s" % e
    return out


def factor_prof_child():
    """EIGD_FACTOR_PROF=1 is set by the parent: one warm-up and three profiled factorisations per mode."""
    from eigd_b200 import device as D
    D.init()
    g = golden()
    for mode in MODES:
        model = make_model(g, mode)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model.initialize()
        print("mode %s" % mode, file=sys.stderr, flush=True)
        factor_times(model, 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3, help="timed gradients per mode (after one warm-up each)")
    ap.add_argument("--factor-reps", type=int, default=8)
    ap.add_argument("--out", default=None)
    ap.add_argument("--factor-prof-child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.factor_prof_child:
        factor_prof_child()
        return
    import torch
    from eigd_b200 import device as D
    if not torch.cuda.is_available():
        raise SystemExit("time_pivoting.py needs a CUDA device")
    D.init()
    g = golden()
    res = {"config": "C3 buckling nx=%d ny=%d N=%d sigma=%g" % (int(g["nx"]), int(g["ny"]), int(g["N"]), float(g["sigma"])),
           "card": card(), "modes": {}}
    models = {m: make_model(g, m) for m in MODES}
    for m in MODES:                                                   # warm-up: symbolic analysis, module loads, caches
        gradient(models[m], g)
    runs = {m: [] for m in MODES}
    for _ in range(args.reps):
        for m in MODES:
            runs[m].append(gradient(models[m], g))
    for m in MODES:
        model = models[m]
        f = model.factor
        xb = model.xb.cpu().numpy()
        r = {"reps": runs[m], "n": int(model.prob.nred),
             "time_to_gradient_s_median": float(np.median([x["time_to_gradient_s"] for x in runs[m]])),
             "eig_s_median": float(np.median([x["eig_s"] for x in runs[m]])),
             "adjoint_s_median": float(np.median([x["adjoint_s"] for x in runs[m]])),
             "factor_info": f.info, "refine_steps": f.refine, "probe_unrefined_chosen": f.probe,
             "probe_refined": f.probe_refined, "probe_unrefined": f._probe_residual(),
             "BLF_rel_err": float(np.abs(np.asarray(model.BLF) - g["BLF"]).max() / np.abs(g["BLF"]).max()),
             "xb_rel_err": float(np.abs(xb - g["xb"]).max() / np.abs(g["xb"]).max())}
        res["modes"][m] = r
    for m in MODES:                                                   # factorisation alone, alternating
        res["modes"][m]["factor_ms"] = []
    for _ in range(2):
        for m in MODES:
            res["modes"][m]["factor_ms"] += factor_times(models[m], args.factor_reps // 2)
    for m in MODES:
        ts = res["modes"][m]["factor_ms"]
        res["modes"][m]["factor_ms_best"] = min(ts)
        res["modes"][m]["factor_ms_median"] = float(np.median(ts))
    del models
    torch.cuda.empty_cache()
    env = dict(os.environ, EIGD_FACTOR_PROF="1")
    child = subprocess.run([sys.executable, os.path.abspath(__file__), "--factor-prof-child"], capture_output=True, text=True,
                           env=env, cwd=ROOT)
    lines = [ln for ln in child.stderr.splitlines() if ln.startswith("mode ") or ln.startswith("[factor prof]")]
    res["factor_prof"] = lines if child.returncode == 0 else {"returncode": child.returncode, "stderr": child.stderr[-4000:]}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
