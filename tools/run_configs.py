"""Full-size runs of the BASELINE.json configurations that are not the bench line (SURVEY.md section 8):

    python tools/run_configs.py c3 [--nx 352 --ny 704 --modes 20]     buckling, ~497k DOF, 20 modes
    python tools/run_configs.py c5 [--designs 8]                      design sweep, 202k-DOF natural-frequency mesh
    python tools/run_configs.py c4 [--nx 408 --ny 408 --modes 20 --fd]   1M-DOF synthetic shell (6 dof/node), crm.py driver
    python tools/run_configs.py h8 [--nx 64 --ny 32 --nz 32 --modes 10 --fd]   free 3-D solid of hexahedra (3 dof/node)
    python tools/run_configs.py h8buck [--nx 32 --ny 24 --nz 128 --modes 10 --fd]   buckling of a clamped 3-D column
    python tools/run_configs.py h8thermal [--nx 80 --ny 64 --nz 48 --modes 10 --ftype spatial|helmholtz --fd]
                                                                       heat conduction in an insulated 3-D box (1 dof/node)
    python tools/run_configs.py t10 [--nx 32 --ny 16 --nz 16 --modes 10 --fd]   the h8 solid on quadratic tetrahedra
    python tools/run_configs.py t10thermal [--nx 40 --ny 32 --nz 24 --modes 10 --ftype spatial|helmholtz --fd]
                                                                       the h8thermal box on quadratic tetrahedra

t10 and t10thermal count cubes of 6 tetrahedra (fe.tet10_mesh): their nodes, DOF and filter radius are those of h8 and
h8thermal at twice the element counts (the defaults 64 x 32 x 32 and 80 x 64 x 48).

h8, h8buck and h8thermal take --fronts resident|pooled (the front memory of the factors) and report, for either mode,
the pool size, the persistent bytes of the factors, torch's peak allocated device memory and the factorisation time.
h8thermal also reports the set-up time, device memory and per-design time (apply + apply_gradient) of its filter.
All four of h8, h8thermal, t10 and t10thermal report the time and bytes of the unit element matrices (the element kernel
alone, into fresh buffers) and the time of one fused df/dx call (stored_quadform on the last adjoint's operands).

Each prints one JSON line: stage times (CUDA-synchronised wall clock of the driver's own timers, as the
reference examples report them), solve counts, factor statistics, and size-independent acceptance checks
(eigen-residuals, B-orthonormality, adjoint residual of the converged psi) -- the reference cannot be run at
these sizes inside the GPU job, so parity at full size is by those properties (tests/test_fullsize_gpu.py does
the same for the bench configuration)."""
import argparse
import json
import os
import sys
import time
import warnings

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def now():
    import torch
    torch.cuda.synchronize()
    return time.perf_counter()


def residuals(model, A, B, lam, Phi_d, mode):
    """max_i ||L_i phi_i|| / (||A phi_i|| + |lam_i| ||B phi_i||) and max |Phi^T B Phi - I| on the device."""
    from eigd_b200 import device as D
    import torch
    AP, BP = A.spmm(Phi_d), B.spmm(Phi_d)
    lam_d = torch.as_tensor(np.asarray(lam), device=Phi_d.device)
    R = (AP - BP * lam_d) if mode == "normal" else (BP + AP * lam_d)
    res = (R.norm(dim=0) / (AP.norm(dim=0) + (BP * lam_d).norm(dim=0))).max().item()      # relative to |A phi| + |lam B phi|
    G = D.gemm_tn(Phi_d, BP).cpu().numpy()
    return res, float(np.abs(G - np.eye(G.shape[0])).max())


def setup_dist():
    """torchrun launch: one process per GPU, per-mode adjoint shards (eigd_b200/dist.py)."""
    import torch
    import torch.distributed as dist
    from eigd_b200 import device as D
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    D.init("cuda:%d" % local)
    if world == 1:
        return None, 0, 1
    dist.init_process_group("nccl")
    from eigd_b200.dist import ModeSharding
    return ModeSharding(), dist.get_rank(), world


def run_c3(args):
    from eigd_b200 import device as D, topo as T
    shard, rank, world = setup_dist()
    t0 = now()
    model = T.make_buckling_model(nx=args.nx, ny=args.ny, N=args.modes, m=60, sigma=3.0, solver_type="IRAM",
                                  adjoint_method="sibk", adjoint_options={"lanczos_guess": True}, rtol=1e-10,
                                  deriv_type="tensor")
    t_setup = now() - t0
    model.sharding = shard
    out = {"config": "C3 buckling nx=%d ny=%d" % (args.nx, args.ny), "n": int(model.prob.nred), "nnz": int(model.prob.nnz),
           "N": args.modes, "host_setup_s": t_setup, "n_gpus": world,
           "parallelism": "1 GPU" if world == 1 else "eigensolve replicated, adjoint modes i -> rank i mod %d" % world}
    rng = np.random.default_rng(0)
    reps = []
    for rep in range(args.reps):
        l0 = D.launch_count()
        ta = now()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model.initialize()
        model.initialize_adjoint()
        if rep == 0:                                                # the dof of largest |phi_1| (non-degenerate objective)
            node = int(np.argmax(np.abs(model.prob.full_vector(model.Qr[:, 0].contiguous()).cpu().numpy())))
        h = model.add_eigenvector_aggregate_derivative(1.0, 100.0, node, mode="tanh")
        model.finalize_adjoint()
        tb = now()
        p = model.profile
        reps.append({"wall_s": tb - ta, "assembly_s": p["matrix assembly time"], "eig_s": p["eigenvalue solve time"],
                     "adjoint_s": p["adjoint solution time"], "dfdx_s": p["total derivative time"],
                     "time_to_gradient_s": model.time_to_gradient(), "eig_solves": p["solve preconditioner count"],
                     "adjoint_solves": p["adjoint preconditioner count"], "launches": D.launch_count() - l0,
                     "symbolic_s": p.get("symbolic analysis time")})
    out["reps"] = reps
    out["BLF"] = [float(v) for v in model.BLF]
    out["factor_info"] = model.factor.info
    out["refine_steps"] = model.factor.refine
    out["probe_residual_unrefined"] = model.factor._probe_residual()
    out["symbolic"] = model.symbolic[0].stats()
    res, orth = residuals(model, model.Gr, model.Kr, model.BLF, model.Qr, "buckling")
    out["eigen_residual_max"] = res
    out["orthonormality_defect"] = orth
    ar, ao = model.eig_solver.eval_adjoint_residual_norm(model.Qrb, model.psir, b_ortho=True)
    rhs = float(model.Qrb.norm(dim=0).max().item())
    out["adjoint_residual_over_rtol_rhs"] = float(np.max(ar)) / (1e-10 * rhs)      # <= O(1): the solver's own acceptance level
    assert out["adjoint_residual_over_rtol_rhs"] < 50.0, out["adjoint_residual_over_rtol_rhs"]
    assert res < 1e-8 and orth < 1e-10, (res, orth)
    out["aggregate_h"] = h
    out["xb_norm"] = float(model.xb.norm().item())
    return out


def run_c4(args):
    """BASELINE configs[3]: CRM-scale synthetic shell, 409 x 409 nodes x 6 DOF = 1 003 686 DOF (1 001 232 free), 20 modes, IRAM +
    sibk, modal compliance, per-mode "vector" total derivative over 400 component thicknesses (driver of examples/crm.py).
    The reference cannot run at this size inside the job (and needs TACS for its own model): acceptance = normalised
    eigen / adjoint residuals and a finite-difference check of the gradient, as SURVEY.md 8d prescribes for C4."""
    from eigd_b200 import device as D, shell as S
    shard, rank, world = setup_dist()
    t0 = now()
    model = S.make_shell_model(nx=args.nx, ny=args.ny, ncx=20, ncy=20, N=args.modes, m=60, omega0=10.0, solver_type="IRAM",
                               adjoint_method="sibk", adjoint_options={"lanczos_guess": True}, rtol=1e-10, deriv_type="vector")
    t_setup = now() - t0
    model.sharding = shard
    x0 = np.random.default_rng(0).uniform(0.6, 1.4, model.prob.ncomp)
    out = {"config": "C4 synthetic shell nx=%d ny=%d (6 dof/node, cylindrical panel, clamped edge)" % (args.nx, args.ny),
           "n": int(model.prob.ndof), "nnz": int(model.prob.nnz), "N": args.modes, "ncomp": int(model.prob.ncomp),
           "host_setup_s": t_setup, "n_gpus": world,
           "parallelism": "1 GPU" if world == 1 else "factorisation + eigensolve replicated, adjoint modes and per-mode derivative "
                          "calls i -> rank i mod %d (one packed all-gather, one all-reduce)" % world}
    reps = []
    for rep in range(args.reps):
        model.set_design_vars(x0)
        l0 = D.launch_count()
        ta = now()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model.initialize()
        model.initialize_adjoint()
        model.add_compliance_derivative()
        model.finalize_adjoint()
        tb = now()
        p = model.profile
        reps.append({"wall_s": tb - ta, "assembly_s": p["matrix assembly time"], "eig_s": p["eigenvalue solve time"],
                     "adjoint_s": p["adjoint solution time"], "dfdx_s": p["total derivative time"],
                     "time_to_gradient_s": model.time_to_gradient(), "eig_solves": p["solve preconditioner count"],
                     "adjoint_solves": p["adjoint preconditioner count"], "launches": D.launch_count() - l0,
                     "symbolic_s": p.get("symbolic analysis time")})
    out["reps"] = reps
    out["lam_first"] = [float(v) for v in model.lam[:4]]
    out["factor_info"] = model.factor.info
    out["symbolic"] = model.symbolic[0].stats()
    res, orth = residuals(model, model.Kr, model.Mr, model.lam, model.Q, "normal")
    out["eigen_residual_max_rel"] = res
    out["orthonormality_defect"] = orth
    ar, ao = model.eig_solver.eval_adjoint_residual_norm(model.Qb, model.psi, b_ortho=True)
    rhs = float(model.Qb.norm(dim=0).max().item())
    out["adjoint_residual_over_rtol_rhs"] = float(np.max(ar)) / (1e-10 * rhs)
    grad = model.grad.cpu().numpy().copy()
    out["grad_norm"] = float(np.linalg.norm(grad))
    if args.fd:
        pert = np.random.default_rng(3).uniform(size=x0.shape)
        h = 1e-4
        vals = []
        for sgn in (1.0, -1.0):
            model.set_design_vars(x0 + sgn * h * pert)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                model.initialize()
            vals.append(model.get_compliance())
        fd = (vals[0] - vals[1]) / (2 * h)
        out["fd_directional"] = fd
        out["adjoint_directional"] = float(grad @ pert)
        out["fd_rel_err"] = abs(fd - float(grad @ pert)) / abs(fd)
    return out


def run_nf(args, tag):
    from eigd_b200 import device as D, topo as T
    D.init()
    t0 = now()
    model = T.make_natural_frequency_model(nx=args.nx, ny=args.ny, Lx=2.0, Ly=1.0, N=args.modes, m=60, sigma=-10.0,
                                           solver_type="IRAM", adjoint_method="sibk",
                                           adjoint_options={"lanczos_guess": True}, rtol=1e-10, deriv_type="tensor")
    t_setup = now() - t0
    out = {"config": "%s natural frequency nx=%d ny=%d" % (tag, args.nx, args.ny), "n": int(model.nvars), "N": args.modes,
           "host_setup_s": t_setup}
    w = np.random.default_rng(99).normal(size=(model.nvars, args.modes))
    w_d = D.to_device(w)
    reps = []
    for b in range(args.designs):
        x = np.random.default_rng(b).uniform(0.3, 1.0, model.fltr.num_design_vars)
        l0 = D.launch_count()
        ta = now()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model.initialize(x=x)
        model.initialize_adjoint()
        model.add_modal_function_derivative(w_d)
        model.finalize_adjoint()
        tb = now()
        p = model.profile
        reps.append({"design": b, "wall_s": tb - ta, "assembly_s": p["matrix assembly time"], "eig_s": p["eigenvalue solve time"],
                     "adjoint_s": p["adjoint solution time"], "dfdx_s": p["total derivative time"],
                     "time_to_gradient_s": model.time_to_gradient(), "eig_solves": p["solve preconditioner count"],
                     "adjoint_solves": p["adjoint preconditioner count"], "launches": D.launch_count() - l0,
                     "lam_first": [float(v) for v in model.lam[:3]]})
    out["reps"] = reps
    out["factor_info"] = model.factor.info
    out["symbolic"] = model.symbolic[0].stats()
    res, orth = residuals(model, model.K, model.M, model.lam0, model.Q0, "normal")
    out["eigen_residual_max"] = res
    out["orthonormality_defect"] = orth
    ar, ao = model.eig_solver.eval_adjoint_residual_norm(model.Q0b, model.psi0, b_ortho=True)
    rhs = float(model.Q0b.norm(dim=0).max().item())
    out["adjoint_residual_over_rtol_rhs"] = float(np.max(ar)) / (1e-10 * rhs)
    assert out["adjoint_residual_over_rtol_rhs"] < 50.0 and orth < 1e-10, (out["adjoint_residual_over_rtol_rhs"], orth)
    out["xb_norm"] = float(model.xb.norm().item())
    return out


def gpu_card():
    """Name and power limit of the GPU the numbers were measured on."""
    import subprocess
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                               os.environ.get("LOCAL_RANK", "0")], capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        return "unavailable: %s" % exc


def _element_setup(prob, reps=3):
    """The element kernel that fills the model's unit matrices, rerun into fresh buffers (device-synchronised, every
    repetition), and the bytes of the resident pair."""
    import torch
    from eigd_b200 import device as D, fe
    K0, M0 = torch.empty_like(prob.K0_d), torch.empty_like(prob.M0_d)
    solid = {fe.H8Problem: D.h8_element_matrices, fe.T10Problem: D.t10_element_matrices}
    scalar = {fe.H8ThermalProblem: D.h8_thermal_element_matrices, fe.T10ThermalProblem: D.t10_thermal_element_matrices}
    times = []
    for _ in range(reps):
        t0 = now()
        if type(prob) in solid:
            solid[type(prob)](prob.conn_d, prob.X_d, 1.0, 0.3, 1.0, K0, M0)
        else:
            scalar[type(prob)](prob.conn_d, prob.X_d, K0, M0)
        times.append(now() - t0)
    return {"kernel_s": times, "bytes": int(prob.K0_d.numel() + prob.M0_d.numel()) * 8, "NE": prob.NE,
            "nelems": int(prob.nelems)}


def _dfdx_kernel(model, reps=5):
    """One fused df/dx call (both terms, stored_quadform over N + nrigid columns) on the last adjoint's operands,
    device-synchronised, every repetition."""
    times = []
    for _ in range(reps):
        t0 = now()
        model.prob.device_call_fused(model.psi0, model.psi0, model.Q0, 1.0, -1.0)
        times.append(now() - t0)
    return times


def run_h8(args):
    """Free nx x ny x nz box of hexahedra (NaturalFrequency3DAnalysis), or with ``args.config == "t10"`` of
    nx x ny x nz cubes of quadratic tetrahedra (NaturalFrequencyTetAnalysis): N flexible modes + 6 rigid-body modes
    about sigma = -10, IRAM + sibk with the Lanczos guess, tensor derivative, f = sum_i (phi_i . w_i)^2 as the seed."""
    import torch
    from eigd_b200 import device as D, topo as T
    D.init()
    tet = args.config == "t10"
    out = {"config": "%s free solid nx=%d ny=%d nz=%d" % ("T10" if tet else "H8", args.nx, args.ny, args.nz),
           "N": args.modes, "gpu": gpu_card()}
    t0 = now()
    make = T.make_natural_frequency_tet_model if tet else T.make_natural_frequency_3d_model
    model = make(args.nx, args.ny, args.nz, N=args.modes, m=60, sigma=-10.0, solver_type="IRAM", adjoint_method="sibk",
                 adjoint_options={"lanczos_guess": True}, rtol=1e-10, deriv_type="tensor", fronts=args.fronts)
    out.update(n=int(model.nvars), nnz=int(model.prob.nnz), fronts=args.fronts, host_setup_s=now() - t0)
    torch.cuda.reset_peak_memory_stats()
    w_d = D.to_device(np.random.default_rng(99).normal(size=(model.nvars, args.modes)))
    x0 = np.random.default_rng(0).uniform(0.3, 1.0, model.fltr.num_design_vars)
    reps = []
    for rep in range(args.reps):
        l0 = D.launch_count()
        ta = now()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model.initialize(x=x0)
        model.initialize_adjoint()
        f = model.add_modal_function_derivative(w_d)
        model.finalize_adjoint()
        tb = now()
        p = model.profile
        reps.append({"wall_s": tb - ta, "assembly_s": p["matrix assembly time"], "eig_s": p["eigenvalue solve time"],
                     "adjoint_s": p["adjoint solution time"], "dfdx_s": p["total derivative time"],
                     "time_to_gradient_s": model.time_to_gradient(), "eig_solves": p["solve preconditioner count"],
                     "adjoint_solves": p["adjoint preconditioner count"], "launches": D.launch_count() - l0,
                     "symbolic_s": p.get("symbolic analysis time")})
    out["reps"] = reps
    out["peak_device_bytes"] = int(torch.cuda.max_memory_allocated())
    out["factorisation_s"] = _time_factorisation(model)
    out["memory"] = _factor_memory(model, [model.factor])
    out["element_matrices"] = _element_setup(model.prob)
    out["dfdx_kernel_s"] = _dfdx_kernel(model)
    out["lam_first"] = [float(v) for v in model.lam[:3]]
    out["rigid_lam"] = [float(v) for v in model.lam0[:6]]
    out["factor_info"] = model.factor.info
    out["symbolic"] = model.symbolic[0].stats()
    res, _ = residuals(model, model.K, model.M, model.lam, model.Q, "normal")      # flexible modes: the rigid ones have
    _, orth = residuals(model, model.K, model.M, model.lam0, model.Q0, "normal")     # lambda ~ 0, their relative residual is 0/0
    out["eigen_residual_max"] = res
    out["orthonormality_defect"] = orth
    ar, ao = model.eig_solver.eval_adjoint_residual_norm(model.Q0b, model.psi0, b_ortho=True)
    rhs = float(model.Q0b.norm(dim=0).max().item())
    out["adjoint_residual_over_rtol_rhs"] = float(np.max(ar)) / (1e-10 * rhs)
    assert out["adjoint_residual_over_rtol_rhs"] < 50.0 and orth < 1e-10, (out["adjoint_residual_over_rtol_rhs"], orth)
    assert res < 1e-8, res
    out["objective"] = f
    xb = model.xb.cpu().numpy().copy()
    out["xb_norm"] = float(np.linalg.norm(xb))
    if args.fd:
        pert = np.random.default_rng(3).uniform(-1.0, 1.0, x0.shape)
        h = 1e-5
        vals = []
        for sgn in (1.0, -1.0):
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                model.initialize(x=x0 + sgn * h * pert)
            vals.append(float(np.sum(D.col_dot(model.Q, w_d).cpu().numpy() ** 2)))
        fd = (vals[0] - vals[1]) / (2 * h)
        out["fd_directional"] = fd
        out["adjoint_directional"] = float(xb @ pert)
        out["fd_rel_err"] = abs(fd - float(xb @ pert)) / abs(fd)
    out["gpu_after"] = gpu_card()
    return out


def run_h8buck(args):
    """Clamped 3-D column of hexahedra (BucklingTopology3DAnalysis, make_buckling_3d_model): N load factors about
    sigma = 3 (indefinite shifted factor), IRAM + sibk with the Lanczos guess, tensor derivative, the tanh eigenvector
    aggregate at the dof of largest |phi_1| as the objective, including the fundamental-path adjoint."""
    import torch
    from eigd_b200 import device as D, topo as T
    D.init()
    out = {"config": "H8 buckling column nx=%d ny=%d nz=%d" % (args.nx, args.ny, args.nz), "N": args.modes, "gpu": gpu_card()}
    t0 = now()
    model = T.make_buckling_3d_model(args.nx, args.ny, args.nz, N=args.modes, m=60, solver_type="IRAM", adjoint_method="sibk",
                                     adjoint_options={"lanczos_guess": True}, rtol=1e-10, deriv_type="tensor",
                                     fronts=args.fronts)
    out.update(n=int(model.prob.nred), nnz=int(model.prob.nnz), sigma=float(model.sigma), fronts=args.fronts,
               host_setup_s=now() - t0)
    x0 = np.random.default_rng(0).uniform(0.3, 0.7, model.fltr.num_design_vars)       # first load factor below sigma
    torch.cuda.reset_peak_memory_stats()
    reps = []
    for rep in range(args.reps):
        l0 = D.launch_count()
        ta = now()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model.initialize(x=x0)
        model.initialize_adjoint()
        if rep == 0:
            node = int(np.argmax(np.abs(model.prob.full_vector(model.Qr[:, 0].contiguous()).cpu().numpy())))
        h = model.add_eigenvector_aggregate_derivative(1.0, 100.0, node, mode="tanh")
        model.finalize_adjoint()
        tb = now()
        p = model.profile
        reps.append({"wall_s": tb - ta, "assembly_s": p["matrix assembly time"], "eig_s": p["eigenvalue solve time"],
                     "adjoint_s": p["adjoint solution time"], "dfdx_s": p["total derivative time"],
                     "time_to_gradient_s": model.time_to_gradient(), "eig_solves": p["solve preconditioner count"],
                     "adjoint_solves": p["adjoint preconditioner count"], "launches": D.launch_count() - l0,
                     "symbolic_s": p.get("symbolic analysis time")})
    out["reps"] = reps
    out["peak_device_bytes"] = int(torch.cuda.max_memory_allocated())
    amap = model.symbolic[1]
    shifted = D.axpby(1.0, model.Kr.data, float(model.sigma), model.Gr.data)
    out["factorisation_s"] = {"K_r": _time_numeric(model.Kfact.lu, model.Kr.data, amap),
                              "K_r + sigma G_r": _time_numeric(model.factor.lu, shifted, amap)}
    out["BLF"] = [float(v) for v in model.BLF]
    out["memory"] = _factor_memory(model, [model.Kfact, model.factor])
    out["factor_info"] = {"K_r": model.Kfact.info, "K_r + sigma G_r": model.factor.info}
    out["refine_steps"] = model.factor.refine
    out["probe_residual_unrefined"] = model.factor._probe_residual()
    out["symbolic"] = model.symbolic[0].stats()
    res, orth = residuals(model, model.Gr, model.Kr, model.BLF, model.Qr, "buckling")
    out["eigen_residual_max"] = res
    out["orthonormality_defect"] = orth
    ar, ao = model.eig_solver.eval_adjoint_residual_norm(model.Qrb, model.psir, b_ortho=True)
    rhs = float(model.Qrb.norm(dim=0).max().item())
    out["adjoint_residual_over_rtol_rhs"] = float(np.max(ar)) / (1e-10 * rhs)
    assert out["adjoint_residual_over_rtol_rhs"] < 50.0, out["adjoint_residual_over_rtol_rhs"]
    assert res < 1e-8 and orth < 1e-10, (res, orth)
    assert out["factor_info"]["K_r + sigma G_r"]["negative_pivots"] > 0, out["factor_info"]
    out["aggregate_h"] = h
    xb = model.xb.cpu().numpy().copy()
    out["xb_norm"] = float(np.linalg.norm(xb))
    if args.fd:
        pert = np.random.default_rng(3).uniform(-1.0, 1.0, x0.shape)
        step = 1e-5
        vals = []
        for sgn in (1.0, -1.0):
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                model.initialize(x=x0 + sgn * step * pert)
            vals.append(model.get_eigenvector_aggregate(100.0, node, mode="tanh"))
        fd = (vals[0] - vals[1]) / (2 * step)
        out["fd_directional"] = fd
        out["adjoint_directional"] = float(xb @ pert)
        out["fd_rel_err"] = abs(fd - float(xb @ pert)) / abs(fd)
        assert out["fd_rel_err"] < 1e-5, out["fd_rel_err"]
        out["peak_device_bytes_with_fd"] = int(torch.cuda.max_memory_allocated())
    out["gpu_after"] = gpu_card()
    return out


def run_h8thermal(args):
    """Insulated nx x ny x nz box of hexahedra (ThermalTopology3DAnalysis; mesh, filter radius and driver of
    make_thermal_3d_model, built step by step so that the filter is timed alone), or with ``args.config ==
    "t10thermal"`` of nx x ny x nz cubes of quadratic tetrahedra (ThermalTopologyTetAnalysis, make_thermal_tet_model):
    N modes about sigma = -0.1, mode 0 the zero mode, IRAM + sibk with the Lanczos guess, tensor derivative, thermal
    compliance against the seeded uniform heat vector of bench.py as the objective, conic or Helmholtz filter
    (--ftype)."""
    import torch
    from eigd_b200 import device as D, fe, topo as T
    D.init()
    tet = args.config == "t10thermal"
    Lx, Ly, Lz = 1.0, 0.8, 0.6
    out = {"config": "%s thermal box nx=%d ny=%d nz=%d" % ("T10" if tet else "H8", args.nx, args.ny, args.nz),
           "N": args.modes, "ftype": args.ftype, "gpu": gpu_card()}
    t0 = time.perf_counter()
    conn, X = (fe.tet10_mesh if tet else fe.hex_mesh)(args.nx, args.ny, args.nz, Lx, Ly, Lz)
    t_mesh = time.perf_counter() - t0
    m0 = torch.cuda.memory_allocated()
    t0 = now()
    fltr = fe.NodeFilter(conn, X, r0=4.0 * Ly / ((2 if tet else 1) * args.ny), ftype=args.ftype)
    filt = {"host_setup_s": now() - t0, "device_bytes": int(torch.cuda.memory_allocated() - m0)}
    if args.ftype == "spatial":
        filt["nnz_F"] = int(fltr.F.nnz)
    else:
        filt.update(factor_bytes=fltr._hA.lu.nbytes(), pool_bytes=fltr._hA.lu.pool_bytes(),
                    symbolic=fltr._hA.lu.sym.stats())
    t0 = now()
    model = (T.ThermalTopologyTetAnalysis if tet else T.ThermalTopology3DAnalysis)(
        fltr, conn, X, N=args.modes, m=60, sigma=-0.1, solver_type="IRAM", adjoint_method="sibk",
        adjoint_options={"lanczos_guess": True}, rtol=1e-10, deriv_type="tensor", fronts=args.fronts)
    out.update(n=int(model.nvars), nnz=int(model.prob.nnz), fronts=args.fronts, mesh_s=t_mesh,
               host_setup_s=now() - t0, filter=filt)
    torch.cuda.reset_peak_memory_stats()
    x0 = np.random.default_rng(0).uniform(0.3, 1.0, model.fltr.num_design_vars)     # bench.py X_SEED, VEC_SEED
    vec_d = D.to_device(np.random.default_rng(12345).uniform(size=model.nnodes))
    reps = []
    for rep in range(args.reps):
        l0 = D.launch_count()
        ta = now()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model.initialize(x=x0)
        model.initialize_adjoint()
        model.add_thermal_compliance_derivative(1.0, vec_d)
        model.finalize_adjoint()
        tb = now()
        p = model.profile
        reps.append({"wall_s": tb - ta, "assembly_s": p["matrix assembly time"], "eig_s": p["eigenvalue solve time"],
                     "adjoint_s": p["adjoint solution time"], "dfdx_s": p["total derivative time"],
                     "time_to_gradient_s": model.time_to_gradient(), "eig_solves": p["solve preconditioner count"],
                     "adjoint_solves": p["adjoint preconditioner count"], "launches": D.launch_count() - l0,
                     "symbolic_s": p.get("symbolic analysis time")})
    out["reps"] = reps
    out["peak_device_bytes"] = int(torch.cuda.max_memory_allocated())
    out["factorisation_s"] = _time_factorisation(model)
    out["memory"] = _factor_memory(model, [model.factor])
    out["element_matrices"] = _element_setup(model.prob)
    out["dfdx_kernel_s"] = _dfdx_kernel(model)
    x_d, g_d = D.to_device(x0), D.to_device(np.random.default_rng(2).normal(size=model.nnodes))
    filt["apply_plus_gradient_s"] = []
    for _ in range(5):
        t0 = now()
        fltr.apply(x_d)
        fltr.apply_gradient(g_d, x_d)
        filt["apply_plus_gradient_s"].append(now() - t0)
    out["lam_first"] = [float(v) for v in model.lam[:4]]
    out["factor_info"] = model.factor.info
    out["symbolic"] = model.symbolic[0].stats()
    # nonzero modes only: mode 0 has lambda = 0 (the constant temperature), its relative residual is 0/0
    res, _ = residuals(model, model.K, model.M, model.lam[1:], model.Q[:, 1:].contiguous(), "normal")
    _, orth = residuals(model, model.K, model.M, model.lam, model.Q.contiguous(), "normal")
    out["eigen_residual_max"] = res
    out["orthonormality_defect"] = orth
    ar, ao = model.eig_solver.eval_adjoint_residual_norm(model.Q0b, model.psi0, b_ortho=True)
    rhs = float(model.Q0b.norm(dim=0).max().item())
    out["adjoint_residual_over_rtol_rhs"] = float(np.max(ar)) / (1e-10 * rhs)
    assert out["adjoint_residual_over_rtol_rhs"] < 50.0 and orth < 1e-10, (out["adjoint_residual_over_rtol_rhs"], orth)
    assert res < 1e-8, res
    out["objective"] = model.get_thermal_compliance(vec_d)
    xb = model.xb.cpu().numpy().copy()
    out["xb_norm"] = float(np.linalg.norm(xb))
    if args.fd:
        pert = np.random.default_rng(3).uniform(-1.0, 1.0, x0.shape)
        h = 1e-5
        vals = []
        for sgn in (1.0, -1.0):
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                model.initialize(x=x0 + sgn * h * pert)
            vals.append(model.get_thermal_compliance(vec_d))
        fd = (vals[0] - vals[1]) / (2 * h)
        out["fd_directional"] = fd
        out["adjoint_directional"] = float(xb @ pert)
        out["fd_rel_err"] = abs(fd - float(xb @ pert)) / abs(fd)
        out["peak_device_bytes_with_fd"] = int(torch.cuda.max_memory_allocated())
    out["gpu_after"] = gpu_card()
    return out


def _factor_memory(model, ops):
    """Front memory of the driver's factors: the pool a pooled factorisation borrows (0 resident), the resident fronts
    of one factor, and the bytes every factor keeps for its life (its workspace: fronts included when resident)."""
    sym = model.symbolic[0]
    return {"pool_bytes": ops[0].lu.pool_bytes(), "resident_front_bytes": 8 * sym.query("front_doubles"),
            "pool_doubles": sym.query("pool_doubles"), "factor_bytes": [op.lu.nbytes() for op in ops]}


def _time_numeric(lu, vals, amap, reps=3):
    """Numeric LDL^T of ``vals`` alone, refactored in place in the factor ``lu``, device-synchronised, every repetition."""
    times = []
    for _ in range(reps):
        t0 = now()
        lu.numeric(vals, amap)
        times.append(now() - t0)
    return times


def _time_factorisation(model, reps=3):
    """Numeric LDL^T of the last design's K - sigma M, alone (the driver's eigensolve time includes it): the driver's
    factor refactored in place on the same values, device-synchronised, every repetition."""
    from eigd_b200 import device as D
    vals = D.axpby(1.0, model.K.data, -float(model.sigma), model.M.data)
    times = []
    for _ in range(reps):
        t0 = now()
        model.factor.lu.numeric(vals, model.symbolic[1])
        times.append(now() - t0)
    return times


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("config", choices=["c3", "c4", "c4plate", "c5", "h8", "h8buck", "h8thermal", "t10", "t10thermal"])
    ap.add_argument("--fd", action="store_true", help="c4: add the finite-difference check of the gradient")
    ap.add_argument("--nx", type=int, default=None)
    ap.add_argument("--ny", type=int, default=None)
    ap.add_argument("--nz", type=int, default=None, help="h8, h8buck, h8thermal, t10, t10thermal: elements (cubes) along z")
    ap.add_argument("--modes", type=int, default=None)
    ap.add_argument("--designs", type=int, default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--fronts", choices=["resident", "pooled"], default="resident",
                    help="h8, h8buck, h8thermal, t10, t10thermal: front memory of the factors")
    ap.add_argument("--ftype", choices=["spatial", "helmholtz"], default="spatial", help="h8thermal, t10thermal: filter type")
    a = ap.parse_args()
    if a.config == "c3":
        a.nx, a.ny, a.modes = a.nx or 352, a.ny or 704, a.modes or 20
        res = run_c3(a)
    elif a.config == "c5":
        a.nx, a.ny, a.modes, a.designs = a.nx or 448, a.ny or 224, a.modes or 6, a.designs or 8
        res = run_nf(a, "C5 design sweep")
    elif a.config == "h8":
        a.nx, a.ny, a.nz, a.modes = a.nx or 64, a.ny or 32, a.nz or 32, a.modes or 10
        res = run_h8(a)
    elif a.config == "h8buck":
        a.nx, a.ny, a.nz, a.modes = a.nx or 32, a.ny or 24, a.nz or 128, a.modes or 10
        res = run_h8buck(a)
    elif a.config == "h8thermal":
        a.nx, a.ny, a.nz, a.modes = a.nx or 80, a.ny or 64, a.nz or 48, a.modes or 10
        res = run_h8thermal(a)
    elif a.config == "t10":
        a.nx, a.ny, a.nz, a.modes = a.nx or 32, a.ny or 16, a.nz or 16, a.modes or 10
        res = run_h8(a)
    elif a.config == "t10thermal":
        a.nx, a.ny, a.nz, a.modes = a.nx or 40, a.ny or 32, a.nz or 24, a.modes or 10
        res = run_h8thermal(a)
    elif a.config == "c4":
        a.nx, a.ny, a.modes = a.nx or 408, a.ny or 408, a.modes or 20
        res = run_c4(a)
    else:
        a.nx, a.ny, a.modes, a.designs = a.nx or 1000, a.ny or 500, a.modes or 20, a.designs or 2
        res = run_nf(a, "round-1 C4 stand-in (1M-DOF 2-dof plate)")
    if int(os.environ.get("RANK", "0")) == 0:
        print(json.dumps(res))
