"""The CRM-shaped path (BASELINE configs[3], reference examples/crm.py): 6-DOF shell model, per-mode "vector" total
derivative, design variables = component thicknesses.

  * device assembly of K(t), M(t) from the stored unit element matrices: bit-exact CSR structure and 1e-13 values against
    the scipy COO assembly of oracle/shell_oracle.py;
  * device sensitivities w^T (dK/dx_c) v, w^T (dM/dx_c) v against the numpy einsum of the oracle;
  * the whole driver (IRAM + sibk + add_eig_total_derivative, vector form) against the frozen output of the UNMODIFIED
    reference solvers run on the oracle's matrices (tests/golden/shell_iram.npz): eigenvalues 1e-10, gradient 1e-8;
  * tensor and vector derivative forms agree; the gradient agrees with a central finite difference of the objective."""
import warnings

import numpy as np
import pytest

from conftest import load_golden, align_signs

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(b).max(), 1e-300)


@pytest.fixture(scope="module")
def setup():
    import shell_oracle as so
    from eigd_b200 import device as D, shell as S
    D.init()
    g = load_golden("shell_iram")
    nx, ny = int(g["nx"]), int(g["ny"])
    model = S.make_shell_model(nx=nx, ny=ny, ncx=int(g["ncx"]), ncy=int(g["ncy"]), Ls=1.0, Ly=0.9, radius=2.0, N=int(g["N"]),
                               m=int(g["m"]), omega0=float(g["omega0"]), solver_type="IRAM", adjoint_method="sibk",
                               adjoint_options={"lanczos_guess": True}, rtol=1e-12)
    E1, E3, F1, F3 = S.shell_unit_matrices(model.prob.conn, model.prob.X)
    nodes = np.arange((nx + 1) * (ny + 1)).reshape(nx + 1, ny + 1)
    orc = so.ShellOracle(model.prob.conn, model.prob.X, model.prob.comp, nodes[:, 0], E1, E3, F1, F3)
    return g, model, orc


def test_shell_assembly_and_sensitivities_vs_oracle(setup):
    from eigd_b200 import device as D
    g, model, orc = setup
    p = model.prob
    assert np.array_equal(p.comp, g["comp"]) and np.array_equal(p.reduced, orc.reduced)
    p.set_design(g["x"])
    K, M = p.assemble()
    Ko, Mo = orc.assemble(g["x"])
    assert np.array_equal(p.indptr, Ko.indptr) and np.array_equal(p.indices, Ko.indices)       # bit-exact structure
    assert np.array_equal(Ko.indptr, g["A_indptr"]) and np.array_equal(Ko.indices, g["A_indices"])
    assert rel(K.data.cpu().numpy(), Ko.data) < 1e-13 and rel(M.data.cpu().numpy(), Mo.data) < 1e-13
    rng = np.random.default_rng(0)
    w, v = rng.normal(size=p.ndof), rng.normal(size=p.ndof)
    assert rel(p.dAdx(w, v), orc.dK(g["x"], w, v)) < 1e-12
    assert rel(p.dBdx(w, v), orc.dM(g["x"], w, v)) < 1e-12
    W, V = rng.normal(size=(p.ndof, 5)), rng.normal(size=(p.ndof, 5))
    tens = p.dAdx.device_call(D.to_device(W), D.to_device(V)).cpu().numpy()
    assert rel(tens, sum(orc.dK(g["x"], W[:, k], V[:, k]) for k in range(5))) < 1e-12


def test_shell_sensitivity_rejects_mismatched_columns(setup):
    """W and V with different column counts are refused: the kernel reads W with V's leading dimension."""
    from eigd_b200 import device as D
    g, model, orc = setup
    p = model.prob
    p.set_design(g["x"])
    rng = np.random.default_rng(1)
    W, V = D.to_device(rng.normal(size=(p.ndof, 6))), D.to_device(rng.normal(size=(p.ndof, 5)))
    with pytest.raises(ValueError):
        p.dAdx.device_call(W, V)


def test_shell_driver_vs_reference_solvers(setup):
    g, model, orc = setup
    model.set_design_vars(g["x"])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.initialize()
    assert rel(model.lam, g["lam"]) < 1e-10
    Q = model.Q.cpu().numpy()
    Qa, s = align_signs(Q, g["Phi"])
    assert rel(Qa, g["Phi"]) < 1e-8
    assert abs(model.get_compliance() - float(g["compliance"])) < 1e-9 * abs(float(g["compliance"]))
    model.initialize_adjoint()
    model.add_compliance_derivative()
    model.finalize_adjoint()
    assert rel(model.psi.cpu().numpy() * s, g["psi"]) < 1e-8
    grad_vec = model.grad.cpu().numpy().copy()
    assert rel(grad_vec, g["grad"]) < 1e-8
    # the fused tensor form gives the same gradient
    model.deriv_type = "tensor"
    model.finalize_adjoint()
    assert rel(model.grad.cpu().numpy(), grad_vec) < 1e-12
    model.deriv_type = "vector"


def test_shell_gradient_finite_difference(setup):
    g, model, orc = setup
    x0 = np.array(g["x"])
    model.set_design_vars(x0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.initialize()
        model.initialize_adjoint()
        model.add_compliance_derivative()
        model.finalize_adjoint()
        grad = model.grad.cpu().numpy().copy()
        pert = np.random.default_rng(3).uniform(size=x0.shape)
        h = 1e-5
        model.set_design_vars(x0 + h * pert)
        model.initialize()
        cp = model.get_compliance()
        model.set_design_vars(x0 - h * pert)
        model.initialize()
        cm = model.get_compliance()
    fd = (cp - cm) / (2 * h)
    assert abs(fd - grad @ pert) <= 1e-5 * abs(fd), (fd, grad @ pert)
