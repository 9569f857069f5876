"""What each model driver hands its eigensolver, and which ``profile`` keys one gradient pass writes.

Small thermal, natural-frequency, buckling and shell models, with IRAM and BasicLanczos, plus the complex-step path of the
thermal driver.  Every case records the arguments the driver passes to the solver's constructor (by name, as given), the
attributes it sets on the solver afterwards (``seed``, ``reference_pairing``, ``block_size``, ``sharding``) and the
default of ``m``, then the profile after initialize -> initialize_adjoint -> objective seed -> finalize_adjoint.  ``tol``
is not the default of any driver or solver, so the cases show which constructions receive it."""
import inspect
import warnings

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

TOL = 1e-9
ATOL = 1e-5                 # eig_atol: every driver's default
SEED = 7

FORWARD_KEYS = {"matrix assembly time", "symbolic analysis time", "solve preconditioner count", "eigenvalue solve time",
                "m", "eig_solver.m"}
ADJOINT_KEYS = {"adjoint preconditioner count", "adjoint solution time", "adjoint residuals", "adjoint correction data",
                "total derivative time"}
HEADER_KEYS = {"solver_type", "adjoint_method", "N"}
Q4_KEYS = {"nnodes", "nelems"} | HEADER_KEYS | FORWARD_KEYS | ADJOINT_KEYS | {"adjoint iterations"}
SHELL_KEYS = HEADER_KEYS | FORWARD_KEYS | ADJOINT_KEYS


def _thermal(solver_type, N):
    from eigd_b200 import topo as T
    return T.make_thermal_model(nx=20, ny=16, Lx=1.0, Ly=0.8, N=N, solver_type=solver_type, tol=TOL, seed=SEED,
                                adjoint_options={"lanczos_guess": True}, rtol=1e-10)


def _seed_thermal(model):
    model.add_thermal_compliance_derivative(1.0, np.random.default_rng(1).uniform(size=model.nnodes))


def _natural_frequency():
    from eigd_b200 import topo as T
    return T.make_natural_frequency_model(nx=40, ny=20, Lx=2.0, Ly=1.0, N=5, solver_type="IRAM", tol=TOL, seed=SEED,
                                          adjoint_options={"lanczos_guess": True}, rtol=1e-10)


def _seed_natural_frequency(model):
    model.add_modal_function_derivative(np.random.default_rng(1).normal(size=(model.nvars, model.N)))


def _buckling(solver_type):
    from eigd_b200 import topo as T
    model = T.make_buckling_model(nx=16, ny=32, N=5, sigma=3.0, solver_type=solver_type, tol=TOL, seed=SEED,
                                  adjoint_method="sibk", adjoint_options={"lanczos_guess": True}, rtol=1e-10)
    model.reference_pairing, model.block_size = True, 1
    return model


def _seed_buckling(model):
    model.add_eigenvector_aggregate_derivative(1.0, 10.0, 592)


def _shell(solver_type):
    from eigd_b200 import shell as S
    return S.make_shell_model(nx=16, ny=14, ncx=4, ncy=3, Ls=1.0, Ly=0.9, radius=2.0, N=6, omega0=10.0,
                              solver_type=solver_type, tol=TOL, seed=SEED, adjoint_options={"lanczos_guess": True},
                              rtol=1e-10)


def _seed_shell(model):
    model.add_compliance_derivative()


IRAM_ATTRS = {"seed": SEED, "reference_pairing": False, "block_size": None}

# id: (model, objective seed, solver class, constructor arguments, attributes set after construction,
#      profile keys of the parent design, keys this refactor may add)
CASES = {
    "thermal-iram": (lambda: _thermal("IRAM", 30), _seed_thermal, "IRAM",
                     dict(N=30, m=61, eig_atol=ATOL, tol=TOL), IRAM_ATTRS, Q4_KEYS, set()),
    "thermal-lanczos": (lambda: _thermal("BasicLanczos", 20), _seed_thermal, "BasicLanczos",
                        dict(N=20, m=61, eig_atol=ATOL, tol=TOL, Ntarget=None), {}, Q4_KEYS, set()),
    "natural-frequency-iram": (_natural_frequency, _seed_natural_frequency, "IRAM",
                               dict(N=5 + 3, m=60, eig_atol=ATOL, tol=TOL), IRAM_ATTRS, Q4_KEYS, set()),
    "buckling-iram": (lambda: _buckling("IRAM"), _seed_buckling, "IRAM",
                      dict(N=5, m=60, eig_atol=ATOL, mode="buckling"),
                      {"seed": SEED, "reference_pairing": True, "block_size": 1}, Q4_KEYS, set()),
    "buckling-lanczos": (lambda: _buckling("BasicLanczos"), _seed_buckling, "BasicLanczos",
                         dict(N=5, m=60, eig_atol=ATOL, tol=TOL, mode="buckling"), {}, Q4_KEYS, set()),
    "shell-iram": (lambda: _shell("IRAM"), _seed_shell, "IRAM", dict(N=6, m=60, eig_atol=ATOL), IRAM_ATTRS, SHELL_KEYS,
                   {"adjoint iterations"}),
    "shell-lanczos": (lambda: _shell("BasicLanczos"), _seed_shell, "BasicLanczos", dict(N=6, m=60, eig_atol=ATOL, tol=TOL),
                      {}, SHELL_KEYS, {"adjoint iterations"}),
}


@pytest.fixture
def constructions(monkeypatch):
    """(class name, arguments as passed) of every IRAM / BasicLanczos construction."""
    from eigd_b200 import device as D
    from eigd_b200.eigenvector_derivatives import IRAM, BasicLanczos
    D.init()
    calls = []
    for cls in (IRAM, BasicLanczos):
        def init(self, *args, _init=cls.__init__, _sig=inspect.signature(cls.__init__), _name=cls.__name__, **kwargs):
            bound = _sig.bind(self, *args, **kwargs).arguments
            calls.append((_name, {k: v for k, v in bound.items() if k != "self"}))
            _init(self, *args, **kwargs)
        monkeypatch.setattr(cls, "__init__", init)
    return calls


def _check_keys(profile, parent_keys, may_add):
    keys = set(profile)
    assert parent_keys <= keys, parent_keys - keys
    assert keys - parent_keys <= may_add, keys - parent_keys


@pytest.mark.parametrize("case", list(CASES))
def test_driver_solver_arguments_and_profile_keys(case, constructions):
    make, seed, cls, args, attrs, parent_keys, may_add = CASES[case]
    model = make()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.initialize()
        assert constructions == [(cls, args)]
        solver = model.eig_solver
        assert type(solver).__name__ == cls and model.m == args["m"]
        for name, value in attrs.items():
            assert getattr(solver, name) == value, name
        assert "sharding" in vars(solver) and solver.sharding is None
        model.initialize_adjoint()
        seed(model)
        model.finalize_adjoint()
        _check_keys(model.profile, parent_keys, may_add)
        assert model.time_to_gradient() == (model.profile["eigenvalue solve time"] + model.profile["adjoint solution time"]
                                            + model.profile["total derivative time"])
        model.initialize()                          # m keeps the value it was given on the first call
    assert constructions == [(cls, args)] * 2


def test_complex_step_solver_arguments(constructions):
    """The complex-step (dual-number) path of the thermal driver builds a BasicLanczos of its own."""
    model = _thermal("BasicLanczos", 4)
    model.x = model.x.astype(complex)
    model.x.imag += 1e-6 * np.random.default_rng(2).uniform(size=model.x.shape)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model.initialize()
    assert np.iscomplexobj(np.asarray(model.lam))
    assert constructions == [("BasicLanczos", dict(N=4, m=60, eig_atol=ATOL, tol=TOL, Ntarget=None))]
    assert "sharding" not in vars(model.eig_solver)
    _check_keys(model.profile, {"nnodes", "nelems"} | HEADER_KEYS, {"symbolic analysis time"})
