"""The pooled front workspace without a GPU: the lifetime-ordered offsets of the symbolic analysis (front k lives from its
own level through its parent's, a root at its own level only) never place two fronts that are live at the same level
on overlapping memory, every front fits in the reported pool, and on 3-D meshes the pool is a fraction of the
resident fronts.  Bad ``fronts`` values are refused before anything touches a device."""
import numpy as np
import pytest

import factor_cases as fc
from eigd_b200 import fe
from eigd_b200.device import Factor, Symbolic


def check_pool(sym):
    """Asserts the lifetime invariants of ``sym``'s pool offsets; returns (pool doubles, resident front doubles)."""
    a = sym.arrays()
    off = sym.pool_offsets()
    total = sym.query("pool_doubles")
    f = np.diff(a["sn_first"]) + np.diff(a["sn_rowptr"])
    size = f * f
    lev, par = a["sn_level"], a["sn_parent"]
    end = np.where(par >= 0, lev[np.maximum(par, 0)], lev)
    assert len(off) == len(f)
    assert np.all(off % 32 == 0), "offsets are 256-byte aligned"
    assert np.all(off >= 0) and np.all(off + size <= total)
    for l in range(int(lev.max()) + 1):
        live = np.nonzero((lev <= l) & (end >= l))[0]
        o = off[live]
        order = np.argsort(o, kind="stable")
        lo, hi = o[order], (o + size[live])[order]
        assert np.all(lo[1:] >= hi[:-1]), "fronts live at level %d overlap" % l
    # every front's interval includes its parent's level: children and parents never share memory
    kids = np.nonzero(par >= 0)[0]
    p = par[kids]
    assert np.all((off[kids] + size[kids] <= off[p]) | (off[p] + size[p] <= off[kids]))
    front_doubles = sym.query("front_doubles")
    assert front_doubles == int(size.sum())
    assert total <= front_doubles + 32 * len(f)
    return total, front_doubles


def case_symbolic(case):
    A = case.A
    return Symbolic(A.indptr, A.indices, A.shape[0], coords=case.coords, dof_per_node=case.dof, opts=case.opts)


CASES = ([("dense", (300, "spd")), ("grid", fc.WIDE_6DOF), ("grid", fc.FRONT_MODE[0]), ("kron", fc.KRON[1])]
         + [("bordered", b) for b in fc.BORDERED])


@pytest.mark.parametrize("kind,args", CASES, ids=["%s-%d" % (k, i) for i, (k, _) in enumerate(CASES)])
def test_pool_offsets_of_factor_cases(kind, args):
    if kind == "dense":
        case = fc.dense_case(*args)
    elif kind == "grid":
        case = fc.grid_case(*args)
    elif kind == "kron":
        case = fc.kron_case(*args)
    else:
        case = fc.bordered_case(*args)
    check_pool(case_symbolic(case))


def test_pool_offsets_of_thermal_grid():
    conn, X = fe.grid_mesh(500, 500, 1.0, 1.0)
    indptr, indices, _, _ = fe.assembly_structure(fe.element_dofs(conn, 1), X.shape[0])
    sym = Symbolic(indptr, indices, X.shape[0], coords=X, dof_per_node=1)
    pool, resident = check_pool(sym)
    assert pool < resident


@pytest.mark.parametrize("n,ratio", [(8, 0.5), (30, 0.25)])
def test_pool_offsets_of_hex_meshes(n, ratio):
    conn, X = fe.hex_mesh(n, n, n)
    ndof = 3 * X.shape[0]
    indptr, indices, _, _ = fe.assembly_structure(fe.element_dofs(conn, 3), ndof)
    sym = Symbolic(indptr, indices, ndof, coords=X, dof_per_node=3)
    pool, resident = check_pool(sym)
    assert pool < ratio * resident, (pool, resident)


def test_pool_size_is_a_query_not_a_stat():
    case = fc.grid_case(*fc.FRONT_MODE[0])
    sym = case_symbolic(case)
    assert "pool_doubles" not in sym.stats()
    assert sym.query("pool_doubles") > 0


def test_unknown_fronts_mode_is_refused():
    case = fc.grid_case(*fc.FRONT_MODE[0])
    sym = case_symbolic(case)
    with pytest.raises(ValueError, match="fronts"):
        Factor(sym, fronts="paged")
    from eigd_b200.eigenvector_derivatives import SpLuOperator
    with pytest.raises(ValueError, match="fronts"):
        SpLuOperator(case.A, fronts="shared")
