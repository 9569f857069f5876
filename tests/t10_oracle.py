"""Numpy restatement of the quadratic tetrahedron (T10) of csrc/t10.cu, written from the textbook definition and never
imported by the product: VTK node order (corners 0-3, then the midside nodes of the edges (0,1), (1,2), (2,0), (0,3),
(1,3), (2,3)), quadratic shape functions in barycentric coordinates, the 14-point degree-5 rule read from
csrc/t10_element.cuh (one table for the kernels and the oracle), isotropic elasticity with strains
(exx, eyy, ezz, gyz, gxz, gxy) and dof order node-major (ux, uy, uz).  Also the scalar (heat conduction) element, the
scipy COO assembly and the fused sensitivities."""
import os
import re

import numpy as np

import h8_oracle as ho

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EDGES = ((0, 1), (1, 2), (2, 0), (0, 3), (1, 3), (2, 3))


def _read_rule():
    """Rows (l1, l2, l3, w) of the rule table of csrc/t10_element.cuh; the weights sum to 1/6."""
    text = open(os.path.join(ROOT, "eigd_b200", "csrc", "t10_element.cuh")).read()
    body = re.search(r"t10_rule\[14\]\[4\]\s*=\s*\{(.*?)\};", text, flags=re.S).group(1)
    rows = re.findall(r"\{([^{}]*)\}", body)
    return np.array([[float(v) for v in r.split(",")] for r in rows])


RULE = _read_rule()


def barycentric(q):
    """(l0, l1, l2, l3) of rule point q, l0 formed as the kernel forms it."""
    l1, l2, l3 = RULE[q, :3]
    return np.array([1.0 - l1 - l2 - l3, l1, l2, l3])


def shape(lam):
    """N (10,) and dN/dxi (10, 3) at the barycentric point lam (4,)."""
    N = np.empty(10)
    dL = np.zeros((10, 4))                      # dN/dl
    for a in range(4):
        N[a] = lam[a] * (2.0 * lam[a] - 1.0)
        dL[a, a] = 4.0 * lam[a] - 1.0
    for m, (i, j) in enumerate(EDGES):
        N[4 + m] = 4.0 * lam[i] * lam[j]
        dL[4 + m, i] = 4.0 * lam[j]
        dL[4 + m, j] = 4.0 * lam[i]
    return N, dL[:, 1:] - dL[:, :1]             # l0 = 1 - xi - eta - zeta


def points():
    """(N, dN/dxi, w) at every rule point."""
    return [shape(barycentric(q)) + (RULE[q, 3],) for q in range(len(RULE))]


def strain_matrix(dNx):
    """B (6, 30) from the physical derivatives dNx (10, 3)."""
    B = np.zeros((6, 30))
    for a in range(10):
        nx, ny, nz = dNx[a]
        B[0, 3 * a], B[1, 3 * a + 1], B[2, 3 * a + 2] = nx, ny, nz
        B[3, 3 * a + 1], B[3, 3 * a + 2] = nz, ny
        B[4, 3 * a], B[4, 3 * a + 2] = nz, nx
        B[5, 3 * a], B[5, 3 * a + 1] = ny, nx
    return B


def element_matrices(xe, E=1.0, nu=0.3, density=1.0):
    """K0 = sum_q w detJ B^T C B and M0 = density sum_q w detJ (N N^T (x) I_3), both (30, 30), of nodes xe (10, 3)."""
    C = ho.elasticity(E, nu)
    K = np.zeros((30, 30))
    M = np.zeros((30, 30))
    for N, dN, w in points():
        J = xe.T @ dN                                   # J[i, j] = d x_i / d xi_j
        det = np.linalg.det(J)
        B = strain_matrix(dN @ np.linalg.inv(J))
        K += w * det * B.T @ C @ B
        M += density * w * det * np.kron(np.outer(N, N), np.eye(3))
    return K, M


def thermal_element_matrices(xe):
    """K0 = sum_q w detJ grad N grad N^T and M0 = sum_q w detJ N N^T, both (10, 10)."""
    K = np.zeros((10, 10))
    M = np.zeros((10, 10))
    for N, dN, w in points():
        J = xe.T @ dN
        det = np.linalg.det(J)
        G = dN @ np.linalg.inv(J)
        K += w * det * G @ G.T
        M += w * det * np.outer(N, N)
    return K, M


def all_element_matrices(conn, X, E=1.0, nu=0.3, density=1.0):
    """(nelems, 30, 30) K0 and M0 of every element."""
    pairs = [element_matrices(X[c], E, nu, density) for c in np.asarray(conn)]
    return np.array([p[0] for p in pairs]), np.array([p[1] for p in pairs])


def all_thermal_element_matrices(conn, X):
    """(nelems, 10, 10) K0 and M0 of every scalar element."""
    pairs = [thermal_element_matrices(X[c]) for c in np.asarray(conn)]
    return np.array([p[0] for p in pairs]), np.array([p[1] for p in pairs])


def volume(xe):
    """Volume of the straight-sided tetrahedron with corners xe[:4]."""
    d = xe[1:4] - xe[:1]
    return np.linalg.det(d.T) / 6.0


def rigid_modes(xe):
    """(30, 6): the three translations and three infinitesimal rotations of the nodes xe (10, 3)."""
    R = np.zeros((30, 6))
    for d in range(3):
        R[d::3, d] = 1.0
    x, y, z = xe[:, 0], xe[:, 1], xe[:, 2]
    R[0::3, 3], R[1::3, 3] = -y, x
    R[1::3, 4], R[2::3, 4] = -z, y
    R[0::3, 5], R[2::3, 5] = z, -x
    return R


def element_dofs(conn, dof):
    conn = np.asarray(conn, dtype=np.int64)
    return (conn[:, :, None] * dof + np.arange(dof)[None, None, :]).reshape(len(conn), -1)


def assemble(var, K0, M0, ks, ms, ndof):
    """scipy COO assembly of sum_e P_e^T (ks_e K0_e) P_e and the same for M over the element dofs var (nelems, ne)."""
    import scipy.sparse as sp
    ne = var.shape[1]
    i = np.repeat(var, ne, axis=1).ravel()
    j = np.tile(var, (1, ne)).ravel()
    K = sp.coo_matrix(((ks[:, None, None] * K0).ravel(), (i, j)), shape=(ndof, ndof)).tocsr()
    M = sp.coo_matrix(((ms[:, None, None] * M0).ravel(), (i, j)), shape=(ndof, ndof)).tocsr()
    K.sort_indices()
    M.sort_indices()
    return K, M


def fused_sensitivities(var, K0, M0, dk, dm, WA, WB, V, cA, cB):
    """cA dk_e sum_k WA_k^T K0_e V_k + cB dm_e sum_k WB_k^T M0_e V_k per element (WA, WB, V (ndof, N))."""
    qK = np.einsum("eak,eab,ebk->e", WA[var], K0, V[var])
    qM = np.einsum("eak,eab,ebk->e", WB[var], M0, V[var])
    return cA * dk * qK + cB * dm * qM


def perturbed_tet_box(nx, ny, nz, L=(1.0, 1.0, 1.0), amp=0.2, seed=0):
    """Node coordinates of ``fe.tet10_mesh(nx, ny, nz, *L)`` with the interior lattice nodes moved by up to amp times
    the half-step in each direction: corner and midside nodes both move, so edges are curved."""
    X = ho.perturbed_box(2 * nx, 2 * ny, 2 * nz, L, amp=amp, seed=seed)
    return X
