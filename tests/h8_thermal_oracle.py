"""Numpy restatement of the scalar (heat conduction) trilinear hexahedron of csrc/h8.cu, written from the textbook
definition and never imported by the product: 2x2x2 Gauss rule, one dof per node in node order, unit conductivity and
capacity.  Shape functions and the Gauss rule are those of tests/h8_oracle.py."""
import numpy as np

import h8_oracle as ho


def element_matrices(xe):
    """K0 = sum_q detJ grad N grad N^T and M0 = sum_q detJ N N^T, both (8, 8), of the element with nodes xe (8, 3)."""
    K = np.zeros((8, 8))
    M = np.zeros((8, 8))
    for g in ho.GAUSS:
        N, dN = ho.shape(g)
        J = xe.T @ dN                                   # J[i, j] = d x_i / d xi_j
        det = np.linalg.det(J)
        G = dN @ np.linalg.inv(J)                       # (8, 3) physical gradients
        K += det * G @ G.T
        M += det * np.outer(N, N)
    return K, M


def all_element_matrices(conn, X):
    """(nelems, 8, 8) K0 and M0 of every element."""
    pairs = [element_matrices(X[c]) for c in np.asarray(conn)]
    return np.array([p[0] for p in pairs]), np.array([p[1] for p in pairs])


def thermal_law(rhoE, p=3.0, kappa=1.0, cap=1.0, beta=1e-6):
    """Conductivity and capacity factors of the thermal law (law 0) and their derivatives per element."""
    ks = kappa * ((1.0 - beta) * rhoE ** p + beta)
    ms = cap * ((1.0 - beta) * rhoE + beta)
    dk = kappa * (1.0 - beta) * p * rhoE ** (p - 1.0)
    dm = cap * (1.0 - beta) * np.ones_like(rhoE)
    return ks, ms, dk, dm


def assemble(conn, K0, M0, ks, ms, ndof):
    """scipy COO assembly of sum_e P_e^T (ks_e K0_e) P_e and the same for M, one dof per node."""
    import scipy.sparse as sp
    var = np.asarray(conn, dtype=np.int64)
    i = np.repeat(var, 8, axis=1).ravel()
    j = np.tile(var, (1, 8)).ravel()
    K = sp.coo_matrix(((ks[:, None, None] * K0).ravel(), (i, j)), shape=(ndof, ndof)).tocsr()
    M = sp.coo_matrix(((ms[:, None, None] * M0).ravel(), (i, j)), shape=(ndof, ndof)).tocsr()
    K.sort_indices()
    M.sort_indices()
    return K, M
