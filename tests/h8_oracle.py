"""Numpy restatement of the trilinear hexahedron (H8) of csrc/h8.cu, written from the textbook definition and never
imported by the product: 2x2x2 Gauss rule, isotropic elasticity with strains (exx, eyy, ezz, gyz, gxz, gxy), dof order
node-major (ux, uy, uz), nodes 0-3 counter-clockwise on the zeta = -1 face and 4-7 above them."""
import numpy as np

SIGNS = np.array([[-1, -1, -1], [1, -1, -1], [1, 1, -1], [-1, 1, -1],
                  [-1, -1, 1], [1, -1, 1], [1, 1, 1], [-1, 1, 1]], dtype=np.float64)
GAUSS = [np.array([i, j, k], dtype=np.float64) / np.sqrt(3.0) for k in (-1, 1) for j in (-1, 1) for i in (-1, 1)]


def shape(xi):
    """N (8,) and dN/dxi (8, 3) at the reference point xi (3,)."""
    f = 1.0 + SIGNS * xi[None, :]
    N = 0.125 * f.prod(axis=1)
    dN = np.empty((8, 3))
    for j in range(3):
        others = [k for k in range(3) if k != j]
        dN[:, j] = 0.125 * SIGNS[:, j] * f[:, others[0]] * f[:, others[1]]
    return N, dN


def elasticity(E, nu):
    lam = E * nu / ((1.0 + nu) * (1.0 - 2.0 * nu))
    mu = E / (2.0 * (1.0 + nu))
    C = np.zeros((6, 6))
    C[:3, :3] = lam
    C[np.arange(3), np.arange(3)] += 2.0 * mu
    C[np.arange(3, 6), np.arange(3, 6)] = mu
    return C


def detj(xe):
    """detJ at the 8 Gauss points of the element with node coordinates xe (8, 3)."""
    return np.array([np.linalg.det(xe.T @ shape(g)[1]) for g in GAUSS])


def strain_matrix(dNx):
    """B (6, 24) from the physical derivatives dNx (8, 3)."""
    B = np.zeros((6, 24))
    for a in range(8):
        nx, ny, nz = dNx[a]
        B[0, 3 * a], B[1, 3 * a + 1], B[2, 3 * a + 2] = nx, ny, nz
        B[3, 3 * a + 1], B[3, 3 * a + 2] = nz, ny
        B[4, 3 * a], B[4, 3 * a + 2] = nz, nx
        B[5, 3 * a], B[5, 3 * a + 1] = ny, nx
    return B


def element_matrices(xe, E=1.0, nu=0.3, density=1.0):
    """K0 = sum_q detJ B^T C B and M0 = density sum_q detJ (N N^T (x) I_3), both (24, 24)."""
    C = elasticity(E, nu)
    K = np.zeros((24, 24))
    M = np.zeros((24, 24))
    for g in GAUSS:
        N, dN = shape(g)
        J = xe.T @ dN                                   # J[i, j] = d x_i / d xi_j
        det = np.linalg.det(J)
        B = strain_matrix(dN @ np.linalg.inv(J))
        K += det * B.T @ C @ B
        M += density * det * np.kron(np.outer(N, N), np.eye(3))
    return K, M


def all_element_matrices(conn, X, E=1.0, nu=0.3, density=1.0):
    """(nelems, 24, 24) K0 and M0 of every element."""
    pairs = [element_matrices(X[c], E, nu, density) for c in np.asarray(conn)]
    return np.array([p[0] for p in pairs]), np.array([p[1] for p in pairs])


def rigid_modes(xe):
    """(24, 6): the three translations and three infinitesimal rotations of the nodes xe (8, 3)."""
    R = np.zeros((24, 6))
    for d in range(3):
        R[d::3, d] = 1.0
    x, y, z = xe[:, 0], xe[:, 1], xe[:, 2]
    R[0::3, 3], R[1::3, 3] = -y, x                      # about z
    R[1::3, 4], R[2::3, 4] = -z, y                      # about x
    R[0::3, 5], R[2::3, 5] = z, -x                      # about y
    return R


def assemble(conn, K0, M0, ks, ms, ndof):
    """scipy COO assembly of sum_e P_e^T (ks_e K0_e) P_e and the same for M."""
    import scipy.sparse as sp
    var = (np.asarray(conn)[:, :, None] * 3 + np.arange(3)[None, None, :]).reshape(len(conn), 24)
    i = np.repeat(var, 24, axis=1).ravel()
    j = np.tile(var, (1, 24)).ravel()
    K = sp.coo_matrix(((ks[:, None, None] * K0).ravel(), (i, j)), shape=(ndof, ndof)).tocsr()
    M = sp.coo_matrix(((ms[:, None, None] * M0).ravel(), (i, j)), shape=(ndof, ndof)).tocsr()
    K.sort_indices()
    M.sort_indices()
    return K, M


def perturbed_box(nx, ny, nz, L=(1.0, 1.0, 1.0), amp=0.2, seed=0):
    """fe.hex_mesh numbering with the interior nodes moved by up to amp * element size in each direction."""
    nodes = np.arange((nx + 1) * (ny + 1) * (nz + 1)).reshape(nx + 1, ny + 1, nz + 1)
    g = np.meshgrid(np.linspace(0, L[0], nx + 1), np.linspace(0, L[1], ny + 1), np.linspace(0, L[2], nz + 1), indexing="ij")
    X = np.stack([a.ravel() for a in g], axis=1)
    inner = nodes[1:-1, 1:-1, 1:-1].ravel()
    h = np.array([L[0] / nx, L[1] / ny, L[2] / nz])
    X[inner] += amp * h * np.random.default_rng(seed).uniform(-1.0, 1.0, (len(inner), 3))
    return X
