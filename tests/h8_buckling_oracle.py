"""Numpy restatement of the linearised buckling of the H8 solid (csrc/h8_buckling.cu, fe.BucklingH8Problem), built on
tests/h8_oracle.py and never imported by the product.  Stress in the Voigt order (xx, yy, zz, yz, xz, xy) with
engineering shear; S is its symmetric 3 x 3 form.

  stress      s_q = kg C B_q u_e
  G0_e        sum_q detJ_q (dNx S_q dNx^T) (x) I_3             (G_e = kg_e G0_e)
  dG/du       sum_e P_e^T kg_e sum_q detJ_q B_q^T C h_q,   h_q = Voigt form of sum_k sum_i grad w_i (x) grad v_i
  dG/dx       dkg_e sum_k w_k^T G0_e(u) v_k,   dK/dx = dk_e sum_k w_k^T K0_e v_k"""
import numpy as np

import h8_oracle as ho


def element_points(xe):
    """detJ (8,), physical shape-function derivatives (8, 8, 3) and B (8, 6, 24) at the Gauss points of one element."""
    dets, dnx, bs = [], [], []
    for g in ho.GAUSS:
        _, dN = ho.shape(g)
        J = xe.T @ dN
        d = dN @ np.linalg.inv(J)
        dets.append(np.linalg.det(J))
        dnx.append(d)
        bs.append(ho.strain_matrix(d))
    return np.array(dets), np.array(dnx), np.array(bs)


def voigt_to_tensor(s):
    return np.array([[s[0], s[5], s[4]], [s[5], s[1], s[3]], [s[4], s[3], s[2]]])


def element_dofs(conn):
    conn = np.asarray(conn)
    return (conn[:, :, None] * 3 + np.arange(3)[None, None, :]).reshape(len(conn), 24)


class H8BucklingOracle:
    def __init__(self, conn, X, E=1.0, nu=0.3):
        self.conn, self.X = np.asarray(conn), np.asarray(X)
        self.C = ho.elasticity(E, nu)
        self.var = element_dofs(self.conn)
        self.ndof = 3 * len(self.X)
        self.points = [element_points(self.X[c]) for c in self.conn]

    def stresses(self, u, kg):
        """(nelems, 8, 6): kg_e C B_q u_e."""
        return np.array([kg[e] * np.einsum("ij,qjk,k->qi", self.C, B, u[self.var[e]])
                         for e, (_, _, B) in enumerate(self.points)])

    def G0(self, u):
        """(nelems, 24, 24) unit stress stiffness about the full displacement u."""
        out = np.zeros((len(self.conn), 24, 24))
        for e, (det, dnx, B) in enumerate(self.points):
            s = np.einsum("ij,qjk,k->qi", self.C, B, u[self.var[e]])
            g = sum(det[q] * dnx[q] @ voigt_to_tensor(s[q]) @ dnx[q].T for q in range(8))
            out[e] = np.kron(g, np.eye(3))
        return out

    def dG_du(self, kg, W, V):
        """Full dof vector d/du sum_k w_k^T G(u) v_k for full (ndof, N) W, V."""
        out = np.zeros(self.ndof)
        for e, (det, dnx, B) in enumerate(self.points):
            we = W[self.var[e]].reshape(8, 3, -1)
            ve = V[self.var[e]].reshape(8, 3, -1)
            de = np.zeros(24)
            for q in range(8):
                gw = np.einsum("aik,am->imk", we, dnx[q])          # grad of component i of w_k
                gv = np.einsum("aik,am->imk", ve, dnx[q])
                T = np.einsum("imk,ink->mn", gw, gv)                # sum_k sum_i grad w_i (x) grad v_i
                h = np.array([T[0, 0], T[1, 1], T[2, 2], T[1, 2] + T[2, 1], T[0, 2] + T[2, 0], T[0, 1] + T[1, 0]])
                de += det[q] * B[q].T @ self.C @ h
            np.add.at(out, self.var[e], kg[e] * de)
        return out

    def quadform(self, Ee, coef, W, V):
        """coef_e sum_k w_k^T Ee v_k per element (dG/dx with (G0, dkg), dK/dx with (K0, dk))."""
        return coef * np.einsum("eak,eab,ebk->e", W[self.var], Ee, V[self.var])
