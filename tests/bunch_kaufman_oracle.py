"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the restricted Bunch-Kaufman pivoting of the multifrontal LDL^T
(diag_factor_bk_kernel and the dense-block variants of trsm_kernel / inverse_init_kernel in eigd_b200/csrc/factor.cu).

An extension of oracle/multifrontal_oracle.py: the same assembly, extend-add and block boundaries, with the pivot rule,
tie break and 2x2 rotation of the kernel, so that the GPU tests can compare pivot decisions and solutions with it.
Only tests/ import this module."""
import numpy as np

import multifrontal_oracle as mo


class BunchKaufmanOracle(mo.MultifrontalOracle):
    """MultifrontalOracle with factor(vals, pivoting="bunch-kaufman") as well as the static factorisation.

    After a pivoted factorisation: info = (negative, perturbed pivots); counts = dict of negative_pivots,
    perturbed_pivots, two_by_two_pivots, interchanges; margin = smallest relative distance of a pivot test from its
    other outcome; L11[k] = M11 of front k (block lower triangular at 32-column granularity)."""

    def __init__(self, sym):
        super().__init__(sym)
        self.L11 = None

    def factor(self, vals, piv_tol=1e-11, pivoting="static"):
        self.L11 = None
        if pivoting == "bunch-kaufman":
            return self._factor_bk(vals, piv_tol)
        if pivoting != "static":
            raise ValueError(pivoting)
        return super().factor(vals, piv_tol)

    def _factor_bk(self, vals, piv_tol):
        """Restricted Bunch-Kaufman LDL^T (diag_factor_bk_kernel in factor.cu): inside every 32-column pivot block
        T = M Lam M^T with M = R^T L, R the product of the block's interchanges and 2x2 rotations, L unit lower,
        Lam diagonal.  The rows below a block get L21 = F21 M^-T Lam^-1 and the trailing matrix F22 - L21 Lam L21^T.
        self.L11[k] holds M11 of front k (block lower triangular at 32-column granularity, dense diagonal blocks)."""
        s = self.sym
        F = np.zeros(s["front_off"][-1])
        amap = s["amap"]
        m = amap >= 0
        F[amap[m]] = vals[m]
        thr = piv_tol * np.abs(vals).max()
        cnt = {"negative_pivots": 0, "perturbed_pivots": 0, "two_by_two_pivots": 0, "interchanges": 0}
        self.margin = np.inf
        dinv = np.zeros(s["sn_first"][-1])
        self.L11 = [None] * self.ns
        for lvl in range(len(s["level_ptr"]) - 1):
            for k in s["level_sn"][s["level_ptr"][lvl]:s["level_ptr"][lvl + 1]]:
                Fk, nc, nb = self._front_view(F, k)
                for ch in np.nonzero(s["sn_parent"] == k)[0]:
                    Fc, ncc, nbc = self._front_view(F, ch)
                    rel = s["rel"][s["sn_rowptr"][ch]:s["sn_rowptr"][ch + 1]]
                    Fk[np.ix_(rel, rel)] += np.tril(Fc[ncc:, ncc:])
                M11 = np.zeros((nc, nc))
                for j0 in range(0, nc, 32):
                    bs = min(32, nc - j0)
                    T = np.tril(Fk[j0:j0 + bs, j0:j0 + bs])
                    L, lam, R = self._bk_block(T + np.tril(T, -1).T, thr, cnt)
                    dinv[s["sn_first"][k] + j0:s["sn_first"][k] + j0 + bs] = 1.0 / lam
                    M11[j0:j0 + bs, j0:j0 + bs] = R.T @ L
                    Li = np.linalg.solve(L, R)                                # M^-1 = L^-1 R
                    L21 = (Fk[j0 + bs:, j0:j0 + bs] @ Li.T) / lam
                    Fk[j0 + bs:, j0:j0 + bs] = L21
                    Fk[j0 + bs:, j0 + bs:] -= np.tril((L21 * lam) @ L21.T)
                    M11[j0 + bs:, j0:j0 + bs] = L21[:nc - j0 - bs]
                self.L11[k] = M11
        self.F, self.dinv = F, dinv
        self.info = (cnt["negative_pivots"], cnt["perturbed_pivots"])
        self.counts = cnt
        return self

    def _bk_block(self, A, thr, cnt):
        """Bunch-Kaufman with alpha = (1 + sqrt 17) / 8 on the symmetric block A, pivot search restricted to it, ties
        to the lowest index; a 2x2 pivot is rotated to diagonal form (Jacobi) and eliminated as two 1x1 pivots.
        Returns unit-lower L, diagonal Lam and orthogonal R with R A R^T = L Lam L^T.  Records in self.margin the
        smallest relative distance of a pivot test (or of the column maximum to its runner-up, where the row of
        the maximum decides) from the other outcome."""
        alpha = (1.0 + np.sqrt(17.0)) / 8.0
        n = A.shape[0]
        W = A.copy()                     # transformed block; columns < j hold d_j * L(:, j)
        R = np.eye(n)
        lam = np.zeros(n)

        def note(x, y):
            self.margin = min(self.margin, abs(x - y) / max(abs(x), abs(y), 1e-300))

        def swap(p, q):
            W[[p, q], :] = W[[q, p], :]
            W[:, [p, q]] = W[:, [q, p]]
            R[[p, q], :] = R[[q, p], :]
            cnt["interchanges"] += 1

        j = 0
        second = False
        while j < n:
            if not second:
                akk = abs(W[j, j])
                col = np.abs(W[j + 1:, j])
                cmax, imax = (col.max(), j + 1 + int(np.argmax(col))) if len(col) else (0.0, j)
                note(akk, alpha * cmax)
                piv, two = j, False
                if not akk >= alpha * cmax:
                    srt = np.sort(col)
                    if len(srt) > 1:
                        note(srt[-1], srt[-2])
                    row = np.abs(W[imax, j:])
                    row[imax - j] = 0.0
                    rmax = row.max()
                    note(akk, alpha * cmax * (cmax / rmax))
                    if akk >= alpha * cmax * (cmax / rmax):
                        pass
                    else:
                        note(abs(W[imax, imax]), alpha * rmax)
                        if abs(W[imax, imax]) >= alpha * rmax:
                            piv = imax
                        else:
                            two = True
                            if imax != j + 1:
                                swap(j + 1, imax)
                if piv != j:
                    swap(j, piv)
                if two:
                    cnt["two_by_two_pivots"] += 1
                    a, b, c = W[j, j], W[j + 1, j], W[j + 1, j + 1]
                    if b != 0.0:
                        tau = (c - a) / (2.0 * b)
                        t = (1.0 if tau >= 0.0 else -1.0) / (abs(tau) + np.sqrt(1.0 + tau * tau))
                        cs = 1.0 / np.sqrt(1.0 + t * t)
                        sn = t * cs
                        G = np.array([[cs, -sn], [sn, cs]])                # rows j, j + 1 <- G @ rows (J^T)
                        W[[j, j + 1], :] = G @ W[[j, j + 1], :]
                        W[:, [j, j + 1]] = W[:, [j, j + 1]] @ G.T
                        R[[j, j + 1], :] = G @ R[[j, j + 1], :]
                        W[j, j], W[j + 1, j + 1] = a - t * b, c + t * b
                        W[j + 1, j] = W[j, j + 1] = 0.0
                    second = True
            else:
                second = False
            d = W[j, j]
            if not np.isfinite(d):
                d = thr if thr > 0 else 1.0
            if abs(d) < thr:
                d = thr if d >= 0 else -thr
                cnt["perturbed_pivots"] += 1
            if d < 0:
                cnt["negative_pivots"] += 1
            lam[j] = d
            colj = W[j + 1:, j].copy()
            W[j + 1:, j + 1:] -= np.outer(colj, colj / d)
            W[j, j + 1:] = 0.0
            j += 1
        L = np.tril(W, -1) / lam + np.eye(n)
        return L, lam, R

    def solve(self, B):
        if self.L11 is None:
            return super().solve(B)
        s = self.sym
        B = np.asarray(B, dtype=float)
        squeeze = B.ndim == 1
        if squeeze:
            B = B[:, None]
        perm = s["perm"]
        y = B[perm].copy()
        for k in range(self.ns):
            Fk, nc, nb = self._front_view(self.F, k)
            c0 = s["sn_first"][k]
            y[c0:c0 + nc] = np.linalg.solve(self.L11[k], y[c0:c0 + nc])
            rows = s["sn_rows"][s["sn_rowptr"][k]:s["sn_rowptr"][k + 1]]
            y[rows] -= Fk[nc:, :nc] @ y[c0:c0 + nc]
        y *= self.dinv[:, None]
        for k in range(self.ns - 1, -1, -1):
            Fk, nc, nb = self._front_view(self.F, k)
            c0 = s["sn_first"][k]
            rows = s["sn_rows"][s["sn_rowptr"][k]:s["sn_rowptr"][k + 1]]
            t = y[c0:c0 + nc] - Fk[nc:, :nc].T @ y[rows]
            y[c0:c0 + nc] = np.linalg.solve(self.L11[k].T, t)
        X = np.empty_like(y)
        X[perm] = y
        return X[:, 0] if squeeze else X
