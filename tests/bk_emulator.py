"""numpy restatement of the dense solver's Bunch-Kaufman pivoting (csrc/bkpivot_kernels.cuh, B2_PIVOT_BUNCH_KAUFMAN).

Same algorithm as the device, step for step: 128 x 128 diagonal blocks; in each, right-looking Bunch-Kaufman with
alpha = (1 + sqrt(17)) / 8 whose search and interchanges stay inside the block; first index on ties; a column whose
diagonal and off-diagonal magnitudes are both below eps becomes a perturbed 1 x 1 pivot of sign(d) * eps.  A 2 x 2 pivot
D_b = Q diag(lam1, lam2) Q' is stored through its Jacobi rotation Q = [[c, s], [-s, c]] (rot[p] = c, rot[p + 1] = s):
L11 unit lower, Lambda on the diagonal, L21' = L21 Q_bd below the block.  The rows below a block are never permuted while
it is factorised; its permutation reaches the columns left of it afterwards (k_bk_swap_left), which here happens at once.

`margin` is the smallest relative distance of any pivot decision from its threshold (the four Bunch-Kaufman comparisons,
and the gap between the largest and the second largest candidate where the choice of r mattered): where it is well above
the rounding difference between the device and numpy, the device must take exactly the same pivots.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

DB = 128
ALPHA = (1.0 + np.sqrt(17.0)) / 8.0
KIND_1X1, KIND_2X2_FIRST, KIND_2X2_SECOND, KIND_PERTURBED = 0, 1, 2, 3


def schur2(a, b, c):
    """[[a, b], [b, c]] = Q diag(l1, l2) Q', Q = [[cs, sn], [-sn, cs]] (the device's bk_schur2)"""
    tau = (c - a) / (2.0 * b)
    t = (1.0 if tau >= 0.0 else -1.0) / (abs(tau) + np.hypot(1.0, tau))
    cs = 1.0 / np.sqrt(1.0 + t * t)
    sn = t * cs
    return cs, sn, a - t * b, c + t * b


def _rel(x, y):
    m = max(abs(x), abs(y))
    return abs(x - y) / m if m > 0 else np.inf


@dataclass
class BKFactor:
    perm: np.ndarray       # int32 [N]: row i of P A P' is row perm[i] of A
    kind: np.ndarray       # int8 [N]: KIND_*
    L: np.ndarray          # [N, N] unit lower: L11 blocks (zero inside a pair) and L21' = L21 Q_bd below them
    lam: np.ndarray        # [N] Lambda
    rot: np.ndarray        # [N] (cos, sin) over each pair, 0 elsewhere
    margin: float
    block: int = DB

    def q_bd(self):
        """the block-diagonal rotation Q_bd (N x N)"""
        Q = np.eye(len(self.lam))
        for p in np.flatnonzero(self.kind == KIND_2X2_FIRST):
            c, s = self.rot[p], self.rot[p + 1]
            Q[p:p + 2, p:p + 2] = [[c, s], [-s, c]]
        return Q

    def l_bd(self):
        """L_bd with P A P' = L_bd diag(Lambda) L_bd': the diagonal blocks L11 Q_k, the stored L21' below them"""
        N, Q = len(self.lam), self.q_bd()
        Lb = self.L.copy()
        for ob in range(0, N, self.block):
            e = min(N, ob + self.block)
            Lb[ob:e, ob:e] = self.L[ob:e, ob:e] @ Q[ob:e, ob:e]
        return Lb

    def inertia(self):
        """(num_pos, num_zero, num_neg); perturbed pivots count as zeros"""
        pert = self.kind == KIND_PERTURBED
        neg = int(np.sum((self.lam < 0) & ~pert))
        zero = int(np.sum(pert))
        return len(self.lam) - neg - zero, zero, neg

    def n_2x2(self):
        return int(np.sum(self.kind == KIND_2X2_FIRST))

    def solve(self, b):
        """x = A^{-1} b the way k_dense_solve_flow<true> does it: b through perm; y_k = Linv_k t_k, publish Q_k' y_k; divide by
        Lambda; rotate z~_k - sum L'^T x_c by Q_k before Linv_k'; x through perm"""
        N, B = len(self.lam), self.block
        Q, L = self.q_bd(), self.L
        bh = np.asarray(b, dtype=np.float64)[self.perm]
        blocks = [(ob, min(N, ob + B)) for ob in range(0, N, B)]
        linv = [np.linalg.inv(L[o:e, o:e]) for o, e in blocks]
        yt = np.zeros(N)
        for k, (o, e) in enumerate(blocks):
            t = bh[o:e] - L[o:e, :o] @ yt[:o]
            yt[o:e] = Q[o:e, o:e].T @ (linv[k] @ t)
        z = yt / self.lam
        xh = np.zeros(N)
        for k in range(len(blocks) - 1, -1, -1):
            o, e = blocks[k]
            s = z[o:e] - L[e:, o:e].T @ xh[e:]
            xh[o:e] = linv[k].T @ (Q[o:e, o:e] @ s)
        x = np.empty(N)
        x[self.perm] = xh
        return x


def _bk_block(D, eps, margin):
    """Bunch-Kaufman of one diagonal block (full symmetric, modified in place) exactly as k_bk_diag128.  Returns the local
    permutation, kinds, Lambda, rot and the unit-lower L11."""
    nb = D.shape[0]
    lp = np.arange(nb)
    kind = np.zeros(nb, dtype=np.int8)
    lam = np.zeros(nb)
    rot = np.zeros(nb)
    L = np.eye(nb)

    def swap(a, b):
        D[[a, b], :] = D[[b, a], :]
        D[:, [a, b]] = D[:, [b, a]]
        L[[a, b], :p] = L[[b, a], :p]        # rows of the multipliers already computed (columns < p)
        lp[[a, b]] = lp[[b, a]]

    p = 0
    while p < nb:
        akk = abs(D[p, p])
        col = np.abs(D[p + 1:, p])
        if col.size:
            r = p + 1 + int(np.argmax(col))
            cmax = col[r - p - 1]
        else:
            r, cmax = nb, -1.0
        step, kd, s = 1, KIND_1X1, None
        if not (akk >= eps) and not (cmax >= eps):
            kd = KIND_PERTURBED
        else:
            margin[0] = min(margin[0], _rel(akk, ALPHA * cmax))
            if not (akk >= ALPHA * cmax):
                if col.size > 1:
                    srt = np.sort(col)
                    margin[0] = min(margin[0], _rel(srt[-1], srt[-2]))
                others = np.abs(np.delete(D[p:, r], r - p))
                smax = others.max() if others.size else 0.0
                margin[0] = min(margin[0], _rel(akk * smax, ALPHA * cmax * cmax))
                if akk * smax >= ALPHA * cmax * cmax:
                    pass
                else:
                    margin[0] = min(margin[0], _rel(abs(D[r, r]), ALPHA * smax))
                    if abs(D[r, r]) >= ALPHA * smax:
                        s = (p, r)
                    else:
                        step, kd = 2, KIND_2X2_FIRST
                        if r != p + 1:
                            s = (p + 1, r)
        if s is not None:
            swap(*s)
        if step == 1:
            d = D[p, p]
            if kd == KIND_PERTURBED:
                d = -eps if d < 0 else eps
            w = D[p + 1:, p].copy()
            D[p + 1:, p + 1:] -= np.outer(w, w) / d
            L[p + 1:, p] = w / d
            lam[p], kind[p] = d, kd
        else:
            a11, a21, a22 = D[p, p], D[p + 1, p], D[p + 1, p + 1]
            det = a11 * a22 - a21 * a21
            E = np.array([[a22, -a21], [-a21, a11]]) / det
            W = D[p + 2:, p:p + 2].copy()
            D[p + 2:, p + 2:] -= W @ E @ W.T
            L[p + 2:, p:p + 2] = W @ E
            cs, sn, l1, l2 = schur2(a11, a21, a22)
            lam[p], lam[p + 1] = l1, l2
            rot[p], rot[p + 1] = cs, sn
            kind[p], kind[p + 1] = KIND_2X2_FIRST, KIND_2X2_SECOND
        p += step
    return lp, kind, lam, rot, L


def bk_factor(A, eps=1e-13, block=DB) -> BKFactor:
    """factorise the symmetric matrix whose LOWER triangle is tril(A) (what b2d_* reads)"""
    A = np.asarray(A, dtype=np.float64)
    N = A.shape[0]
    W = np.tril(A) + np.tril(A, -1).T
    perm = np.arange(N, dtype=np.int32)
    kind = np.zeros(N, dtype=np.int8)
    lam = np.zeros(N)
    rot = np.zeros(N)
    L = np.zeros((N, N))
    margin = [np.inf]
    for ob in range(0, N, block):
        e = min(N, ob + block)
        lp, kd, lm, rt, L11 = _bk_block(W[ob:e, ob:e].copy(), eps, margin)
        g = ob + lp
        W[ob:e, :] = W[g, :]                  # symmetric interchange inside the block (rows below it stay)
        W[:, ob:e] = W[:, g]
        L[ob:e, :ob] = L[g, :ob]              # k_bk_swap_left
        perm[ob:e] = perm[g]
        kind[ob:e], lam[ob:e], rot[ob:e] = kd, lm, rt
        L[ob:e, ob:e] = L11
        if e < N:
            Q = np.eye(e - ob)
            for p in np.flatnonzero(kd == KIND_2X2_FIRST):
                Q[p:p + 2, p:p + 2] = [[rt[p], rt[p + 1]], [-rt[p + 1], rt[p]]]
            # L21' = A21 P' L11^{-T} Q_bd Lambda^{-1}   (k_big_trsm<true>)
            L21 = (W[e:, ob:e] @ np.linalg.inv(L11).T @ Q) / lm
            L[e:, ob:e] = L21
            W[e:, e:] -= (L21 * lm) @ L21.T
    return BKFactor(perm, kind, L, lam, rot, float(margin[0]), block)


def static_inertia(A, eps=1e-13):
    """(num_pos, num_zero, num_neg) of unpivoted LDL^T with |d| < eps perturbed, as the static path computes it"""
    W = np.tril(A) + np.tril(A, -1).T
    W = W.astype(np.float64).copy()
    N = W.shape[0]
    neg = zero = 0
    for k in range(N):
        d = W[k, k]
        if not (abs(d) >= eps):
            d = -eps if d < 0 else eps
            zero += 1
        elif d < 0:
            neg += 1
        w = W[k + 1:, k].copy()
        W[k + 1:, k + 1:] -= np.outer(w, w) / d
    return N - neg - zero, zero, neg


# ------------------------------------------------------------------------------------------------ test matrices
def swap_pairs(n):
    """block diagonal of [[0, 1], [1, 0]]: every 1 x 1 pivot in order is exactly zero"""
    A = np.zeros((n, n))
    for i in range(0, n - 1, 2):
        A[i + 1, i] = A[i, i + 1] = 1.0
    if n % 2:
        A[n - 1, n - 1] = 1.0
    return A


def random_indefinite(n, seed):
    """random symmetric matrix with a zero diagonal (a bilinear form: indefinite, no usable 1 x 1 pivot at the start)"""
    rng = np.random.default_rng(seed)
    B = rng.standard_normal((n, n))
    A = np.tril(B, -1)
    return A + A.T


def augmented(n, m, seed):
    """[[H, J'], [J, 0]] with an indefinite bilinear H (zero diagonal) and du_diag = 0"""
    rng = np.random.default_rng(seed)
    H = random_indefinite(n, seed + 1000)
    J = rng.standard_normal((m, n))
    K = np.zeros((n + m, n + m))
    K[:n, :n] = H
    K[n:, :n] = J
    K[:n, n:] = J.T
    return K


def spd(n, seed):
    rng = np.random.default_rng(seed)
    M = rng.standard_normal((n, n))
    return M @ M.T + n * np.eye(n)


def pivot_test_matrices(sizes=(7, 128, 129, 300)):
    """name -> matrix: the set on which static pivoting perturbs a pivot and Bunch-Kaufman must not"""
    cases = {"swap_pairs_8": swap_pairs(8), "swap_pairs_131": swap_pairs(131)}
    for seed, n in enumerate(sizes, start=1):
        cases[f"random_{n}"] = random_indefinite(n, seed)
    cases["augmented_200_60"] = augmented(200, 60, 5)
    cases["augmented_150_100"] = augmented(150, 100, 6)
    return cases
