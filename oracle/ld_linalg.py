"""Extended-precision dense linear algebra: the reference the dense Cholesky, triangular inverse and Sigma^-1 are
tested against.

Plain numpy on np.longdouble (the x87 80-bit format on x86-64: 64-bit significand, eps = 2^-64 ~ 1.1e-19, exponent
range far beyond fp64's, so fp64 inputs -- subnormal or graded ones included -- convert exactly).  Blocked so that the
O(n^3) work goes through longdouble matmul (~0.4 GF/s, no BLAS): a full reference is meant for n <= 1024; larger
matrices are checked with the O(n^2) probe residuals, which stream the fp64 operands in row blocks and never hold an
n x n longdouble copy.
"""
from __future__ import annotations

import numpy as np

LD = np.longdouble
EPS_LD = float(np.finfo(LD).eps)
_NB = 64


def _ld(a) -> np.ndarray:
    return np.asarray(a).astype(LD)


def cholesky(S, nb: int = _NB):
    """Lower Cholesky factor of S (only the lower triangle is read) and LAPACK's info: 0, or the 1-based index of the
    first pivot that is not positive (NaN included).  On failure the rows of L before that pivot are final, the rest
    is zero."""
    A = _ld(S)
    n = A.shape[0]
    L = np.zeros((n, n), dtype=LD)
    for k0 in range(0, n, nb):
        k1 = min(n, k0 + nb)
        Lk = L[k0:k1, :k0]
        D = np.tril(A[k0:k1, k0:k1]) - Lk @ Lk.T
        for j in range(k1 - k0):
            jj = k0 + j
            d = D[j, j] - L[jj, k0:jj] @ L[jj, k0:jj]
            if not d > 0:
                return L, jj + 1
            L[jj, jj] = np.sqrt(d)
            L[jj + 1:k1, jj] = (D[j + 1:, j] - L[jj + 1:k1, k0:jj] @ L[jj, k0:jj]) / L[jj, jj]
        if k1 < n:
            P = A[k1:, k0:k1] - L[k1:, :k0] @ Lk.T
            for j in range(k1 - k0):
                jj = k0 + j
                L[k1:, jj] = (P[:, j] - L[k1:, k0:jj] @ L[jj, k0:jj]) / L[jj, jj]
    return L, 0


def tri_inv(L, nb: int = _NB) -> np.ndarray:
    """W = L^-1 for lower triangular L (forward substitution, block rows)."""
    L = _ld(L)
    n = L.shape[0]
    W = np.zeros((n, n), dtype=LD)
    for i0 in range(0, n, nb):
        i1 = min(n, i0 + nb)
        B = np.zeros((i1 - i0, i1), dtype=LD)
        B[:, :i0] = -(L[i0:i1, :i0] @ W[:i0, :i0])
        B[:, i0:i1] = np.eye(i1 - i0, dtype=LD)
        for r in range(i1 - i0):
            B[r] = (B[r] - L[i0 + r, i0:i0 + r] @ B[:r]) / L[i0 + r, i0 + r]
        W[i0:i1, :i1] = B
    return W


def wtw(W, nb: int = _NB) -> np.ndarray:
    """S = W^T W for lower triangular W (full symmetric result): block row k of W only reaches its first k1 columns."""
    W = _ld(W)
    n = W.shape[0]
    S = np.zeros((n, n), dtype=LD)
    for k0 in range(0, n, nb):
        k1 = min(n, k0 + nb)
        Wk = W[k0:k1, :k1]
        S[:k1, :k1] += Wk.T @ Wk
    return S


def logdet(L) -> LD:
    """log det (L L^T) = 2 sum log L_ii."""
    return LD(2) * np.sum(np.log(np.diagonal(_ld(L))))


def tri_solve(L, b, trans: bool = False) -> np.ndarray:
    """x = L^-1 b (trans: L^-T b) for lower triangular L, by substitution."""
    L = _ld(L)
    x = _ld(b).copy()
    n = L.shape[0]
    if not trans:
        for i in range(n):
            x[i] = (x[i] - L[i, :i] @ x[:i]) / L[i, i]
    else:
        for i in range(n - 1, -1, -1):
            x[i] = (x[i] - L[i + 1:, i] @ x[i + 1:]) / L[i, i]
    return x


def componentwise_backward_error(L, S, rows: int = 128) -> float:
    """max_ij |L L^T - S|_ij / (|L| |L|^T)_ij over the lower triangle, with L L^T formed in longdouble (S and L are
    taken as exact).  An entry whose denominator is 0 counts as 0 if its residual is 0 too, else as inf."""
    L = np.tril(np.asarray(L, dtype=np.float64))
    S = np.asarray(S, dtype=np.float64)
    n = L.shape[0]
    Lld = L.astype(LD)
    Lab = np.abs(Lld)
    worst = 0.0
    for r0 in range(0, n, rows):
        r1 = min(n, r0 + rows)
        num = np.abs(Lld[r0:r1, :r1] @ Lld[:r1, :r1].T - S[r0:r1, :r1].astype(LD))
        den = Lab[r0:r1, :r1] @ Lab[:r1, :r1].T
        low = np.tril(np.ones((r1 - r0, r1), dtype=bool), k=r0)
        if np.any(np.isnan(num[low])):
            return float("inf")
        zero = low & (den == 0)
        if np.any(num[zero] != 0):
            return float("inf")
        ok = low & (den != 0)
        if np.any(ok):
            worst = max(worst, float(np.max(num[ok] / den[ok])))
    return worst


def normwise_backward_error(L, S, rows: int = 128) -> float:
    """max |L L^T - S| / max |S| over the lower triangle, L L^T in longdouble."""
    L = np.tril(np.asarray(L, dtype=np.float64))
    S = np.asarray(S, dtype=np.float64)
    n = L.shape[0]
    Lld = L.astype(LD)
    worst = LD(0)
    for r0 in range(0, n, rows):
        r1 = min(n, r0 + rows)
        R = np.tril(Lld[r0:r1, :r1] @ Lld[:r1, :r1].T - S[r0:r1, :r1].astype(LD), k=r0)
        worst = max(worst, np.max(np.abs(R)))
    return float(worst / LD(np.max(np.abs(np.tril(S)))))


def _symv(M, v, rows: int, absolute: bool = False) -> np.ndarray:
    """M v in longdouble for symmetric M given by its lower triangle (absolute: |M| |v|), fp64 M streamed in row
    blocks."""
    n = M.shape[0]
    v = np.abs(v) if absolute else v
    out = np.zeros((n,) + v.shape[1:], dtype=LD)
    for r0 in range(0, n, rows):
        r1 = min(n, r0 + rows)
        blk = np.tril(np.asarray(M[r0:r1, :r1], dtype=np.float64), k=r0)
        blk = (np.abs(blk) if absolute else blk).astype(LD)
        out[r0:r1] += blk @ v[:r1]
        strict = np.tril(blk, k=r0 - 1)
        out[:r1] += strict.T @ v[r0:r1]
    return out


def _trmv(L, v, rows: int, trans: bool = False) -> np.ndarray:
    """tril(L) v (trans: tril(L)^T v) in longdouble, fp64 L streamed in row blocks."""
    n = L.shape[0]
    out = np.zeros((n,) + v.shape[1:], dtype=LD)
    for r0 in range(0, n, rows):
        r1 = min(n, r0 + rows)
        blk = np.tril(np.asarray(L[r0:r1, :r1], dtype=np.float64), k=r0).astype(LD)
        if trans:
            out[:r1] += blk.T @ v[r0:r1]
        else:
            out[r0:r1] = blk @ v[:r1]
    return out


def chol_probe_residual(L, S, v, rows: int = 256) -> float:
    """max_i |L (L^T v) - S v|_i / max_i (|S| |v|)_i in longdouble, O(n^2); L and S are read in their lower
    triangles, v is n x k."""
    v = _ld(v)
    r = _trmv(L, _trmv(L, v, rows, trans=True), rows) - _symv(S, v, rows)
    return float(np.max(np.abs(r)) / np.max(_symv(S, v, rows, absolute=True)))


def sinv_probe_residual(Sinv, S, v, rows: int = 256) -> float:
    """max |Sinv (S v) - v| / max |v| in longdouble, O(n^2); Sinv and S are read in their lower triangles."""
    v = _ld(v)
    r = _symv(Sinv, _symv(S, v, rows), rows) - v
    return float(np.max(np.abs(r)) / np.max(np.abs(v)))
