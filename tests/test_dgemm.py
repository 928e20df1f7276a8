"""The dense path's DMMA GEMM (csrc/dgemm.cu, lfm_dgemm_kernel) launched directly through lfm_debug_dgemm.

Nearly every flop of the blocked Cholesky, the triangular inverse, Sigma^-1 = W^T W and the posterior products runs in this
kernel, and each of those callers relies on a per-tile contract: the k-range of its kmode, the k-window, the epilogue mode,
which tiles are launched at all.  The references here model that contract tile by tile in numpy.  With integer operands in
[-16, 16] every fp64 product and partial sum is exact, so the kernel has to match them bit for bit whatever order it sums
in; operands the contract says are never read hold NaN, so a k-range one tile too wide shows up as NaN in the result.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BK = 16
FULL, LE_ROW, GE_ROW, GE_ROWCOL, LAUUM_LATE = 0, 1, 3, 4, 5
KMODES = (FULL, LE_ROW, GE_ROW, GE_ROWCOL, LAUUM_LATE)
TRANS = ((0, 0), (0, 1), (1, 0), (1, 1))
# (alpha, beta) for each epilogue mode of the kernel; every result is exactly representable on integer operands
EPILOGUES = {0: ((1.0, 0.0), (-3.0, 0.0), (0.5, 0.0)),
             1: ((0.5, -0.25), (-1.0, 2.0), (-3.0, 1.0), (1.0, -0.25), (0.5, 1.0)),
             2: ((1.0, 1.0),),
             3: ((-1.0, 1.0),)}
TILE_OF_REQUEST = {1: 142, 2: 444, 3: 422}


# ---- reference of the per-tile contract (numpy, CPU) ----------------------------------------------------------------
def tile_shape(variant):
    """(BM, BN) of the instantiation coded TA TBN WM WN GM: 8 WM GM x 32 WN."""
    wm, wn, gm = variant // 100 % 10, variant // 10 % 10, variant % 10
    return 8 * wm * gm, 32 * wn


def c_mode(alpha, beta):
    if beta == 0.0:
        return 0
    if beta == 1.0 and alpha in (1.0, -1.0):
        return 2 if alpha == 1.0 else 3
    return 1


def tile_k_range(kmode, row0, col0, BM, K, k_split, k_lo, k_hi):
    kb, ke = 0, K
    if kmode == LE_ROW:
        ke = min(K, row0 + BM)
    elif kmode == GE_ROW:
        kb = row0
    elif kmode == GE_ROWCOL:
        kb = max(row0, col0)
    elif kmode == LAUUM_LATE:
        kb = k_split if row0 < k_split else max(row0, col0)
    return max(kb, k_lo), min(ke, k_hi)


def launched_tiles(M, N, BM, BN, lower_only=False, tri_skip=0):
    for i in range(M // BM):
        if lower_only and i < tri_skip // BM:
            continue
        for j in range(i + 1 if lower_only else N // BN):
            yield i * BM, j * BN


def tile_rule(opA, opB, C0, BM, BN, alpha, beta, kmode=FULL, lower_only=False, tri_skip=0, k_split=0, k_lo=0,
              k_hi=1 << 62):
    """C after one launch: op(A) (M x K), op(B) (K x N) and C0 (M x N) as arrays, tile by tile as the kernel does."""
    M, K = opA.shape
    N = opB.shape[1]
    out = C0.copy()
    full = None
    for row0, col0 in launched_tiles(M, N, BM, BN, lower_only, tri_skip):
        kb, ke = tile_k_range(kmode, row0, col0, BM, K, k_split, k_lo, k_hi)
        cm = (2 if row0 < k_split else 0) if kmode == LAUUM_LATE else c_mode(alpha, beta)
        nk = (ke - kb) // BK if ke > kb else 0
        if nk == 0 and cm >= 2:
            continue                                   # accumulate mode with nothing to add: the tile is not touched
        r, c = slice(row0, row0 + BM), slice(col0, col0 + BN)
        ke = kb + nk * BK
        if nk == 0:
            acc = np.zeros((BM, BN))
        elif kb == 0 and ke == K:
            if full is None:
                full = opA @ opB
            acc = full[r, c]
        else:
            acc = opA[r, kb:ke] @ opB[kb:ke, c]
        old = C0[r, c]
        if cm == 0:
            out[r, c] = alpha * acc
        elif cm == 1:
            out[r, c] = alpha * acc + beta * old
        elif cm == 2:
            out[r, c] = old + acc
        else:
            out[r, c] = old - acc
    return out


def mat(buf, off, rows, cols, ld):
    """rows x cols row-major view with leading dimension ld at element offset off of a 1-D buffer."""
    return np.lib.stride_tricks.as_strided(buf[off:], shape=(rows, cols), strides=(8 * ld, 8))


def reference(bufA, bufB, bufC, variant, M, N, K, lda, ldb, ldc, transA=0, transB=0, offA=0, offB=0, offC=0,
              alpha=1.0, beta=0.0, lower_only=False, kmode=FULL, batch=1, strideA=0, strideB=0, strideC=0, tile=0,
              tri_skip=0, k_split=0, k_lo=0, k_hi=1 << 62):
    """The whole C buffer after the launch (bufC is bufA: in place, every tile reading its operands before it writes)."""
    BM, BN = tile_shape(variant)
    out = bufC.copy()
    for y in range(max(batch, 1)):
        opA = mat(bufA, offA + y * strideA, K, M, lda).T if transA else mat(bufA, offA + y * strideA, M, K, lda)
        opB = mat(bufB, offB + y * strideB, N, K, ldb).T if transB else mat(bufB, offB + y * strideB, K, N, ldb)
        C0 = np.array(mat(bufC, offC + y * strideC, M, N, ldc))
        res = tile_rule(opA, opB, C0, BM, BN, alpha, beta, kmode, lower_only, tri_skip, k_split, k_lo, k_hi)
        mat(out, offC + y * strideC, M, N, ldc)[...] = res
    return out


def ints(rng, n):
    return rng.integers(-16, 17, size=n).astype(np.float64)


def buf_len(rows, cols, ld, off=0, batch=1, stride=0):
    return off + (max(batch, 1) - 1) * stride + (rows - 1) * ld + cols


# ---- launching ------------------------------------------------------------------------------------------------------
def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64).reshape(-1)).cuda()


def run(bufA, bufB, bufC, **d):
    """One launch over copies of the numpy buffers (bufC is bufA: C aliases A); returns (variant, C buffer after)."""
    from dis_project_b200 import ops
    tA = dev(bufA)
    tB = dev(bufB)
    tC = tA if bufC is bufA else dev(bufC)
    v = ops.debug_dgemm(tA, tB, tC, **d)
    return v, tC.cpu().numpy()


def assert_same(got, exp, what):
    if not np.array_equal(got, exp, equal_nan=True):
        bad = np.flatnonzero(~((got == exp) | (np.isnan(got) & np.isnan(exp))))
        raise AssertionError(f"{what}: {bad.size} elements differ, first at {bad[0]}: got {got[bad[0]]}, "
                             f"expected {exp[bad[0]]}")


def check(bufA, bufB, bufC, want=None, **d):
    v, got = run(bufA, bufB, bufC, **d)
    assert v // 1000 == 10 * d.get("transA", 0) + d.get("transB", 0), (v, d)
    if want is not None:
        assert v % 1000 == want, (v, want, d)
    assert_same(got, reference(bufA, bufB, bufC, v, **d), f"variant {v}, {d}")
    return v


def tile_requests(lower_only):
    return (0, 2, 3) if lower_only else (0, 1, 2, 3)


# ---- CPU self-checks of the reference -------------------------------------------------------------------------------
def test_tile_shapes_of_every_instantiation():
    assert {v: tile_shape(v) for v in (142, 242, 422, 442, 444, 842)} == {
        142: (16, 128), 242: (32, 128), 422: (64, 64), 442: (64, 128), 444: (128, 128), 842: (128, 128)}
    assert tile_shape(11142) == (16, 128) and [c_mode(a, b) for a, b in ((3, 0), (0.5, 1), (1, 1), (-1, 1), (1, 2))] == \
        [0, 1, 2, 3, 1]


def test_tile_rule_reproduces_the_products_it_stands_for():
    """The reference against plain products: each kmode on the operand structure it exists for gives the whole product;
    k-windows add up to the full range; accumulate tiles with an empty range stay as they were."""
    rng = np.random.default_rng(1)
    M, K = 256, 256
    A, B, C = ints(rng, (M, K)), ints(rng, (K, M)), ints(rng, (M, M))
    L = np.tril(A)
    for BM, BN in ((16, 128), (64, 64), (128, 128), (32, 128)):
        assert np.array_equal(tile_rule(A, B, C, BM, BN, -3.0, 0.5), -3.0 * (A @ B) + 0.5 * C)
        assert np.array_equal(tile_rule(L, B, C, BM, BN, 1.0, 0.0, LE_ROW), L @ B)
        assert np.array_equal(tile_rule(L.T, B, C, BM, BN, -1.0, 1.0, GE_ROW), C - L.T @ B)
        if BM == BN:
            low = tile_rule(L.T, L, C, BM, BN, 1.0, 0.0, GE_ROWCOL, lower_only=True)
            assert np.array_equal(np.tril(low), np.tril(L.T @ L))
            assert np.array_equal(np.triu(low, BM), np.triu(C, BM))           # tiles above the diagonal: untouched
            S11 = C.copy()
            S11[:128, :128] = L[:128, :128].T @ L[:128, :128]
            late = tile_rule(L.T, L, S11, BM, BN, 1.0, 0.0, LAUUM_LATE, lower_only=True, k_split=128)
            assert np.array_equal(np.tril(late), np.tril(L.T @ L))
            skip = tile_rule(A, B, C, BM, BN, -1.0, 1.0, lower_only=True, tri_skip=128)
            assert np.array_equal(skip[:128], C[:128]) and np.array_equal(np.tril(skip)[128:], np.tril(C - A @ B)[128:])
        part = C
        for k0 in range(0, K, 48):       # k-windows on 16-multiples, not tile-aligned
            part = tile_rule(A, B, part, BM, BN, 1.0, 0.0 if k0 == 0 else 1.0, k_lo=k0, k_hi=k0 + 48)
        assert np.array_equal(part, A @ B)
        # GE_ROW with an accumulate epilogue over a window that misses the lower rows' ranges: those tiles untouched
        win = tile_rule(A, B, C, BM, BN, 1.0, 1.0, GE_ROW, k_lo=0, k_hi=128)
        assert np.array_equal(win[128:], C[128:]) and np.array_equal(win[:BM], C[:BM] + A[:BM, :128] @ B[:128])
        # ... and with beta = 0 the same tiles are written with zeros
        assert np.array_equal(tile_rule(A, B, C, BM, BN, 1.0, 0.0, GE_ROW, k_hi=128)[128:], np.zeros((128, M)))


def test_reference_reads_buffers_with_offsets_strides_and_aliasing():
    rng = np.random.default_rng(2)
    M, N, K, lda, ldb, ldc = 128, 256, 32, 136, 40, 262
    bufA, bufB = ints(rng, buf_len(K, M, lda, 4, 2, 5000)), ints(rng, buf_len(N, K, ldb, 2, 2, 11000))
    bufC = ints(rng, buf_len(M, N, ldc, 6, 2, 40000))
    out = reference(bufA, bufB, bufC, 11422, M, N, K, lda=lda, ldb=ldb, ldc=ldc, transA=1, transB=1, offA=4, offB=2,
                    offC=6, alpha=0.5, beta=2.0, batch=2, strideA=5000, strideB=11000, strideC=40000)
    for y in range(2):
        opA = np.array([bufA[4 + 5000 * y + k * lda:][:M] for k in range(K)]).T
        opB = np.array([bufB[2 + 11000 * y + c * ldb:][:K] for c in range(N)]).T
        C0 = np.array([bufC[6 + 40000 * y + r * ldc:][:N] for r in range(M)])
        got = np.array([out[6 + 40000 * y + r * ldc:][:N] for r in range(M)])
        assert np.array_equal(got, 0.5 * opA @ opB + 2.0 * C0)
    mask = np.ones(bufC.size, bool)
    for y in range(2):
        for r in range(M):
            mask[6 + 40000 * y + r * ldc:][:N] = False
    assert np.array_equal(out[mask], bufC[mask])
    # in place: C is A's first 128 columns, the product reads A as it was
    A = ints(rng, 256 * 160)
    W = ints(rng, 128 * 144)
    out = reference(A, W, A, 242, 256, 128, 144, lda=160, ldb=144, ldc=160, transB=1)
    assert np.array_equal(out.reshape(256, 160)[:, :128], A.reshape(256, 160)[:, :144] @ W.reshape(128, 144).T)
    assert np.array_equal(out.reshape(256, 160)[:, 128:], A.reshape(256, 160)[:, 128:])


# ---- (a) the contract grid ------------------------------------------------------------------------------------------
GRID_SHAPES = ((256, 256, 16), (128, 128, 32), (256, 256, 48), (256, 384, 48), (384, 384, 144), (512, 512, 1040))


@pytest.mark.gpu
@pytest.mark.parametrize("kmode", KMODES)
@pytest.mark.parametrize("ta,tb", TRANS)
def test_contract_grid(cuda, ta, tb, kmode):
    """Every kmode x epilogue mode x lower_only x tile request, K from one k-tile to 65 (odd: the last unit is the
    4-step one), M > K so that the GE modes have tiles with empty ranges."""
    rng = np.random.default_rng(100 * ta + 10 * tb + kmode)
    n = 0
    for M, N, K in GRID_SHAPES:
        bufA, bufB = ints(rng, M * K), ints(rng, K * N)
        for cm in (0, 1, 2, 3):
            alpha, beta = EPILOGUES[cm][n % len(EPILOGUES[cm])]
            n += 1
            bufC = ints(rng, M * N)
            for lower in (False, True):
                if lower and M != N:
                    continue
                for tile in tile_requests(lower):
                    check(bufA, bufB, bufC, want=TILE_OF_REQUEST.get(tile), M=M, N=N, K=K,
                          lda=M if ta else K, ldb=K if tb else N, ldc=N, transA=ta, transB=tb, alpha=alpha, beta=beta,
                          lower_only=lower, kmode=kmode, tile=tile, k_split=(M // 2 // BK) * BK if kmode == LAUUM_LATE else 0)


@pytest.mark.gpu
@pytest.mark.parametrize("kmode", KMODES)
@pytest.mark.parametrize("ta,tb", TRANS)
def test_contract_windows_padding_offsets_batches(cuda, ta, tb, kmode):
    """k-windows on 16-multiples that are not tile-aligned, padded leading dimensions, offset base pointers, batches
    whose strides are not tile multiples, tri_skip, and C aliasing A."""
    rng = np.random.default_rng(1000 + 100 * ta + 10 * tb + kmode)
    n = 0

    def one(M, N, K, lower, tile, pad=(0, 0, 0), off=(0, 0, 0), batch=1, gap=(0, 0, 0), **kw):
        nonlocal n
        cm = n % 4 if "cm" not in kw else kw.pop("cm")
        alpha, beta = EPILOGUES[cm][n % len(EPILOGUES[cm])]
        n += 1
        rA, cA = (K, M) if ta else (M, K)
        rB, cB = (N, K) if tb else (K, N)
        lda, ldb, ldc = cA + pad[0], cB + pad[1], N + pad[2]
        sA, sB, sC = (rA * lda + gap[0], rB * ldb + gap[1], M * ldc + gap[2]) if batch > 1 else (0, 0, 0)
        bufA = ints(rng, buf_len(rA, cA, lda, off[0], batch, sA))
        bufB = ints(rng, buf_len(rB, cB, ldb, off[1], batch, sB))
        bufC = ints(rng, buf_len(M, N, ldc, off[2], batch, sC))
        if kmode == LAUUM_LATE:
            kw.setdefault("k_split", 128)
        check(bufA, bufB, bufC, want=TILE_OF_REQUEST.get(tile), M=M, N=N, K=K, lda=lda, ldb=ldb, ldc=ldc, transA=ta,
              transB=tb, offA=off[0], offB=off[1], offC=off[2], alpha=alpha, beta=beta, lower_only=lower, kmode=kmode,
              tile=tile, batch=batch, strideA=sA, strideB=sB, strideC=sC, **kw)

    for lower in (False, True):
        for tile in tile_requests(lower):
            one(256, 256, 256, lower, tile, pad=(6, 10, 2), off=(2, 6, 4), k_lo=48, k_hi=208)
            one(256, 256, 256, lower, tile, k_lo=0, k_hi=64, cm=2 + n % 2)     # first chunk, accumulating
            one(256, 256, 256, lower, tile, k_lo=160, k_hi=1 << 62, cm=2)
            one(256, 256, 96, lower, tile, pad=(2, 0, 4), off=(0, 2, 2), batch=3, gap=(34, 18, 66))
            one(384, 384, 144, lower, tile, k_split=48 if kmode == LAUUM_LATE else 0, off=(8, 0, 0))
        if lower:
            one(512, 512, 160, True, 0, tri_skip=128)
            one(512, 512, 160, True, 3, tri_skip=192, batch=2, gap=(2, 4, 6))
            one(512, 512, 160, True, 2, tri_skip=256, k_lo=16, k_hi=112)
    if ta == 0:
        # C aliasing A: one tile across the full width N = 128 (32-row tiles from the heuristic, 16-row on request)
        for tile in (0, 1, 3):
            for K, lda, k_lo, k_hi in ((144, 160, 0, 1 << 62), (128, 128, 32, 96), (256, 258, 0, 1 << 62)):
                cm = n % 4
                alpha, beta = EPILOGUES[cm][n % len(EPILOGUES[cm])]
                n += 1
                bufA = ints(rng, buf_len(256, lda, lda, 2))
                bufB = ints(rng, buf_len(128, K, K) if tb else buf_len(K, 128, 128))
                check(bufA, bufB, bufA, want=142 if tile == 1 else 242, M=256, N=128, K=K, lda=lda, ldb=K if tb else 128,
                      ldc=lda, offA=2, offC=2, transB=tb, alpha=alpha, beta=beta, kmode=kmode, tile=tile,
                      k_split=64 if kmode == LAUUM_LATE else 0, k_lo=k_lo, k_hi=k_hi)


# ---- (b) what the callers rely on, with the never-read parts poisoned ----------------------------------------------
def poisoned_lower(rng, n, nb=128):
    """(poisoned, clean): a lower-triangular integer matrix with exact zeros above the diagonal inside the diagonal
    128-blocks, and NaN in every strictly upper 128-block in the poisoned copy."""
    clean = np.tril(ints(rng, (n, n)))
    bad = clean.copy()
    for i in range(0, n, nb):
        bad[i:i + nb, i + nb:] = np.nan
    return bad, clean


def tile_mask(M, N, BM, BN, lower_only=False, tri_skip=0):
    m = np.zeros((M, N), bool)
    for r, c in launched_tiles(M, N, BM, BN, lower_only, tri_skip):
        m[r:r + BM, c:c + BN] = True
    return m


def check_product(v, got, C0, want, lower_only=False, tri_skip=0, elementwise_lower=False):
    """Launched tiles hold `want` bit for bit and no NaN; the rest of C is as it was (NaN included)."""
    mask = tile_mask(*got.shape, *tile_shape(v), lower_only, tri_skip)
    if elementwise_lower:       # only the lower triangle of the diagonal tiles is meaningful to the caller
        mask &= np.tril(np.ones(got.shape, bool))
        outside = ~tile_mask(*got.shape, *tile_shape(v), lower_only, tri_skip)
        assert_same(got[outside], C0[outside], f"variant {v}: tiles that are not launched")
    else:
        assert_same(got[~mask], C0[~mask], f"variant {v}: tiles that are not launched")
    assert not np.isnan(got[mask]).any(), f"variant {v}: NaN from a part of an operand that must not be read"
    assert_same(got[mask], want[mask], f"variant {v}: launched tiles")


def launch_np(A, B, C, inplace=False, **d):
    """Launch on 2-D numpy operands (contiguous, ld = column count unless given); returns (variant, C after)."""
    d.setdefault("lda", A.shape[1])
    d.setdefault("ldb", B.shape[1])
    d.setdefault("ldc", C.shape[1] if not inplace else A.shape[1])
    bA = A.reshape(-1).copy()
    v, out = run(bA, B.reshape(-1), bA if inplace else C.reshape(-1), **d)
    return v, out.reshape(A.shape if inplace else C.shape)


@pytest.mark.gpu
@pytest.mark.parametrize("tile", (0, 1, 2, 3))
def test_trtri_products_never_read_the_upper_blocks(cuda, tile):
    """lfm_trtri / trtri_levels (chol.cu): T^T = W11^T L21^T with kmode GE_ROW (TT) and W21 = -W22 T with LE_ROW (NT),
    one problem and batched along the diagonal with the production stride 2 m (ld + 1)."""
    rng = np.random.default_rng(20 + tile)
    m = 384
    Wp, W = poisoned_lower(rng, m)
    L21 = ints(rng, (m, m))
    C0 = np.full((m, m), np.nan)
    v, got = launch_np(Wp, L21, C0, M=m, N=m, K=m, transA=1, transB=1, kmode=GE_ROW, tile=tile)
    check_product(v, got, C0, W.T @ L21.T)
    Tt = got
    v, got = launch_np(Wp, Tt, C0, M=m, N=m, K=m, transB=1, alpha=-1.0, kmode=LE_ROW, tile=tile)
    check_product(v, got, C0, -(W @ Tt.T))
    # trtri_levels at n = 1024, level m = 256: two nodes in one launch
    n, h = 1024, 256
    from dis_project_b200 import ops
    Lp, Lc = poisoned_lower(rng, n)
    Wbig_p, Wbig = poisoned_lower(rng, n)
    for o in (0, 2 * h):   # W21 is written with beta = 0: NaN before
        Wbig_p[o + h:o + 2 * h, o:o + h] = np.nan
    tW, tL = dev(Wbig_p), dev(Lp)
    stride = 2 * h * (n + 1)
    v = ops.debug_dgemm(tW, tL, tW, h, h, h, lda=n, ldb=n, ldc=n, offA=0, offB=h * n, offC=h, transA=1, transB=1,
                        kmode=GE_ROW, batch=2, strideA=stride, strideB=stride, strideC=stride, tile=tile)
    v2 = ops.debug_dgemm(tW, tW, tW, h, h, h, lda=n, ldb=n, ldc=n, offA=h * n + h, offB=h, offC=h * n, transB=1,
                         alpha=-1.0, kmode=LE_ROW, batch=2, strideA=stride, strideB=stride, strideC=stride, tile=tile)
    assert v % 1000 == v2 % 1000
    got = tW.cpu().numpy().reshape(n, n)
    for o in (0, 2 * h):
        W11, W22 = Wbig[o:o + h, o:o + h], Wbig[o + h:o + 2 * h, o + h:o + 2 * h]
        L21 = Lc[o + h:o + 2 * h, o:o + h]
        Tt = W11.T @ L21.T
        assert_same(got[o:o + h, o + h:o + 2 * h], Tt, f"variant {v}: T^T of the node at {o}")
        assert_same(got[o + h:o + 2 * h, o:o + h], -(W22 @ Tt.T), f"variant {v2}: W21 of the node at {o}")
        assert_same(got[o:o + 2 * h, o:o + 2 * h][np.tril(np.ones((2 * h, 2 * h), bool))],
                    np.tril(np.block([[W11, np.zeros((h, h))], [-(W22 @ Tt.T), W22]]))[np.tril(np.ones((2 * h, 2 * h), bool))],
                    "the node's lower triangle")


@pytest.mark.gpu
@pytest.mark.parametrize("tile", (0, 1, 2, 3))
def test_posterior_product_never_reads_the_upper_blocks(cuda, tile):
    """posterior.cu: V = W K_xf with W lower-triangular, kmode LE_ROW, NN."""
    rng = np.random.default_rng(30 + tile)
    Wp, W = poisoned_lower(rng, 512)
    Kxf = ints(rng, (512, 384))
    C0 = np.full((512, 384), np.nan)
    v, got = launch_np(Wp, Kxf, C0, M=512, N=384, K=512, kmode=LE_ROW, tile=tile)
    check_product(v, got, C0, W @ Kxf)


@pytest.mark.gpu
@pytest.mark.parametrize("tile", (0, 2, 3))
def test_lauum_never_reads_the_scratch_blocks(cuda, tile):
    """lfm_lauum: Sigma^-1 (lower tiles) = W^T W, kmode GE_ROWCOL, TN, lower_only; the strictly upper blocks of W hold
    lfm_trtri's scratch (NaN here).  The gene posterior's V^T V (FULL, TN, lower_only) beside it."""
    rng = np.random.default_rng(40 + tile)
    Wp, W = poisoned_lower(rng, 640)
    C0 = np.full((640, 640), np.nan)
    v, got = launch_np(Wp, Wp, C0, M=640, N=640, K=640, transA=1, lower_only=True, kmode=GE_ROWCOL, tile=tile)
    check_product(v, got, C0, W.T @ W, lower_only=True)
    V = ints(rng, (512, 384))
    C0 = np.full((384, 384), np.nan)
    v, got = launch_np(V, V, C0, M=384, N=384, K=512, transA=1, lower_only=True, tile=tile)
    check_product(v, got, C0, V.T @ V, lower_only=True)


@pytest.mark.gpu
@pytest.mark.parametrize("tile", (0, 2, 3))
def test_lauum_late_never_reads_w11(cuda, tile):
    """lfm_lauum_late: S = W^T W in one launch when the top-left half of S already holds S11' = W11^T W11.  Tiles of the
    rows < k_split add W21^T W21 (k >= k_split only), the others are lfm_lauum's.  Nothing reads W11 (all NaN here) or
    the strictly upper blocks."""
    rng = np.random.default_rng(50 + tile)
    n, h = 512, 256
    Wp, W = poisoned_lower(rng, n)
    Wp[:h, :h] = np.nan
    C0 = np.full((n, n), np.nan)
    C0[:h, :h] = np.tril(W[:h, :h].T @ W[:h, :h])
    C0[:h, :h][np.triu_indices(h, 1)] = np.nan
    v, got = launch_np(Wp, Wp, C0, M=n, N=n, K=n, transA=1, lower_only=True, kmode=LAUUM_LATE, k_split=h, tile=tile)
    check_product(v, got, C0, W.T @ W, lower_only=True, elementwise_lower=True)


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", (256, 512))
def test_early_s11_in_k_chunks_never_reads_the_upper_blocks(cuda, chunk):
    """potrf_right_looking's early S11' = W11^T W11 (GE_ROWCOL, TN, lower_only, 64 x 64 tiles) in k-chunks: the first
    with beta = 0, the rest accumulating, as gemm_kchunked launches it."""
    from dis_project_b200 import ops
    rng = np.random.default_rng(60 + chunk)
    h = 1024
    Wp, W = poisoned_lower(rng, h)
    C0 = np.full((h, h), np.nan)
    tW, tC = dev(Wp), dev(C0)
    for k0 in range(0, h, chunk):
        v = ops.debug_dgemm(tW, tW, tC, h, h, h, lda=h, ldb=h, ldc=h, transA=1, beta=0.0 if k0 == 0 else 1.0,
                            lower_only=True, kmode=GE_ROWCOL, tile=3, k_lo=k0, k_hi=k0 + chunk)
        assert v == 10422
    check_product(v, tC.cpu().numpy().reshape(h, h), C0, W.T @ W, lower_only=True)


@pytest.mark.gpu
@pytest.mark.parametrize("tile", (0, 2, 3))
def test_trailing_update_reads_and_writes_only_its_tiles(cuda, tile):
    """The blocked Cholesky's trailing update A22 -= P P^T (NT, lower_only, beta = 1, alpha = -1: C in the accumulators),
    whole and with the first block row skipped (tri_skip: the look-ahead chain owns it).  Upper blocks and skipped rows of
    C are NaN and must stay so."""
    rng = np.random.default_rng(70 + tile)
    m = 512
    P = ints(rng, (m, 128))
    C0 = np.tril(ints(rng, (m, m)))
    for i in range(0, m, 128):
        C0[i:i + 128, i + 128:] = np.nan
    for skip in (0, 128):
        Cs = C0.copy()
        Cs[:skip] = np.nan
        v, got = launch_np(P, P, Cs, M=m, N=m, K=128, transB=1, alpha=-1.0, beta=1.0, lower_only=True, tri_skip=skip,
                           tile=tile)
        check_product(v, got, Cs, Cs - P @ P.T, lower_only=True, tri_skip=skip)


@pytest.mark.gpu
@pytest.mark.parametrize("tile", (0, 1))
def test_panel_multiply_in_place(cuda, tile):
    """The factorisation's panel P <- P W_kk^T in place (C aliasing A, NT, beta = 0), with W_kk lower-triangular; tile 1
    is the unfused chain's 16 x 128 launch.  The rest of the rows of P's storage (columns >= 128) stays."""
    rng = np.random.default_rng(80 + tile)
    m, ld = 640, 384
    A = ints(rng, (m, ld))
    Wkk = np.tril(ints(rng, (128, 128)))
    v, got = launch_np(A, Wkk, None, inplace=True, M=m, N=128, K=128, lda=ld, ldb=128, ldc=ld, transB=1, tile=tile)
    assert v % 1000 == (142 if tile == 1 else 242)
    assert_same(got[:, :128], A[:, :128] @ Wkk.T, f"variant {v}: panel")
    assert_same(got[:, 128:], A[:, 128:], f"variant {v}: beyond the panel")


# ---- (c) the tile heuristic and where it switches ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("M,N,lower,batch,tri_skip,want", [
    (2688, 2688, False, 1, 0, 422), (2816, 2688, False, 1, 0, 444),     # 441 vs 462 tiles of 128 x 128
    (3712, 3712, True, 1, 0, 422), (3840, 3840, True, 1, 0, 444),       # 435 vs 465 lower tiles
    (128, 128, False, 443, 0, 422), (128, 128, False, 444, 0, 444),     # batches of one tile
    (3840, 3840, True, 1, 128, 422),                                    # tri_skip: 64 x 64 tiles whatever the count
])
def test_tile_heuristic_thresholds(cuda, M, N, lower, batch, tri_skip, want):
    rng = np.random.default_rng(M + N + batch)
    K = 32
    sA, sB, sC = (M * K + 2, N * K + 2, M * N + 2) if batch > 1 else (0, 0, 0)
    bufA = ints(rng, buf_len(M, K, K, 0, batch, sA))
    bufB = ints(rng, buf_len(N, K, K, 0, batch, sB))
    bufC = ints(rng, buf_len(M, N, N, 0, batch, sC))
    check(bufA, bufB, bufC, want=want, M=M, N=N, K=K, lda=K, ldb=K, ldc=N, transB=1, alpha=-1.0, beta=1.0,
          lower_only=lower, tri_skip=tri_skip, batch=batch, strideA=sA, strideB=sB, strideC=sC)


@pytest.mark.gpu
@pytest.mark.parametrize("M,want", [(9344, 242), (9472, 442), (18816, 442), (18944, 842)])
@pytest.mark.parametrize("ta,tb", TRANS)
def test_in_place_tile_thresholds(cuda, M, want, ta, tb):
    """C aliasing A: 32-row tiles below 148 tiles of 64 rows, 64-row tiles below 148 of 128 rows, 128-row tiles above.
    With op(A) = A^T the product reads columns of A that other tiles' rows overwrite; the operands are laid out so that
    every such element is written with the value it already has (the first K M / 128 columns of A are zero, so the rows of
    C that hold them only add zeros), and the result is defined."""
    rng = np.random.default_rng(M + 10 * ta + tb)
    K = 16
    bufB = ints(rng, 128 * K)
    if ta == 0:
        lda = 136
        bufA = ints(rng, M * lda)
        d = dict(lda=lda, ldc=lda, alpha=-1.0, beta=1.0)
    else:
        bufA = ints(rng, M * 128)
        A = bufA[:K * M].reshape(K, M)
        A[:, :K * M // 128] = 0.0
        d = dict(lda=M, ldc=128, alpha=1.0, beta=1.0)
    check(bufA, bufB, bufA, want=want, M=M, N=128, K=K, ldb=K if tb else 128, transA=ta, transB=tb, **d)


@pytest.mark.gpu
def test_large_triangular_launch_decodes_every_tile(cuda):
    """M = N = 16384 with 64 x 64 tiles on request (32 896 lower tiles; the heuristic alone would take 128 x 128): the
    single-precision triangular-index decode far from zero, each tile written once where the tile rule says."""
    from dis_project_b200 import ops
    rng = np.random.default_rng(90)
    n, K = 16384, 16
    A, B = ints(rng, (n, K)), ints(rng, (n, K))
    tC = torch.full((n * n,), 0.5, dtype=torch.float64, device="cuda")
    v = ops.debug_dgemm(dev(A), dev(B), tC, n, n, K, lda=K, ldb=K, ldc=n, transB=1, lower_only=True, tile=3)
    assert v == 1422
    C = tC.view(n, n)
    tiles_r = np.arange(n) // 64
    for r0 in range(0, n, 1024):
        got = C[r0:r0 + 1024].cpu().numpy()
        want = np.where(tiles_r[r0:r0 + 1024, None] >= tiles_r[None, :], A[r0:r0 + 1024] @ B.T, 0.5)
        assert_same(got, want, f"rows {r0}..{r0 + 1024}")


# ---- (d) precision and invariance on random operands ----------------------------------------------------------------
def ld_product(opA, opB):
    return opA.astype(np.longdouble) @ opB.astype(np.longdouble)


@pytest.mark.gpu
@pytest.mark.parametrize("ta,tb", TRANS)
def test_fp64_error_bound_on_normal_operands(cuda, ta, tb):
    """|C - C_ref| <= (K + 2) 2^-53 (|alpha| |A||B| + |beta| |C|) against a long-double product: no reduced-precision
    path anywhere in the kernel."""
    rng = np.random.default_rng(110 + 10 * ta + tb)
    for (M, N, K), (alpha, beta) in zip(((256, 256, 1008), (384, 128, 144), (128, 256, 496)),
                                        ((1.0, 0.0), (-1.0, 1.0), (0.7, -1.3))):
        A = rng.standard_normal((K, M) if ta else (M, K))
        B = rng.standard_normal((N, K) if tb else (K, N))
        C0 = rng.standard_normal((M, N))
        opA, opB = (A.T if ta else A), (B.T if tb else B)
        ref = alpha * ld_product(opA, opB) + beta * C0.astype(np.longdouble)
        bound = (K + 2) * 2.0 ** -53 * (abs(alpha) * (np.abs(opA) @ np.abs(opB)) + abs(beta) * np.abs(C0))
        for tile in (0, 1, 2, 3):
            v, got = launch_np(A, B, C0, M=M, N=N, K=K, transA=ta, transB=tb, alpha=alpha, beta=beta, tile=tile)
            err = np.abs(got.astype(np.longdouble) - ref).astype(np.float64)
            assert np.all(err <= bound), (v, float(np.max(err / bound)))


@pytest.mark.gpu
@pytest.mark.parametrize("ta,tb", TRANS)
def test_tile_variants_agree_bit_for_bit(cuda, ta, tb):
    """Every variant runs the same DMMA sequence over k in ascending order, so FULL products agree to the bit across tile
    shapes; on triangular operands the k-ranges differ by whole groups of structural zeros, which add exact zeros."""
    rng = np.random.default_rng(120 + 10 * ta + tb)
    M, N, K = 384, 256, 400
    A = rng.standard_normal((K, M) if ta else (M, K))
    B = rng.standard_normal((N, K) if tb else (K, N))
    C0 = rng.standard_normal((M, N))
    for alpha, beta in ((1.0, 0.0), (-1.0, 1.0), (0.3, 0.9)):
        outs = {}
        for tile in (0, 1, 2, 3):
            v, outs[v] = launch_np(A, B, C0, M=M, N=N, K=K, transA=ta, transB=tb, alpha=alpha, beta=beta, tile=tile)
        first = next(iter(outs.values()))
        assert len(outs) == 3 and all(np.array_equal(o, first) for o in outs.values()), (alpha, beta, sorted(outs))
    if ta == 0:
        # C aliasing A (N = 128): the in-place variant against the out-of-place ones on the same numbers
        lda = 416
        Ai = rng.standard_normal((M, lda))
        Bi = rng.standard_normal((128, K) if tb else (K, 128))
        Ci = Ai[:, :128].copy()
        ref = {launch_np(Ai[:, :K].copy(), Bi, Ci, M=M, N=128, K=K, transB=tb, alpha=-1.0, beta=1.0, tile=t)[1].tobytes()
               for t in (1, 2, 3)}
        v, got = launch_np(Ai, Bi, None, inplace=True, M=M, N=128, K=K, lda=lda, ldc=lda, transB=tb, alpha=-1.0, beta=1.0)
        assert v % 1000 == 242 and ref == {np.ascontiguousarray(got[:, :128]).tobytes()}
    # triangular: LE_ROW on lower-triangular A, GE_ROW on A^T with A lower-triangular, GE_ROWCOL on the lower tiles
    Lt = np.tril(rng.standard_normal((M, M)))
    B = rng.standard_normal((M, N) if not tb else (N, M))
    for kmode, A_, transA in ((LE_ROW, Lt, 0), (GE_ROW, Lt, 1)):
        outs = {launch_np(A_, B, C0, M=M, N=N, K=M, transA=transA, transB=tb, kmode=kmode, tile=t)[1].tobytes()
                for t in (0, 1, 2, 3)}
        assert len(outs) == 1, kmode
        full = launch_np(A_, B, C0, M=M, N=N, K=M, transA=transA, transB=tb, kmode=FULL)[1]
        assert {full.tobytes()} == outs, kmode
    S0 = rng.standard_normal((M, M))
    lows = [np.tril(launch_np(Lt, Lt, S0, M=M, N=M, K=M, transA=1, lower_only=True, kmode=GE_ROWCOL, tile=t)[1])
            for t in (2, 3)]
    assert np.array_equal(lows[0], lows[1])


@pytest.mark.gpu
@pytest.mark.parametrize("alpha", (1.0, -1.0))
def test_k_chunked_launches_equal_one_launch(cuda, alpha):
    """gemm_kchunked (chol.cu): beta = 0 for the first chunk, then beta = 1, equals the single launch to the bit when
    alpha = +-1 -- the accumulate epilogue starts the accumulators from C (sign-flipped for alpha = -1) and continues
    the same sum."""
    from dis_project_b200 import ops
    rng = np.random.default_rng(130)
    M, K = 512, 1024
    for kmode, lower in ((FULL, False), (GE_ROWCOL, True)):
        W = np.tril(rng.standard_normal((K, M))) if kmode == GE_ROWCOL else rng.standard_normal((K, M))
        tW = dev(W)
        for tile in (2, 3):
            one = dev(np.zeros(M * M))
            ops.debug_dgemm(tW, tW, one, M, M, K, lda=M, ldb=M, ldc=M, transA=1, alpha=alpha, lower_only=lower,
                            kmode=kmode, tile=tile)
            for chunk in (16, 256, 512):
                ch = dev(np.full(M * M, np.nan))
                for k0 in range(0, K, chunk):
                    ops.debug_dgemm(tW, tW, ch, M, M, K, lda=M, ldb=M, ldc=M, transA=1, alpha=alpha,
                                    beta=0.0 if k0 == 0 else 1.0, lower_only=lower, kmode=kmode, tile=tile, k_lo=k0,
                                    k_hi=k0 + chunk)
                a, b = one.cpu().numpy().reshape(M, M), ch.cpu().numpy().reshape(M, M)
                mask = tile_mask(M, M, *tile_shape(TILE_OF_REQUEST[tile]), lower)
                assert np.array_equal(a[mask], b[mask]), (kmode, tile, chunk)


# ---- (e) descriptors the library refuses ----------------------------------------------------------------------------
@pytest.mark.gpu
def test_rejected_descriptors_leave_c_unchanged(cuda):
    from dis_project_b200 import _lib, ops
    rng = np.random.default_rng(140)
    A, B = dev(ints(rng, 1 << 18)), dev(ints(rng, 1 << 18))
    C0 = ints(rng, 1 << 18)
    tC = dev(C0)
    ok = dict(M=256, N=256, K=64, lda=64, ldb=64, ldc=256, transB=1)
    INVALID, UNSUPPORTED = -1, -3
    cases = [
        (INVALID, dict(offA=1)), (INVALID, dict(offB=3)), (INVALID, dict(offC=1)),          # 8-byte aligned pointers
        (INVALID, dict(lda=65)), (INVALID, dict(ldb=67)), (INVALID, dict(ldc=257)),          # odd leading dimensions
        (INVALID, dict(batch=2, strideA=1, strideB=64, strideC=256)),                        # odd batch strides
        (INVALID, dict(batch=2, strideA=64, strideB=3, strideC=256)),
        (INVALID, dict(batch=2, strideA=64, strideB=64, strideC=255)),
        (INVALID, dict(M=192)), (INVALID, dict(N=200, ldc=200)), (INVALID, dict(K=40, lda=40, ldb=40)),
        (INVALID, dict(M=-128)),
        (INVALID, dict(lower_only=True, N=128, ldc=128)),                                     # lower_only needs M = N
        (INVALID, dict(lower_only=True, tri_skip=64, tile=2)),                               # tri_skip % BM
        (INVALID, dict(lower_only=True, tile=1)),                                            # 16 x 128 tiles: not square
        (INVALID, dict(kmode=2)), (INVALID, dict(kmode=6)), (INVALID, dict(kmode=-1)),       # no such k-range mode
        (INVALID, dict(transA=2)), (INVALID, dict(transB=-1)),
        (INVALID, dict(k_lo=8)), (INVALID, dict(k_hi=40)), (INVALID, dict(kmode=LAUUM_LATE, k_split=24)),
        (UNSUPPORTED, dict(batch=65536, strideA=0, strideB=0, strideC=0)),                   # more than gridDim.y holds
    ]
    for status, change in cases:
        d = dict(ok, **change)
        with pytest.raises(_lib.LfmError) as e:
            ops.debug_dgemm(A, B, tC, **d)
        assert e.value.status == status, change
        assert torch.equal(tC, dev(C0)), change
    # in place (C aliasing A): N must be 128, and the tiles (16 / 32 / 64 / 128 x 128) cannot serve lower_only
    for status, change in ((INVALID, dict(N=256)), (INVALID, dict(lower_only=True, M=128))):
        d = dict(dict(M=256, N=128, K=128, lda=256, ldb=128, ldc=256, transB=1), **change)
        before = A.clone()
        with pytest.raises(_lib.LfmError) as e:
            ops.debug_dgemm(A, B, A, **d)
        assert e.value.status == status, change
        assert torch.equal(A, before)
    # the bounds check refuses before the library is called
    small = dev(np.zeros(256 * 64 - 1))
    for bad in (dict(A=small), dict(B=small), dict(C=small), dict(offA=-2)):
        args = dict(A=A, B=B, C=tC)
        args.update({k: bad.pop(k) for k in ("A", "B", "C") if k in bad})
        with pytest.raises(ValueError):
            ops.debug_dgemm(args["A"], args["B"], args["C"], **dict(ok, **bad))
    assert torch.equal(tC, dev(C0))
    assert ops.debug_dgemm(A, B, tC, **ok) == 1422                                           # the valid launch runs


# ---- (f) the unfused chain step -------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_unfused_chain_step_gives_the_same_bits(cuda, tmp_path):
    """LFM_CHAIN_FUSED=0 replaces the factorisation's fused chain step (one 8-CTA cluster launch) by two 16 x 128-tile
    launches of the DMMA GEMM.  Both sum the same DMMA sequence in the same order, and the second product's
    C - sum a b (fused: the accumulators start from C, A negated) and -(-C + sum a b) (unfused: alpha = -1, beta = 1,
    sign-bit flips) are the same numbers under round-to-nearest, so the Cholesky factor, Sigma^-1 and a whole N = 2048
    NLML gradient must not change by a bit.  The child process reports the 16 x 128-tile launches it made."""
    from oracle import lfm_oracle as o
    from dis_project_b200 import _lib, ops
    rng = np.random.default_rng(150)
    inputs = {}
    mine = {}
    for n in (1024, 1536):
        X = rng.standard_normal((n, 160))
        S = X @ X.T + np.diag(np.linspace(1.0, 3.0, n))
        inputs[f"S{n}"] = S
        L, Sinv, info = ops.debug_potrf_potri(torch.as_tensor(S.copy()).cuda())
        assert int(info.item()) == 0
        mine[f"L{n}"] = np.tril(L.cpu().numpy())
        mine[f"Sinv{n}"] = np.tril(Sinv.cpu().numpy())
    G, T = 16, 128
    x, y, _, _ = o.synthetic_problem(G, T, 1, seed=8)
    th = o.Params.reference_init(G).pack()
    out, info = ops.nlml_grad(x, y, th, 1e-4, G)
    assert int(info.item()) == 0
    mine["nlml_grad"] = out.cpu().numpy()
    np.savez(tmp_path / "in.npz", x=x, y=y, th=th, **inputs)
    code = f"""
import sys, ctypes, numpy as np, torch
sys.path.insert(0, {ROOT!r})
from dis_project_b200 import _lib, ops
d = np.load({str(tmp_path / 'in.npz')!r})
res = {{}}
l = _lib.lib()
l.lfm_debug_profile_begin()
for n in (1024, 1536):
    L, Sinv, info = ops.debug_potrf_potri(torch.as_tensor(d['S%d' % n]).cuda())
    assert int(info.item()) == 0
    res['L%d' % n] = np.tril(L.cpu().numpy())
    res['Sinv%d' % n] = np.tril(Sinv.cpu().numpy())
out, info = ops.nlml_grad(d['x'], d['y'], d['th'], 1e-4, {G})
assert int(info.item()) == 0
res['nlml_grad'] = out.cpu().numpy()
ms, fl, nl = ctypes.c_double(), ctypes.c_double(), ctypes.c_longlong()
l.lfm_debug_profile_end(ctypes.byref(ms), ctypes.byref(fl), ctypes.byref(nl))
l.lfm_debug_profile_chain(ctypes.byref(ms), ctypes.byref(fl), ctypes.byref(nl))
res['chain_launches'] = np.array(nl.value)
np.savez({str(tmp_path / 'out.npz')!r}, **res)
"""
    env = dict(os.environ, LFM_CHAIN_FUSED="0")
    subprocess.run([sys.executable, "-c", code], check=True, env=env, timeout=600)
    other = np.load(tmp_path / "out.npz")
    assert int(other["chain_launches"]) > 0          # the unfused path ran: 16 x 128-tile launches of the chain
    for k, v in mine.items():
        assert np.array_equal(other[k], v), k
