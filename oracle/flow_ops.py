"""Exact-order numpy model of cv2.calcOpticalFlowFarneback (flags 0, poly_n 5 or 7) -- TEST INFRASTRUCTURE ONLY.

Every float operation is written as one numpy float32 or float64 operation, in the order OpenCV's CPU code performs it
(optflowgf.cpp for the flow, filter.simd.hpp for the blur, resize.cpp for INTER_LINEAR, matrix_decomp.cpp for the Gram
inverse).  numpy and the C++ compiler both round each such operation to nearest and neither fuses a multiply with an add,
so the model reproduces cv2's scalar path (``cv2.setUseOptimized(False)``) bit for bit; tests/test_flow_oracle_cpu.py checks
that stage by stage.  Recurrences (the running box sums) loop over rows or columns; every loop body is a vector across the
pixels and pairs that do not depend on each other.  Nothing here calls cv2.

Arrays carry a leading batch axis: frames [N][H][W], flows [N][H][W][2].
"""
from __future__ import annotations

import math
from fractions import Fraction

import numpy as np

F32, F64 = np.float32, np.float64
MIN_LEVEL_SIDE = 32                     # cv2 adds no pyramid level whose side drops below this

# getGaussianKernel's fixed kernels for sigma <= 0 (getGaussianKernelBitExact)
_FIXED_TAPS = {1: [1.0], 3: [0.25, 0.5, 0.25], 5: [0.0625, 0.25, 0.375, 0.25, 0.0625],
               7: [0.03125, 0.109375, 0.21875, 0.28125, 0.21875, 0.109375, 0.03125],
               9: [4 / 256, 13 / 256, 30 / 256, 51 / 256, 60 / 256, 51 / 256, 30 / 256, 13 / 256, 4 / 256]}


# ---- Gaussian taps and pyramid geometry ---------------------------------------------------------------------------------
def gauss_taps(n: int, sigma: float) -> np.ndarray:
    """cv2.getGaussianKernel(n, sigma, CV_32F): getGaussianKernelBitExact in double (exp at doubled coordinates, sum of the
    half taps doubled plus the centre, one reciprocal), then each tap rounded to float32."""
    if sigma <= 0 and n in _FIXED_TAPS:
        return np.array(_FIXED_TAPS[n], F32)
    # sigma <= 0 otherwise: mulAdd(n, 0.15, 0.35), one rounding
    sx = float(sigma) if sigma > 0 else float(Fraction(n) * Fraction(0.15) + Fraction(0.35))
    scale2x = -0.125 / (sx * sx)
    n2 = (n - 1) // 2
    vals, s = [], 0.0
    for i in range(n2):
        x = 1 - n + 2 * i
        t = math.exp(float(x * x) * scale2x)
        vals.append(t)
        s += t
    s *= 2.0
    s += 1.0
    if n % 2 == 0:
        s += 1.0
    mul1 = 1.0 / s
    out = [0.0] * n
    for i in range(n2):
        out[i] = out[n - 1 - i] = vals[i] * mul1
    out[n2] = mul1
    if n % 2 == 0:
        out[n2 + 1] = mul1
    return np.array(out, F64).astype(F32)


def cv_round(v: float) -> int:
    """cvRound: to nearest, ties to even."""
    return int(round(v))


def pyramid(H: int, W: int, pyr_scale: float, levels: int):
    """Per level, finest first: (w, h, ksize, sigma) of calcOpticalFlowFarneback's pyramid."""
    scale, k = 1.0, 0
    while k < levels:
        scale *= pyr_scale
        if W * scale < MIN_LEVEL_SIDE or H * scale < MIN_LEVEL_SIDE:
            break
        k += 1
    out = []
    for lv in range(k + 1):
        s = 1.0
        for _ in range(lv):
            s *= pyr_scale
        sigma = (1.0 / s - 1) * 0.5
        ks = max(cv_round(sigma * 5) | 1, 3)
        out.append((cv_round(W * s), cv_round(H * s), ks, sigma))
    return out


# ---- level image --------------------------------------------------------------------------------------------------------
def reflect101(i: np.ndarray, n: int) -> np.ndarray:
    """borderInterpolate(i, n, BORDER_REFLECT_101)."""
    i = np.asarray(i, np.int64).copy()
    if n == 1:
        return np.zeros_like(i)
    while True:
        lo, hi = i < 0, i >= n
        if not (lo.any() or hi.any()):
            return i
        i = np.where(lo, -i, np.where(hi, 2 * (n - 1) - i, i))


def gaussian_blur(img: np.ndarray, taps: np.ndarray) -> np.ndarray:
    """cv2.GaussianBlur / sepFilter2D on float32 [N][H][W], REFLECT_101, scalar path.  Row pass: for ksize <= 5 the small
    symmetric filter c*k0 + (l1 + r1)*k1 + (l2 + r2)*k2, otherwise the generic filter summed left to right.  Column pass:
    the symmetric filter k0*c, then + k_i*(below_i + above_i) for i = 1..ksize/2."""
    n = len(taps)
    r = n // 2
    H, W = img.shape[-2:]
    padx = img[..., reflect101(np.arange(-r, W + r), W)]
    cols = lambda d: padx[..., r + d:r + d + W]                        # noqa: E731  cols(d)[..., x] = img[..., x + d]
    if n <= 5:
        row = cols(0) * taps[r]
        for i in range(1, r + 1):
            row = row + (cols(-i) + cols(i)) * taps[r + i]
    else:
        row = taps[0] * cols(-r)
        for j in range(1, n):
            row = row + taps[j] * cols(j - r)
    pady = row[..., reflect101(np.arange(-r, H + r), H), :]
    rows = lambda d: pady[..., r + d:r + d + H, :]                     # noqa: E731
    out = taps[r] * row + F32(0)
    for i in range(1, r + 1):
        out = out + taps[r + i] * (rows(i) + rows(-i))
    return out


def resize_taps(dst: int, src: int):
    """resizeGeneric's INTER_LINEAR table for one axis: source index and float weight per destination index."""
    scale = 1.0 / (dst / src)
    f = ((np.arange(dst, dtype=F64) + 0.5) * scale - 0.5).astype(F32)
    s = np.floor(f).astype(np.int64)
    return s, f - s.astype(F32)


def resize_linear(img: np.ndarray, w: int, h: int) -> np.ndarray:
    """cv2.resize(img, (w, h), INTER_LINEAR) on float32 [N][H][W] or [N][H][W][C], scalar path.  Horizontal ends take one
    tap of weight 1; vertical ends clamp the rows and keep both weights."""
    H, W = img.shape[1], img.shape[2]
    if (w, h) == (W, H):
        return img.copy()
    sx, fx = resize_taps(w, W)
    sy, fy = resize_taps(h, H)
    edge = (sx < 0) | (sx >= W - 1)
    fx = np.where(edge, F32(0), fx)
    sx = np.clip(sx, 0, W - 1)
    sx1 = np.minimum(sx + 1, W - 1)
    y0, y1 = np.clip(sy, 0, H - 1), np.clip(sy + 1, 0, H - 1)
    ex = (slice(None),) + (None,) * (img.ndim - 3)
    a0, a1 = (F32(1) - fx)[ex], fx[ex]
    b0, b1 = (F32(1) - fy)[(slice(None), None) + ex[1:]], fy[(slice(None), None) + ex[1:]]
    rowsx = lambda r: img[:, r][:, :, sx] * a0 + img[:, r][:, :, sx1] * a1     # noqa: E731
    out = rowsx(y0) * b0 + rowsx(y1) * b1
    if W == 2 * w and H == 2 * h:
        # An exact 2x reduction runs INTER_AREA's fast path.  Its 4-lane vector loop computes ((a + b) + (c + d)) / 4, which
        # is the formula above; the last w % 4 columns of each row take its scalar loop, (((a + b) + c) + d) / 4.
        t = (w // 4) * 4
        a, b, c, d = img[:, 0::2, 2 * t::2], img[:, 0::2, 2 * t + 1::2], img[:, 1::2, 2 * t::2], img[:, 1::2, 2 * t + 1::2]
        out[:, :, t:] = (((a + b) + c) + d) * F32(0.25)
    return out


def level_image(frames_u8: np.ndarray, w: int, h: int, ks: int, sigma: float) -> np.ndarray:
    """float32 frame -> GaussianBlur(ks, sigma) -> resize INTER_LINEAR to (w, h)."""
    img = gaussian_blur(frames_u8.astype(F32), gauss_taps(ks, sigma))
    return resize_linear(img, w, h)


# ---- polynomial expansion -----------------------------------------------------------------------------------------------
def cholesky_inverse(G) -> list:
    """Mat::inv(DECOMP_CHOLESKY) of a symmetric positive definite matrix: hal::Cholesky64f (L with reciprocal diagonal,
    then forward and back substitution against the identity), every operation in double, sums in its order."""
    m = len(G)
    L = [list(map(float, r)) for r in G]
    for i in range(m):
        for j in range(i):
            s = L[i][j]
            for k in range(j):
                s -= L[i][k] * L[j][k]
            L[i][j] = s * L[j][j]
        s = L[i][i]
        for k in range(i):
            t = L[i][k]
            s -= t * t
        L[i][i] = 1.0 / math.sqrt(s)
    b = [[1.0 if i == j else 0.0 for j in range(m)] for i in range(m)]
    for i in range(m):
        for j in range(m):
            s = b[i][j]
            for k in range(i):
                s -= L[i][k] * b[k][j]
            b[i][j] = s * L[i][i]
    for i in range(m - 1, -1, -1):
        for j in range(m):
            s = b[i][j]
            for k in range(m - 1, i, -1):
                s -= L[k][i] * b[k][j]
            b[i][j] = s * L[i][i]
    return b


def gram_matrix(n: int, sigma: float):
    """FarnebackPrepareGaussian: float32 taps g, xg, xxg for k = -n..n and the 6 x 6 Gram matrix (float products summed
    in double)."""
    if sigma < float(np.finfo(F32).eps):
        sigma = n * 0.3
    g = np.zeros(2 * n + 1, F32)
    s = 0.0
    for x in range(-n, n + 1):
        g[x + n] = F32(math.exp(-x * x / (2 * sigma * sigma)))
        s += float(g[x + n])
    s = 1.0 / s
    for x in range(-n, n + 1):
        g[x + n] = F32(float(g[x + n]) * s)
    xs = np.arange(-n, n + 1).astype(F32)
    xg, xxg = xs * g, (xs * xs) * g
    G = [[0.0] * 6 for _ in range(6)]
    for y in range(-n, n + 1):
        for x in range(-n, n + 1):
            gy, gx, fx, fy = g[y + n], g[x + n], F32(x), F32(y)
            G[0][0] += float(gy * gx)
            G[1][1] += float(gy * gx * fx * fx)
            G[3][3] += float(gy * gx * fx * fx * fx * fx)
            G[5][5] += float(gy * gx * fx * fx * fy * fy)
    G[2][2] = G[0][3] = G[0][4] = G[3][0] = G[4][0] = G[1][1]
    G[4][4] = G[3][3]
    G[3][4] = G[4][3] = G[5][5]
    return g[n:], xg[n:], xxg[n:], G


def poly_consts(n: int, sigma: float):
    """(g, xg, xxg for k = 0..n, ig11, ig03, ig33, ig55)."""
    g, xg, xxg, G = gram_matrix(n, sigma)
    ig = cholesky_inverse(G)
    return g, xg, xxg, ig[1][1], ig[0][3], ig[3][3], ig[5][5]


def poly_exp(img: np.ndarray, n: int, sigma: float) -> np.ndarray:
    """FarnebackPolyExp: float32 [N][h][w] -> R [N][h][w][5].  Vertical pass in float over k = 1..n with replicated rows,
    horizontal pass in double over k = 1..n with replicated columns."""
    g, xg, xxg, ig11, ig03, ig33, ig55 = poly_consts(n, sigma)
    h, w = img.shape[-2:]
    ry = lambda d: img[..., np.clip(np.arange(h) + d, 0, h - 1), :]       # noqa: E731
    r0, r1, r2 = img * g[0], np.zeros_like(img), np.zeros_like(img)
    for k in range(1, n + 1):
        a, b = ry(-k), ry(k)
        p = a + b
        r0 = r0 + g[k] * p
        r1 = r1 + xg[k] * (b - a)
        r2 = r2 + xxg[k] * p
    pad = np.clip(np.arange(-n, w + n), 0, w - 1)                           # replicated columns
    p0, p1, p2 = r0[..., pad], r1[..., pad], r2[..., pad]
    cx = lambda p, d: p[..., n + d:n + d + w]                               # noqa: E731
    b1 = (r0 * g[0]).astype(F64)
    b3 = (r1 * g[0]).astype(F64)
    b5 = (r2 * g[0]).astype(F64)
    b2 = np.zeros_like(b1)
    b4 = np.zeros_like(b1)
    b6 = np.zeros_like(b1)
    for k in range(1, n + 1):
        r0p, r0m, r1p, r1m, r2p, r2m = cx(p0, k), cx(p0, -k), cx(p1, k), cx(p1, -k), cx(p2, k), cx(p2, -k)
        tg = (r0p + r0m).astype(F64)
        b1 = b1 + tg * F64(g[k])
        b4 = b4 + tg * F64(xxg[k])
        b2 = b2 + ((r0p - r0m) * xg[k]).astype(F64)
        b3 = b3 + ((r1p + r1m) * g[k]).astype(F64)
        b6 = b6 + ((r1p - r1m) * xg[k]).astype(F64)
        b5 = b5 + ((r2p + r2m) * g[k]).astype(F64)
    return np.stack([b3 * ig11, b2 * ig11, b1 * ig03 + b5 * ig33, b1 * ig03 + b4 * ig33, b6 * ig55], -1).astype(F32)


# ---- update matrices ----------------------------------------------------------------------------------------------------
_BORDER = np.array([0.14, 0.14, 0.4472, 0.4472, 0.4472], F32)


def _border_lo_hi(length: int):
    i = np.arange(length)
    lo = np.where(i < 5, _BORDER[np.minimum(i, 4)], F32(1))
    hi = np.where(i >= length - 5, _BORDER[np.clip(length - i - 1, 0, 4)], F32(1))
    return lo, hi


def update_matrices(R0: np.ndarray, R1: np.ndarray, flow: np.ndarray) -> np.ndarray:
    """FarnebackUpdateMatrices: M [N][h][w][5] = (G11, G12, G22, h1, h2) for the flow [N][h][w][2]."""
    N, h, w = flow.shape[:3]
    dx, dy = flow[..., 0], flow[..., 1]
    xs = np.arange(w, dtype=F32)[None, None, :]
    ys = np.arange(h, dtype=F32)[None, :, None]
    fx, fy = xs + dx, ys + dy
    flx, fly = np.floor(fx), np.floor(fy)
    inside = (flx >= 0) & (flx < F32(w - 1)) & (fly >= 0) & (fly < F32(h - 1))      # cv2's unsigned x1 < w - 1 test
    fx, fy = fx - flx, fy - fly
    x1 = np.where(inside, flx, 0).astype(np.int64)
    y1 = np.where(inside, fly, 0).astype(np.int64)
    one = F32(1)
    a00, a01 = (one - fx) * (one - fy), fx * (one - fy)
    a10, a11 = (one - fx) * fy, fx * fy
    R1c = np.moveaxis(R1, -1, 0).reshape(5, -1)                              # channel-first gathers
    i00 = (np.arange(N)[:, None, None] * h + y1) * w + x1
    i01 = i00 + np.where(inside, 1, 0)
    i10, i11 = i00 + np.where(inside, w, 0), i01 + np.where(inside, w, 0)
    p00, p01, p10, p11 = R1c[:, i00], R1c[:, i01], R1c[:, i10], R1c[:, i11]
    r = [a00 * p00[c] + a01 * p01[c] + a10 * p10[c] + a11 * p11[c] for c in range(5)]
    q = list(np.moveaxis(R0, -1, 0))
    half, quarter = F32(0.5), F32(0.25)
    r2 = np.where(inside, r[0], F32(0))
    r3 = np.where(inside, r[1], F32(0))
    r4 = np.where(inside, (q[2] + r[2]) * half, q[2])
    r5 = np.where(inside, (q[3] + r[3]) * half, q[3])
    r6 = np.where(inside, (q[4] + r[4]) * quarter, q[4] * half)
    r2 = (q[0] - r2) * half
    r3 = (q[1] - r3) * half
    r2 = r2 + (r4 * dy + r6 * dx)
    r3 = r3 + (r6 * dy + r5 * dx)
    xi, yi = np.arange(w), np.arange(h)
    bx = ((xi - 5) % (1 << 32) >= (w - 10) % (1 << 32))[None, None, :]        # cv2's unsigned border tests
    by = ((yi - 5) % (1 << 32) >= (h - 10) % (1 << 32))[None, :, None]
    xlo, xhi = _border_lo_hi(w)
    ylo, yhi = _border_lo_hi(h)
    scale = ((xlo * xhi)[None, None, :] * ylo[None, :, None]) * yhi[None, :, None]     # ((x_lo * x_hi) * y_lo) * y_hi
    sel = bx | by
    r2, r3, r4, r5, r6 = (np.where(sel, v * scale, v) for v in (r2, r3, r4, r5, r6))
    return np.stack([r4 * r4 + r6 * r6, (r4 + r5) * r6, r5 * r5 + r6 * r6, r4 * r2 + r6 * r3, r6 * r2 + r5 * r3], -1)


# ---- box sums and solve -------------------------------------------------------------------------------------------------
def box_sums(M: np.ndarray, winsize: int) -> np.ndarray:
    """FarnebackUpdateFlow_Blur's running sums: float32 M [N][h][w][5] -> unscaled double sums.  The vertical sum adds the
    float32 difference of the entering and leaving rows, the horizontal one the double difference of the columns.  Both
    start from the edge taken m + 2 times plus entries 1..m-1 (clamped), which for winsize 1 adds row 0 and column 0."""
    h, w = M.shape[1], M.shape[2]
    m = winsize // 2
    V = np.empty(M.shape, F64)
    v = (M[:, 0] * F32(m + 2)).astype(F64)
    for r in range(1, m):
        v = v + M[:, min(r, h - 1)].astype(F64)
    for y in range(h):
        v = v + (M[:, min(y + m, h - 1)] - M[:, max(y - m - 1, 0)]).astype(F64)
        V[:, y] = v
    S = np.empty_like(V)
    g = V[:, :, 0] * F64(m + 2)
    for x in range(1, m):
        g = g + V[:, :, min(x, w - 1)]
    for x in range(w):
        g = g + (V[:, :, min(x + m, w - 1)] - V[:, :, max(x - m - 1, 0)])
        S[:, :, x] = g
    return S


def solve(S: np.ndarray, winsize: int) -> np.ndarray:
    """Box sums scaled by 1 / winsize^2, then the regularised 2 x 2 solve: flow [N][h][w][2] float32."""
    scale = 1.0 / (winsize * winsize)
    g11, g12, g22, h1, h2 = (S[..., c] * scale for c in range(5))
    idet = 1.0 / (g11 * g22 - g12 * g12 + 1e-3)
    return np.stack([(g11 * h2 - g12 * h1) * idet, (g22 * h1 - g12 * h2) * idet], -1).astype(F32)


# ---- driver -------------------------------------------------------------------------------------------------------------
def _check(pyr_scale, levels, winsize, iterations, poly_n, flags):
    if flags != 0 or poly_n not in (5, 7):
        raise NotImplementedError("the model covers flags 0 and poly_n 5 / 7")
    if not (0 < pyr_scale < 1) or levels < 0 or winsize < 1 or iterations < 1:
        raise ValueError("bad Farneback parameters")


def poly_pyramid(frames_u8: np.ndarray, pyr, poly_n: int, poly_sigma: float):
    """Per level (finest first): R [N][h][w][5] of every frame."""
    return [poly_exp(level_image(frames_u8, w, h, ks, sigma), poly_n, poly_sigma) for (w, h, ks, sigma) in pyr]


def flow_from_pyramids(P0, P1, pyr, pyr_scale: float, winsize: int, iterations: int) -> np.ndarray:
    """Coarse to fine: the starting flow (zero, or the coarser flow resized INTER_LINEAR times float32(1 / pyr_scale)
    through cv2's x * a + 0), its matrices, then `iterations` rounds of box sum and solve."""
    flow = None
    up = F32(1.0 / pyr_scale)
    for lv in range(len(pyr) - 1, -1, -1):
        w, h = pyr[lv][0], pyr[lv][1]
        R0, R1 = P0[lv], P1[lv]
        if flow is None:
            flow = np.zeros(R0.shape[:3] + (2,), F32)
        else:
            flow = resize_linear(flow, w, h) * up + F32(0)
        M = update_matrices(R0, R1, flow)
        for it in range(iterations):
            flow = solve(box_sums(M, winsize), winsize)
            if it < iterations - 1:
                M = update_matrices(R0, R1, flow)
    return flow


def farneback(prev: np.ndarray, next: np.ndarray, pyr_scale: float = 0.3, levels: int = 2, winsize: int = 9,
              iterations: int = 2, poly_n: int = 5, poly_sigma: float = 1.1, flags: int = 0) -> np.ndarray:
    """cv2.calcOpticalFlowFarneback(prev, next, None, ...) for uint8 [H][W] or [N][H][W] pairs -> float32 flow."""
    _check(pyr_scale, levels, winsize, iterations, poly_n, flags)
    single = prev.ndim == 2
    p, q = (prev[None], next[None]) if single else (prev, next)
    pyr = pyramid(p.shape[1], p.shape[2], pyr_scale, levels)
    flow = flow_from_pyramids(poly_pyramid(p, pyr, poly_n, poly_sigma), poly_pyramid(q, pyr, poly_n, poly_sigma), pyr,
                              pyr_scale, winsize, iterations)
    return flow[0] if single else flow


def magnitude(flow: np.ndarray) -> np.ndarray:
    """cv2.cartToPolar's magnitude in float32: sqrt(fx * fx + fy * fy)."""
    fx, fy = flow[..., 0], flow[..., 1]
    return np.sqrt(fx * fx + fy * fy)


def flow_masks(grays: np.ndarray, flow_threshold: float, pyr_scale: float = 0.3, levels: int = 2, winsize: int = 9,
               iterations: int = 2, poly_n: int = 5, poly_sigma: float = 1.1, flags: int = 0) -> np.ndarray:
    """Raw masks of a gray sequence [N+1][H][W]: mask i = 255 where |flow(frame i -> frame i + 1)| > float32(thr)."""
    _check(pyr_scale, levels, winsize, iterations, poly_n, flags)
    pyr = pyramid(grays.shape[1], grays.shape[2], pyr_scale, levels)
    P = poly_pyramid(grays, pyr, poly_n, poly_sigma)
    flow = flow_from_pyramids([r[:-1] for r in P], [r[1:] for r in P], pyr, pyr_scale, winsize, iterations)
    return (magnitude(flow) > F32(flow_threshold)).astype(np.uint8) * 255
