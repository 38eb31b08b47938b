// Dense optical flow: cv2.calcOpticalFlowFarneback (motion_compression_opt.py:72-81) with flags 0, box-filtered solve.
//
// The stages follow OpenCV's CPU code (optflowgf.cpp) and were pinned down against cv2 4.13 as a black box:
//   level image   float32 frame -> GaussianBlur(ksize, sigma), REFLECT_101 -> resize INTER_LINEAR   k_flow_level
//   polynomial    separable Gaussian-weighted fit, replicated borders, 5 coefficients per pixel       k_flow_poly
//   matrices      R1 sampled bilinearly at x + flow, border taper, M = (G11, G12, G22, h1, h2)       k_flow_matrices
//   box sum       cv2's vertical and horizontal running sums, in cv2's order                         k_flow_vsum, k_flow_hsum
//   solve         regularised 2x2 solve (+1e-3), then either the next matrices or the mask           k_flow_solve
// Float products and sums that cv2 rounds one by one are written with __fmul_rn / __fadd_rn so that ptxas cannot
// contract them.  Every sum has a fixed order: results are identical from run to run.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"
#include "k_front.cuh"      // reflect101 (BORDER_REFLECT_101)

namespace dvc {

constexpr int FLOW_MAX_POLY_N = 7;
constexpr int FLOW_MAX_BLUR_HALF = 127;      // GaussianBlur ksize <= 255 per pyramid level

// FarnebackPrepareGaussian: taps for k = 0..n (the fit only reads the non-negative half) and the inverse-Gram constants.
struct FlowPolyTab {
    float g[FLOW_MAX_POLY_N + 1], xg[FLOW_MAX_POLY_N + 1], xxg[FLOW_MAX_POLY_N + 1];
    double ig11, ig03, ig33, ig55;
    int n;
};

// One pyramid level's image: the symmetric half of the float32 Gaussian kernel (k[0] = centre) and the resize geometry.
struct FlowLevelGeom {
    float k[FLOW_MAX_BLUR_HALF + 1];
    int half;                   // ksize / 2
    int w, h;                   // level size
    double scale_x, scale_y;    // cv2.resize's 1 / (dst / src)
};

// cv2.resize INTER_LINEAR source index and weight of destination index d (resizeGeneric's table)
DEVI void resize_tap(int d, double scale, int& s, float& f) {
    const float fx = (float)__dadd_rn(__dmul_rn((double)d + 0.5, scale), -0.5);
    s = (int)floorf(fx);
    f = __fsub_rn(fx, (float)s);
}

// ---- level image ---------------------------------------------------------------------------------------------------
// Row filter then column filter (cv2's separable order), each as k0 * c + sum k_i * (l_i + r_i).
DEVI float blur_row(const uint8_t* src, int W, int r, int c, const FlowLevelGeom& g) {
    const uint8_t* row = src + (size_t)r * W;
    float s = __fmul_rn((float)row[c], g.k[0]);
    for (int i = 1; i <= g.half; ++i)
        s = __fadd_rn(s, __fmul_rn(g.k[i], __fadd_rn((float)row[reflect101(c - i, W)], (float)row[reflect101(c + i, W)])));
    return s;
}
DEVI float blur_at(const uint8_t* src, int H, int W, int r, int c, const FlowLevelGeom& g) {
    float s = __fmul_rn(blur_row(src, W, r, c, g), g.k[0]);
    for (int i = 1; i <= g.half; ++i)
        s = __fadd_rn(s, __fmul_rn(g.k[i], __fadd_rn(blur_row(src, W, reflect101(r - i, H), c, g),
                                                      blur_row(src, W, reflect101(r + i, H), c, g))));
    return s;
}

// grid (ceil(w*h / 256), frames): dst[f] = resize(GaussianBlur(float(src[f])), (w, h))
__global__ void __launch_bounds__(256) k_flow_level(const uint8_t* __restrict__ src, int H, int W, float* __restrict__ dst,
                                                    size_t dst_stride, FlowLevelGeom g) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= g.w * g.h) return;
    const int x = idx % g.w, y = idx / g.w;
    src += (size_t)blockIdx.y * H * W;
    float v;
    if (g.w == W && g.h == H) {                          // cv2.resize to the same size copies
        v = blur_at(src, H, W, y, x, g);
    } else {
        int sx, sy;
        float fx, fy;
        resize_tap(x, g.scale_x, sx, fx);
        resize_tap(y, g.scale_y, sy, fy);
        if (sx < 0) { sx = 0; fx = 0.f; }               // horizontal ends: one tap with weight 1
        if (sx >= W - 1) { sx = W - 1; fx = 0.f; }
        const int sx1 = min(sx + 1, W - 1);
        const int y0 = min(max(sy, 0), H - 1), y1 = min(max(sy + 1, 0), H - 1);    // vertical ends: clamped rows
        const float a0 = __fsub_rn(1.f, fx), b0 = __fsub_rn(1.f, fy);
        const float h0 = __fadd_rn(__fmul_rn(blur_at(src, H, W, y0, sx, g), a0), __fmul_rn(blur_at(src, H, W, y0, sx1, g), fx));
        const float h1 = __fadd_rn(__fmul_rn(blur_at(src, H, W, y1, sx, g), a0), __fmul_rn(blur_at(src, H, W, y1, sx1, g), fx));
        v = __fadd_rn(__fmul_rn(h0, b0), __fmul_rn(h1, fy));
    }
    dst[(size_t)blockIdx.y * dst_stride + idx] = v;
}

// ---- polynomial expansion (FarnebackPolyExp) ---------------------------------------------------------------------------
constexpr int POLY_TW = 32, POLY_TH = 8;

// grid (ceil(w/32), ceil(h/8), frames), block 256: img [h][w] -> R [h][w][5]
__global__ void __launch_bounds__(256) k_flow_poly(const float* __restrict__ img, size_t img_stride, int w, int h,
                                                   float* __restrict__ R, size_t R_stride, FlowPolyTab t) {
    __shared__ float row[POLY_TH][POLY_TW + 2 * FLOW_MAX_POLY_N][3];
    const int n = t.n, tw = POLY_TW + 2 * n;
    const int x0 = blockIdx.x * POLY_TW, y0 = blockIdx.y * POLY_TH;
    img += (size_t)blockIdx.z * img_stride;
    // vertical part: float, k = 1..n in order; columns outside the image replicate the edge column
    for (int i = threadIdx.x; i < POLY_TH * tw; i += blockDim.x) {
        const int ry = i / tw, cx = i % tw;
        const int y = min(y0 + ry, h - 1), x = min(max(x0 + cx - n, 0), w - 1);
        float r0 = __fmul_rn(img[(size_t)y * w + x], t.g[0]), r1 = 0.f, r2 = 0.f;
        for (int k = 1; k <= n; ++k) {
            const float a = img[(size_t)max(y - k, 0) * w + x], b = img[(size_t)min(y + k, h - 1) * w + x];
            const float p = __fadd_rn(a, b);
            r0 = __fadd_rn(r0, __fmul_rn(t.g[k], p));
            r1 = __fadd_rn(r1, __fmul_rn(t.xg[k], __fsub_rn(b, a)));
            r2 = __fadd_rn(r2, __fmul_rn(t.xxg[k], p));
        }
        row[ry][cx][0] = r0; row[ry][cx][1] = r1; row[ry][cx][2] = r2;
    }
    __syncthreads();
    const int tx = threadIdx.x % POLY_TW, ty = threadIdx.x / POLY_TW;
    const int x = x0 + tx, y = y0 + ty;
    if (x >= w || y >= h) return;
    const float (*c)[3] = row[ty] + tx + n;          // c[k] = column x + k
    const float g0 = t.g[0];
    double b1 = __fmul_rn(c[0][0], g0), b2 = 0, b3 = __fmul_rn(c[0][1], g0), b4 = 0, b5 = __fmul_rn(c[0][2], g0), b6 = 0;
    for (int k = 1; k <= n; ++k) {
        const double tg = __fadd_rn(c[k][0], c[-k][0]);
        b1 = __dadd_rn(b1, __dmul_rn(tg, (double)t.g[k]));
        b4 = __dadd_rn(b4, __dmul_rn(tg, (double)t.xxg[k]));
        b2 = __dadd_rn(b2, (double)__fmul_rn(__fsub_rn(c[k][0], c[-k][0]), t.xg[k]));
        b3 = __dadd_rn(b3, (double)__fmul_rn(__fadd_rn(c[k][1], c[-k][1]), t.g[k]));
        b6 = __dadd_rn(b6, (double)__fmul_rn(__fsub_rn(c[k][1], c[-k][1]), t.xg[k]));
        b5 = __dadd_rn(b5, (double)__fmul_rn(__fadd_rn(c[k][2], c[-k][2]), t.g[k]));
    }
    float* d = R + (size_t)blockIdx.z * R_stride + ((size_t)y * w + x) * 5;
    d[0] = (float)__dmul_rn(b3, t.ig11);
    d[1] = (float)__dmul_rn(b2, t.ig11);
    d[2] = (float)__dadd_rn(__dmul_rn(b1, t.ig03), __dmul_rn(b5, t.ig33));
    d[3] = (float)__dadd_rn(__dmul_rn(b1, t.ig03), __dmul_rn(b4, t.ig33));
    d[4] = (float)__dmul_rn(b6, t.ig55);
}

// ---- update matrices (FarnebackUpdateMatrices) for one pixel -----------------------------------------------------------
DEVI float flow_border(int i, int len) {
    const float tab[5] = {0.14f, 0.14f, 0.4472f, 0.4472f, 0.4472f};
    return __fmul_rn(i < 5 ? tab[i] : 1.f, i >= len - 5 ? tab[len - i - 1] : 1.f);
}

DEVI void flow_matrix(const float* __restrict__ R0, const float* __restrict__ R1, int w, int h, int x, int y, float dx, float dy,
                      float* __restrict__ M) {
    const float* r0 = R0 + ((size_t)y * w + x) * 5;
    float fx = __fadd_rn((float)x, dx), fy = __fadd_rn((float)y, dy);
    const float flx = floorf(fx), fly = floorf(fy);
    float r2, r3, r4, r5, r6;
    if (flx >= 0.f && flx < (float)(w - 1) && fly >= 0.f && fly < (float)(h - 1)) {     // cv2's unsigned x1 < w - 1 test
        const int x1 = (int)flx, y1 = (int)fly;
        fx = __fsub_rn(fx, flx);
        fy = __fsub_rn(fy, fly);
        const float a00 = __fmul_rn(__fsub_rn(1.f, fx), __fsub_rn(1.f, fy)), a01 = __fmul_rn(fx, __fsub_rn(1.f, fy));
        const float a10 = __fmul_rn(__fsub_rn(1.f, fx), fy), a11 = __fmul_rn(fx, fy);
        const float* p = R1 + ((size_t)y1 * w + x1) * 5;
        const float* q = p + (size_t)w * 5;
        float r[5];
#pragma unroll
        for (int c = 0; c < 5; ++c)
            r[c] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(a00, p[c]), __fmul_rn(a01, p[c + 5])), __fmul_rn(a10, q[c])),
                             __fmul_rn(a11, q[c + 5]));
        r2 = r[0]; r3 = r[1];
        r4 = __fmul_rn(__fadd_rn(r0[2], r[2]), 0.5f);
        r5 = __fmul_rn(__fadd_rn(r0[3], r[3]), 0.5f);
        r6 = __fmul_rn(__fadd_rn(r0[4], r[4]), 0.25f);
    } else {
        r2 = r3 = 0.f;
        r4 = r0[2];
        r5 = r0[3];
        r6 = __fmul_rn(r0[4], 0.5f);
    }
    r2 = __fmul_rn(__fsub_rn(r0[0], r2), 0.5f);
    r3 = __fmul_rn(__fsub_rn(r0[1], r3), 0.5f);
    r2 = __fadd_rn(r2, __fadd_rn(__fmul_rn(r4, dy), __fmul_rn(r6, dx)));
    r3 = __fadd_rn(r3, __fadd_rn(__fmul_rn(r6, dy), __fmul_rn(r5, dx)));
    if ((unsigned)(x - 5) >= (unsigned)(w - 10) || (unsigned)(y - 5) >= (unsigned)(h - 10)) {
        const float s = __fmul_rn(flow_border(x, w), flow_border(y, h));
        r2 = __fmul_rn(r2, s); r3 = __fmul_rn(r3, s); r4 = __fmul_rn(r4, s); r5 = __fmul_rn(r5, s); r6 = __fmul_rn(r6, s);
    }
    M[0] = __fadd_rn(__fmul_rn(r4, r4), __fmul_rn(r6, r6));
    M[1] = __fmul_rn(__fadd_rn(r4, r5), r6);
    M[2] = __fadd_rn(__fmul_rn(r5, r5), __fmul_rn(r6, r6));
    M[3] = __fadd_rn(__fmul_rn(r4, r2), __fmul_rn(r6, r3));
    M[4] = __fadd_rn(__fmul_rn(r6, r2), __fmul_rn(r5, r3));
}

// Pair p reads R0 + p * r_stride and R1 + p * r_stride (sequence: R1 = R0 + one frame); M, V and flow are [p][h][w][...]
// with a stride of `px_stride` pixels.
struct FlowPair {
    const float* R0;
    const float* R1;
    size_t r_stride, px_stride;
    int w, h;
};

// grid (ceil(w*h / 256), pairs): the level's starting flow (zero, or the coarser level's flow resized INTER_LINEAR and
// multiplied by 1 / pyr_scale) and its matrices
__global__ void __launch_bounds__(256) k_flow_matrices(FlowPair pr, const float2* __restrict__ coarse, int cw, int ch,
                                                       double scale_x, double scale_y, float up, float* __restrict__ M) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= pr.w * pr.h) return;
    const int x = idx % pr.w, y = idx / pr.w;
    const size_t p = blockIdx.y;
    float dx = 0.f, dy = 0.f;
    if (coarse) {
        const float2* c = coarse + p * pr.px_stride;
        int sx, sy;
        float fx, fy;
        resize_tap(x, scale_x, sx, fx);
        resize_tap(y, scale_y, sy, fy);
        if (sx < 0) { sx = 0; fx = 0.f; }
        if (sx >= cw - 1) { sx = cw - 1; fx = 0.f; }
        const int sx1 = min(sx + 1, cw - 1);
        const int y0 = min(max(sy, 0), ch - 1), y1 = min(max(sy + 1, 0), ch - 1);
        const float a0 = __fsub_rn(1.f, fx), b0 = __fsub_rn(1.f, fy);
        const float2 p00 = c[(size_t)y0 * cw + sx], p01 = c[(size_t)y0 * cw + sx1];
        const float2 p10 = c[(size_t)y1 * cw + sx], p11 = c[(size_t)y1 * cw + sx1];
        const float hx0 = __fadd_rn(__fmul_rn(p00.x, a0), __fmul_rn(p01.x, fx)), hx1 = __fadd_rn(__fmul_rn(p10.x, a0), __fmul_rn(p11.x, fx));
        const float hy0 = __fadd_rn(__fmul_rn(p00.y, a0), __fmul_rn(p01.y, fx)), hy1 = __fadd_rn(__fmul_rn(p10.y, a0), __fmul_rn(p11.y, fx));
        dx = __fmul_rn(__fadd_rn(__fmul_rn(hx0, b0), __fmul_rn(hx1, fy)), up);
        dy = __fmul_rn(__fadd_rn(__fmul_rn(hy0, b0), __fmul_rn(hy1, fy)), up);
    }
    float m[5];
    flow_matrix(pr.R0 + p * pr.r_stride, pr.R1 + p * pr.r_stride, pr.w, pr.h, x, y, dx, dy, m);
    float* d = M + (p * pr.px_stride + idx) * 5;
#pragma unroll
    for (int c = 0; c < 5; ++c) d[c] = m[c];
}

// ---- box sum (FarnebackUpdateFlow_Blur's running sums) -------------------------------------------------------------------
// cv2 keeps one running double per column: vsum = M[0] * (m + 2) + M[1] + ... + M[m - 1], then per row y it adds the float
// difference M[min(y + m, h - 1)] - M[max(y - m - 1, 0)]; along each row it keeps one running double per channel,
// g = vsum[0] * (m + 2) + vsum[1] + ... + vsum[m - 1], then per x adds vsum[min(x + m, w - 1)] - vsum[max(x - m - 1, 0)].
// The flow of ill-conditioned pixels and of flat regions (where the sums do not return to exactly zero) depends on every one
// of those roundings, so both recurrences run serially, in cv2's order: one thread per column (k_flow_vsum) and one per
// row and channel (k_flow_hsum).  For m = 0 the recurrences yield M[y][x] + M[0][x] + M[y][0] + M[0][0], which is cv2's box
// for winsize 1, and that is what is reproduced.
// grid (ceil(w*5 / 128), pairs), block 128: M [h][w][5] float -> V [h][w][5] double
__global__ void __launch_bounds__(128) k_flow_vsum(const float* __restrict__ M, double* __restrict__ V, int w, int h, int m,
                                                   size_t px_stride) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x, cols = w * 5;
    if (col >= cols) return;
    const size_t base = (size_t)blockIdx.y * px_stride * 5 + col;
    const float* Mc = M + base;
    double* Vc = V + base;
    double v = (double)__fmul_rn(Mc[0], (float)(m + 2));
    for (int r = 1; r < m; ++r) v = __dadd_rn(v, (double)Mc[(size_t)min(r, h - 1) * cols]);
    for (int y = 0; y < h; ++y) {
        v = __dadd_rn(v, (double)__fsub_rn(Mc[(size_t)min(y + m, h - 1) * cols], Mc[(size_t)max(y - m - 1, 0) * cols]));
        Vc[(size_t)y * cols] = v;
    }
}

// grid (ceil(h*5 / 128), pairs), block 128: V -> S [h][w][5] double, the unscaled box sums
__global__ void __launch_bounds__(128) k_flow_hsum(const double* __restrict__ V, double* __restrict__ S, int w, int h, int m,
                                                   size_t px_stride) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= h * 5) return;
    const int y = t / 5, c = t % 5;
    const size_t base = ((size_t)blockIdx.y * px_stride + (size_t)y * w) * 5 + c;
    const double* v = V + base;
    double* o = S + base;
    double g = __dmul_rn(v[0], (double)(m + 2));
    for (int x = 1; x < m; ++x) g = __dadd_rn(g, v[(size_t)min(x, w - 1) * 5]);
    for (int x = 0; x < w; ++x) {
        g = __dadd_rn(g, __dsub_rn(v[(size_t)min(x + m, w - 1) * 5], v[(size_t)max(x - m - 1, 0) * 5]));
        o[(size_t)x * 5] = g;
    }
}

// ---- solve ------------------------------------------------------------------------------------------------------------
// Box sums scaled by 1 / winsize^2, then the regularised solve.  Outputs: the flow (flow != NULL), the mask
// 255 * (|flow| > thr) (mask != NULL), and the matrices of the new flow for the next iteration (M != NULL).
// grid (ceil(w*h / 256), pairs)
__global__ void __launch_bounds__(256) k_flow_solve(FlowPair pr, const double* __restrict__ S, double scale,
                                                    float2* __restrict__ flow, size_t flow_stride, uint8_t* __restrict__ mask,
                                                    size_t mask_stride, float thr, float* __restrict__ M) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int w = pr.w, h = pr.h;
    if (idx >= w * h) return;
    const int x = idx % w, y = idx / w;
    const size_t p = blockIdx.y;
    const double* s = S + (p * pr.px_stride + idx) * 5;
    const double g11 = __dmul_rn(s[0], scale), g12 = __dmul_rn(s[1], scale), g22 = __dmul_rn(s[2], scale);
    const double h1 = __dmul_rn(s[3], scale), h2 = __dmul_rn(s[4], scale);
    const double idet = 1.0 / __dadd_rn(__dsub_rn(__dmul_rn(g11, g22), __dmul_rn(g12, g12)), 1e-3);
    const float fx = (float)__dmul_rn(__dsub_rn(__dmul_rn(g11, h2), __dmul_rn(g12, h1)), idet);
    const float fy = (float)__dmul_rn(__dsub_rn(__dmul_rn(g22, h1), __dmul_rn(g12, h2)), idet);
    if (flow) flow[p * flow_stride + idx] = make_float2(fx, fy);
    if (mask) {                                                   // cv2.cartToPolar magnitude, then mag > thr
        const float mag = __fsqrt_rn(__fadd_rn(__fmul_rn(fx, fx), __fmul_rn(fy, fy)));
        mask[p * mask_stride + idx] = mag > thr ? 255 : 0;
    }
    if (M) {
        float mm[5];
        flow_matrix(pr.R0 + p * pr.r_stride, pr.R1 + p * pr.r_stride, w, h, x, y, fx, fy, mm);
        float* d = M + (p * pr.px_stride + idx) * 5;
#pragma unroll
        for (int c = 0; c < 5; ++c) d[c] = mm[c];
    }
}

}  // namespace dvc
