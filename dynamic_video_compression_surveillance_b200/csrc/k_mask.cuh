// K2 / K3: everything that happens to the motion mask between the threshold and the degrade kernel,
// done on bit-planes (see common.cuh).
//   k_window_vote   deque(maxlen=K) + np.sum + compare (motion_compression_opt.py:61,84-86):
//                   ring buffer of raw masks in HBM/L2, running per-pixel count kept bit-sliced in
//                   registers while a thread walks a segment of frames (add the new plane, subtract the
//                   evicted one) instead of re-summing the window
//   k_ema           cv2.addWeighted(acc, rf, dilated, 1-rf, 0) (frame_differencing.py:107): the uint8
//                   accumulator plane is stream state; per frame the kernel emits the two bit-planes the
//                   rest of the loop needs: acc > 127 (overlay, :111) and acc != 0 (block test, :120)
//   k_morph_chain   cv2.erode / dilate / morphologyEx chains (frame_differencing.py:106,
//                   motion_compression_opt.py:89-90): a row band plus halo is staged into shared memory
//                   with one cp.async.bulk (TMA) copy, every primitive of the chain runs out of shared
//                   memory (separable OR-doubling: the binary form of van Herk/Gil-Werman), one
//                   write of the final band
//   k_mlarge_*      primitives whose element is larger than MORPH_MAX_K: doubling tables for the horizontal runs, van Herk
//                   down the columns for rectangles, one launch group per primitive between global bit-planes
#pragma once
#include "common.cuh"
#include "k_front.cuh"

namespace dvc {

// ------------------------------------------------------------------------------------------------
// window vote
// ------------------------------------------------------------------------------------------------
constexpr int WINDOW_MAX = 127;        // window_size limit: the bit-sliced count has 5 bits up to 31 frames, 7 bits beyond
struct MinCounts { uint8_t v[128]; };  // v[L-1] = smallest count that passes with L masks in the window

template <int CB>
DEVI void bs_add(uint32_t (&c)[CB], uint32_t x) {
#pragma unroll
    for (int i = 0; i < CB; ++i) { uint32_t t = c[i] & x; c[i] ^= x; x = t; }
}
template <int CB>
DEVI void bs_sub(uint32_t (&c)[CB], uint32_t x) {
#pragma unroll
    for (int i = 0; i < CB; ++i) { uint32_t t = ~c[i] & x; c[i] ^= x; x = t; }
}
template <int CB>
DEVI uint32_t bs_ge(const uint32_t (&c)[CB], uint32_t m) {   // per-lane count >= m
    if (m >= (1u << CB)) return 0u;
    uint32_t ge = 0xffffffffu;
#pragma unroll
    for (int i = 0; i < CB; ++i) ge = ((m >> i) & 1u) ? (c[i] & ge) : (c[i] | ge);
    return ge;
}

// slot0 = slot of frame f0 in the ring; all slot arithmetic is 32-bit with wrap-around compares
template <int CNT_BITS>
__global__ void __launch_bounds__(256)
k_window_vote(const uint32_t* __restrict__ ring, int ring_cap, int H, int W, int wpr, long long f0, int slot0, int T,
              int K, const __grid_constant__ MinCounts mc, uint32_t* __restrict__ voted, int seg_len) {
    __shared__ uint8_t s_mc[128];
    if (threadIdx.x < 128) s_mc[threadIdx.x] = mc.v[threadIdx.x];
    __syncthreads();
    const size_t plane_words = (size_t)H * wpr;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= plane_words) return;
    ring += (size_t)blockIdx.z * ring_cap * plane_words;          // blockIdx.z = stream of a lock-step group
    voted += (size_t)blockIdx.z * T * plane_words;
    const int t0 = blockIdx.y * seg_len, t1 = min(T, t0 + seg_len);
    const uint32_t vm = valid_mask((int)(idx % wpr), W);
    uint32_t c[CNT_BITS] = {};
    const long long fs = f0 + t0;
    int s_new = (slot0 + t0) % ring_cap;
    const int nh = (int)min((long long)(K - 1), fs);       // history planes fs-nh .. fs-1
    int s = s_new - nh;
    if (s < 0) s += ring_cap;
    for (int i = 0; i < nh; ++i) {
        bs_add(c, ring[(size_t)s * plane_words + idx]);
        s = s + 1 == ring_cap ? 0 : s + 1;
    }
    int s_old = s_new - K;                                  // slot of the plane leaving the window
    if (s_old < 0) s_old += ring_cap;
    int L = nh;                                             // masks in the window before adding frame t
    // The counter chain is serial in t, the plane loads are not: the entering and leaving words of eight frames are fetched
    // together (sixteen L2 loads in flight), then the counters are walked.
    constexpr int PF = 8;
    for (int tb = t0; tb < t1; tb += PF) {
        uint32_t w_new[PF], w_old[PF];
        int sn = s_new, so = s_old;
#pragma unroll
        for (int u = 0; u < PF; ++u) {
            const bool live = tb + u < t1;
            w_new[u] = live ? ring[(size_t)sn * plane_words + idx] : 0u;
            // frame t evicts a plane once the window is full and t is not the first frame of the segment (whose history was
            // added above without the evicted plane)
            const bool evict = live && (L + u >= K) && (tb + u > t0);
            w_old[u] = evict ? ring[(size_t)so * plane_words + idx] : 0u;
            sn = sn + 1 == ring_cap ? 0 : sn + 1;
            so = so + 1 == ring_cap ? 0 : so + 1;
        }
#pragma unroll
        for (int u = 0; u < PF; ++u) {
            const int t = tb + u;
            if (t < t1) {
                if (L == K) { if (t > t0) bs_sub(c, w_old[u]); }
                else ++L;
                bs_add(c, w_new[u]);
                voted[(size_t)t * plane_words + idx] = bs_ge(c, s_mc[L - 1]) & vm;
            }
        }
        s_new = sn; s_old = so;
    }
}

// ------------------------------------------------------------------------------------------------
// K1 + K2 fused (window mode, window_size <= 8): the K1 thread that turns 16 pixels of a segment of frames into raw mask
// bits also keeps their window count (bit-sliced, 4 bits per pixel in four registers) and the last K raw pieces (a 128-bit
// shift register), so the vote costs a dozen ALU instructions per frame instead of a second kernel that re-reads the ring
// (motion_compression_opt.py:84-86 on top of frame_differencing.py:92,96-97).  A segment that does not start the batch
// rebuilds its K - 1 frames of history from the frames themselves (K extra frame reads per segment: segments are long);
// the first segment reads the previous batch's raw planes from the ring.  The ring is still written: it is the stream's
// mask_queue state (dvc_get_state) and the next batch's history.
// ------------------------------------------------------------------------------------------------
template <int K>
__global__ void __launch_bounds__(256)
k_gray_diff_vote(const uint8_t* __restrict__ frames, int T, int H, int W, const uint8_t* __restrict__ prev_gray_in,
                 uint8_t* __restrict__ gray_state_out, uint32_t* __restrict__ ring, int wpr, int ring_cap, long long f0,
                 uint32_t thr, int seg_len, const __grid_constant__ MinCounts mc, uint32_t* __restrict__ voted) {
    const int gpr = W >> 4;                                     // W % 16 == 0 (host guarantees)
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)gpr * H) return;
    const int y = (int)(gid / gpr), gx = (int)(gid % gpr), x0 = gx << 4;
    const int t0 = blockIdx.y * seg_len, t1 = min(T, t0 + seg_len);
    const size_t frame_bytes = (size_t)H * W * 3, plane_bytes = (size_t)H * W, plane_words = (size_t)H * wpr;
    const size_t row_off = (size_t)y * W * 3 + (size_t)x0 * 3, px_off = (size_t)y * W + x0;
    {
        const size_t s = blockIdx.z;
        frames += s * T * frame_bytes;
        prev_gray_in += s * plane_bytes;
        if (gray_state_out) gray_state_out += s * plane_bytes;
        ring += s * ring_cap * plane_words;
        voted += s * T * plane_words;
    }
    uint16_t* const ring16 = reinterpret_cast<uint16_t*>(ring) + (size_t)y * wpr * 2 + gx;
    uint16_t* const vote16 = reinterpret_cast<uint16_t*>(voted) + (size_t)y * wpr * 2 + gx;
    auto gray_of_frame = [&](int t, uint32_t (&g)[4]) {
        const uint8_t* fr = frames + (size_t)t * frame_bytes + row_off;
        uint32_t w[12];
        load16(fr, *reinterpret_cast<uint32_t(*)[4]>(&w[0]));
        load16(fr + 16, *reinterpret_cast<uint32_t(*)[4]>(&w[4]));
        load16(fr + 32, *reinterpret_cast<uint32_t(*)[4]>(&w[8]));
        gray16_dp2a(w, g);
    };
    uint32_t hst[4] = {0u, 0u, 0u, 0u};                          // raw pieces, newest in the low half of hst[0]
    uint32_t c[4] = {0u, 0u, 0u, 0u};                            // bit-sliced count of the window (<= 8)
    auto push = [&](uint32_t b) {
        hst[3] = __funnelshift_l(hst[2], hst[3], 16); hst[2] = __funnelshift_l(hst[1], hst[2], 16);
        hst[1] = __funnelshift_l(hst[0], hst[1], 16); hst[0] = (hst[0] << 16) | b;
    };
    auto add = [&](uint32_t x) {
#pragma unroll
        for (int i = 0; i < 4; ++i) { const uint32_t tt = c[i] & x; c[i] ^= x; x = tt; }
    };
    auto sub = [&](uint32_t x) {
#pragma unroll
        for (int i = 0; i < 4; ++i) { const uint32_t tt = ~c[i] & x; c[i] ^= x; x = tt; }
    };
    const long long fs = f0 + t0;                               // stream index of the segment's first frame
    int nin = (int)min((long long)(K - 1), fs);                 // raw masks in the window before frame t0
    uint32_t pg[4];
    if (t0 == 0) {
        load16(prev_gray_in + px_off, pg);
        for (int i = nin; i >= 1; --i) {                         // previous batch's planes, oldest first
            const uint32_t b = ring16[(size_t)((f0 - i) % ring_cap) * plane_words * 2];
            push(b); add(b);
        }
    } else {
        gray_of_frame(t0 - nin - 1, pg);                         // t0 >= seg_len >= K: these frames are in this batch
        for (int t = t0 - nin; t < t0; ++t) {
            uint32_t g[4];
            gray_of_frame(t, g);
            const uint32_t b = diff_gt_bits16(g, pg, thr);
#pragma unroll
            for (int q = 0; q < 4; ++q) pg[q] = g[q];
            push(b); add(b);
        }
    }
    for (int t = t0; t < t1; ++t) {
        uint32_t g[4];
        gray_of_frame(t, g);
        const uint32_t b = diff_gt_bits16(g, pg, thr);
#pragma unroll
        for (int q = 0; q < 4; ++q) pg[q] = g[q];
        if (nin == K) sub((hst[(K - 1) >> 1] >> (((K - 1) & 1) * 16)) & 0xffffu);      // the piece pushed K frames ago leaves
        else ++nin;
        add(b);
        push(b);
        const uint32_t m = mc.v[nin - 1];
        uint32_t ge = 0u;
        if (m < 16u) {
            ge = 0xffffu;
#pragma unroll
            for (int i = 0; i < 4; ++i) ge = ((m >> i) & 1u) ? (c[i] & ge) : (c[i] | ge);
        }
        const size_t slot = (size_t)((f0 + t) % ring_cap);
        ring16[slot * plane_words * 2] = (uint16_t)b;
        vote16[(size_t)t * plane_words * 2] = (uint16_t)ge;
    }
    if (t1 == T && gray_state_out) store16(gray_state_out + px_off, pg);
}

// ------------------------------------------------------------------------------------------------
// EMA (addWeighted).  cv2 computes, in float32: t = dilated * beta (rounded), s = fma(acc, alpha, t),
// result = saturate(round-half-even(s)).  One thread owns 16 pixels, keeps their accumulator bytes in
// registers over the whole batch.
// ------------------------------------------------------------------------------------------------
template <bool ALIGNED, int PX = 16>                     // PX pixels per thread: 16, or 8 (twice the threads: the walk over the batch is
#ifndef DVC_EMA_MINB
#define DVC_EMA_MINB 4
#endif
__global__ void __launch_bounds__(256, PX == 8 ? DVC_EMA_MINB : 1)   // a chain of dependent table look-ups, more resident warps hide it better)
k_ema(uint8_t* __restrict__ acc, const uint32_t* __restrict__ dilated, uint32_t* __restrict__ over127,
      uint32_t* __restrict__ nonzero, uint8_t* __restrict__ acc_all, int T, int H, int W, int wpr, float alpha,
      float beta) {
    static_assert(PX == 16 || PX == 8, "k_ema: 8 or 16 pixels per thread");
    constexpr int NQ = PX / 4;
    __shared__ uint8_t s_lut[512];                           // [dilated bit][acc] -> acc'
    {
        const float on = __fmul_rn(255.0f, beta);
        for (int i = threadIdx.x; i < 512; i += blockDim.x) {
            const float sv = __fmaf_rn((float)(i & 255), alpha, (i >> 8) ? on : 0.0f);
            s_lut[i] = (uint8_t)max(0, min(255, __float2int_rn(sv)));
        }
    }
    __syncthreads();
    const int gpr = (W + PX - 1) / PX;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)gpr * H) return;
    const int y = (int)(gid / gpr), gx = (int)(gid % gpr), x0 = gx * PX;
    const size_t plane_words = (size_t)H * wpr, plane_bytes = (size_t)H * W;
    const int npx = min(PX, W - x0);
    {   // blockIdx.y = stream of a lock-step group: one accumulator plane per stream, T planes of everything else
        const size_t s = blockIdx.y;
        acc += s * plane_bytes;
        dilated += s * T * plane_words; over127 += s * T * plane_words; nonzero += s * T * plane_words;
        if (acc_all) acc_all += s * T * plane_bytes;
    }
    uint32_t a[NQ];
    uint8_t* arow = acc + (size_t)y * W;
    if (ALIGNED) {
        if (PX == 16) { uint4 t = *reinterpret_cast<const uint4*>(arow + x0); a[0] = t.x; a[1] = t.y; a[NQ - 2] = t.z; a[NQ - 1] = t.w; }
        else { uint2 t = *reinterpret_cast<const uint2*>(arow + x0); a[0] = t.x; a[1] = t.y; }
    } else { for (int i = 0; i < NQ; ++i) a[i] = 0; for (int i = 0; i < npx; ++i) a[i >> 2] |= (uint32_t)arow[x0 + i] << ((i & 3) * 8); }
    // accumulator update as a table: acc' depends only on (acc, dilated bit), so the float expression of cv2.addWeighted
    // is evaluated once per CTA for the 2 x 256 cases (no int <-> float conversions, which run on the quarter-rate XU
    // pipe, in the per-frame loop)
    auto piece = [&](int t) -> uint32_t {
        const size_t wo = (size_t)t * plane_words + (size_t)y * wpr;
        return PX == 16 ? (uint32_t)reinterpret_cast<const uint16_t*>(dilated + wo)[gx] : (uint32_t)reinterpret_cast<const uint8_t*>(dilated + wo)[gx];
    };
    auto step = [&](int t, uint32_t bits) {
        const size_t woff = (size_t)t * plane_words + (size_t)y * wpr;
        uint32_t hi = 0, nz = 0, any = bits;
#pragma unroll
        for (int q = 0; q < NQ; ++q) any |= a[q];
        if (any != 0u) {
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                uint32_t nw = 0;
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    const int i = q * 4 + p;
                    const uint32_t v = s_lut[(((bits >> i) & 1u) << 8) | ((a[q] >> (8 * p)) & 0xffu)];
                    nw |= v << (8 * p);
                }
                a[q] = nw;
                hi |= ((((nw >> 7) & 0x01010101u) * 0x00204081u >> 21) & 0xfu) << (4 * q);                                   // byte > 127
                nz |= (((((nw | ((nw & 0x7f7f7f7fu) + 0x7f7f7f7fu)) & 0x80808080u) >> 7) * 0x00204081u >> 21) & 0xfu) << (4 * q);  // byte != 0
            }
            if (npx < PX) { const uint32_t m = (1u << npx) - 1u; hi &= m; nz &= m; }
        }
        if (PX == 16) {
            reinterpret_cast<uint16_t*>(over127 + woff)[gx] = (uint16_t)hi;
            reinterpret_cast<uint16_t*>(nonzero + woff)[gx] = (uint16_t)nz;
        } else {
            reinterpret_cast<uint8_t*>(over127 + woff)[gx] = (uint8_t)hi;
            reinterpret_cast<uint8_t*>(nonzero + woff)[gx] = (uint8_t)nz;
        }
        if (acc_all) {
            uint8_t* o = acc_all + (size_t)t * plane_bytes + (size_t)y * W;
            if (ALIGNED) {
                if (PX == 16) *reinterpret_cast<uint4*>(o + x0) = make_uint4(a[0], a[1], a[NQ - 2], a[NQ - 1]);
                else *reinterpret_cast<uint2*>(o + x0) = make_uint2(a[0], a[1]);
            } else for (int i = 0; i < npx; ++i) o[x0 + i] = (uint8_t)(a[i >> 2] >> ((i & 3) * 8));
        }
    };
    // the walk over the frames is a chain of dependent look-ups; the mask pieces it consumes are not: PF of them are loaded ahead
    constexpr int PF = PX == 8 ? 8 : 1;                      // (4: no gain; 16, or 8 under a 48-register cap: slightly slower)
    int t = 0;
    for (; t + PF <= T; t += PF) {
        uint32_t pf[PF];
#pragma unroll
        for (int j = 0; j < PF; ++j) pf[j] = piece(t + j);
#pragma unroll
        for (int j = 0; j < PF; ++j) step(t + j, pf[j]);
    }
    for (; t < T; ++t) step(t, piece(t));
    if (ALIGNED) {
        if (PX == 16) *reinterpret_cast<uint4*>(arow + x0) = make_uint4(a[0], a[1], a[NQ - 2], a[NQ - 1]);
        else *reinterpret_cast<uint2*>(arow + x0) = make_uint2(a[0], a[1]);
    } else for (int i = 0; i < npx; ++i) arow[x0 + i] = (uint8_t)(a[i >> 2] >> ((i & 3) * 8));
}

// ------------------------------------------------------------------------------------------------
// morphology chain
// ------------------------------------------------------------------------------------------------
constexpr int MORPH_MAX_K = 33;        // kernel extent limit (one neighbour word each side)
constexpr int MORPH_MAX_PRIMS = 6;

struct MorphPrim {
    int8_t erode;                      // 0 = dilate (OR), 1 = erode (AND; run as NOT dilate NOT)
    int8_t separable;                  // all rows share one run and rows are contiguous
    int8_t nrows;                      // rows of the structuring element that are non-empty
    int8_t small;                      // fits in 3x3 around the anchor: small_rows[] holds per-row flags
    int16_t kind;                      // 0 = runtime paths; 1xx = rect_pass<xx>; 1, 2 = small_pass specialisations; 3 = MORPH_ELLIPSE 2x2 twice
    int8_t small_rows[3];              // dy = -1, 0, +1: bit0 present, bit1 dx=-1 present, bit2 dx=+1 present
    int8_t dy[MORPH_MAX_K];            // row offset (kernel row - anchor)
    int8_t lo[MORPH_MAX_K];            // run of column offsets [lo, hi] in that row
    int8_t hi[MORPH_MAX_K];
};
struct MorphChain {
    int n;
    int pad;                           // zero rows kept above / below the staged planes: the largest reach of a rect_pass<K> primitive
    int halo_top, halo_bot;            // rows of input needed above / below an output band
    MorphPrim p[MORPH_MAX_PRIMS];
};

// OR over column offsets [-L, R] of one bit row: out(x) = OR_d in(x + d).  Pixels to the right are higher
// bits: the right reach works on (next:cur), the left reach on (cur:prev), each log-doubled on a 64-bit
// value with a shift schedule precomputed on the host (MorphPrim::rsh / lsh).
struct HRun { int nr, nl; };      // window sizes: nr = hi + 1 (right reach + centre), nl = 1 - lo

DEVI HRun make_hrun(int lo, int hi) { HRun h; h.nr = hi + 1; h.nl = 1 - lo; return h; }

DEVI uint32_t hrun_or(uint32_t prev, uint32_t cur, uint32_t next, const HRun& h) {
    uint32_t res = cur;
    if (h.nr > 1) {
        uint64_t a = ((uint64_t)next << 32) | cur;
        const int n = h.nr;
        int c = 1;
        if (n >= 2) { a |= a >> 1; c = 2; }
        if (n >= 4) { a |= a >> 2; c = 4; }
        if (n >= 8) { a |= a >> 4; c = 8; }
        if (n >= 16) { a |= a >> 8; c = 16; }
        if (n >= 32) { a |= a >> 16; c = 32; }
        if (n > c) a |= a >> (n - c);
        res |= (uint32_t)a;
    }
    if (h.nl > 1) {
        uint64_t b = ((uint64_t)cur << 32) | prev;
        const int n = h.nl;
        int c = 1;
        if (n >= 2) { b |= b << 1; c = 2; }
        if (n >= 4) { b |= b << 2; c = 4; }
        if (n >= 8) { b |= b << 4; c = 8; }
        if (n >= 16) { b |= b << 8; c = 16; }
        if (n >= 32) { b |= b << 16; c = 32; }
        if (n > c) b |= b << (n - c);
        res |= (uint32_t)(b >> 32);
    }
    return res;
}

DEVI uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Shared per-thread view of the staged band used by the primitive passes.
struct BandCtx {
    int wpr, j, jp, jn, ra, rb, r_lo, r_hi;
    uint32_t vm, pm, nm;
};

// OR over a compile-time window: NR = right reach + 1 (bits x .. x+NR-1), NL = left reach + 1
template <int NR, int NL>
DEVI uint32_t hrun_or_c(uint32_t prev, uint32_t cur, uint32_t next) {
    uint32_t res = cur;
    if (NR > 1) {
        uint64_t a = ((uint64_t)next << 32) | cur;
        int c = 1;
#pragma unroll
        for (int s = 1; s <= 16; s *= 2) if (NR >= 2 * s) { a |= a >> s; c = 2 * s; }
        if (NR > c) a |= a >> (NR - c);
        res |= (uint32_t)a;
    }
    if (NL > 1) {
        uint64_t b = ((uint64_t)cur << 32) | prev;
        int c = 1;
#pragma unroll
        for (int s = 1; s <= 16; s *= 2) if (NL >= 2 * s) { b |= b << s; c = 2 * s; }
        if (NL > c) b |= b << (NL - c);
        res |= (uint32_t)(b >> 32);
    }
    return res;
}

// OR over the symmetric bit window [i - R, i + R] (K = 2R + 1 <= 33) of word x with neighbours p (lower bits) and n: the
// 64-bit window T = (n:x:p) >> (32 - R) puts global bit i - R at bit i, then a one-sided log-doubling OR of width K leaves
// the answer in the low word (the high word only ever needs its low K - 1 bits).
template <int K>
DEVI uint32_t hwin_or(uint32_t p, uint32_t x, uint32_t n) {
    constexpr int R = K / 2;
    uint32_t lo = __funnelshift_r(p, x, 32 - R), hi = __funnelshift_r(x, n, 32 - R);
    int c = 1;
#pragma unroll
    for (int s = 1; 2 * s <= K; s *= 2) { lo |= __funnelshift_r(lo, hi, s); hi |= hi >> s; c = 2 * s; }
    if (K > c) lo |= __funnelshift_r(lo, hi, K - c);
    return lo;
}

// MorphChain::pad rows of padding above and below each staged plane (zero = "ignored" in the dilation domain) let the
// vertical passes read beyond the band without range checks.

// k x k rectangle, k odd (anchor in the middle): horizontal pass A -> B, vertical pass B -> A.
// B holds dilation-domain values; its rows outside the image (and the padding) stay zero for the whole kernel, so the
// vertical pass needs no range checks.
template <int K>
DEVI void rect_pass(uint32_t* A, uint32_t* B, const BandCtx& c, uint32_t flip) {
    constexpr int R = K / 2;
    const int n = c.rb - c.ra, wpr = c.wpr;
    {
        const uint32_t* row = A + c.ra * wpr;
        uint32_t* out = B + c.ra * wpr + c.j;
        for (int i = 0; i < n; ++i, row += wpr, out += wpr) {
            const uint32_t p = (row[c.jp] ^ flip) & c.pm, x = (row[c.j] ^ flip) & c.vm, nx = (row[c.jn] ^ flip) & c.nm;
            *out = hwin_or<K>(p, x, nx) & c.vm;
        }
    }
    __syncthreads();
    // vertical: van Herk / Gil-Werman on the thread's run of rows.  Rows are cut into blocks of K starting at ra - R; the
    // window of output ra + m K + u is the suffix of block m from offset u OR the prefix of block m + 1 up to offset u - 1.
    // Per output: one shared-memory load, one OR into the running prefix, one OR for the suffix scan, one OR to combine --
    // independent of K.
    if (n > 0) {
        const uint32_t* q = B + (c.ra - R) * wpr + c.j;         // next row to load
        uint32_t* o = A + c.ra * wpr + c.j;                     // next output row
        uint32_t sfx[K];                                        // suffix ORs of the current block (the only per-row state kept)
#pragma unroll
        for (int d = 0; d < K; ++d, q += wpr) sfx[d] = *q;
#pragma unroll
        for (int d = K - 2; d >= 0; --d) sfx[d] |= sfx[d + 1];
        for (int left = n; left > 0; left -= K) {
            uint32_t pfx = 0u;
            *o = (sfx[0] ^ flip) & c.vm;
            o += wpr;
            const uint32_t* qb = q;                             // first row of the next block
#pragma unroll
            for (int u = 1; u < K; ++u, q += wpr, o += wpr) {
                if (u < left) {
                    pfx |= *q;
                    *o = ((sfx[u] | pfx) ^ flip) & c.vm;
                }
            }
            if (left > K) {                                     // suffix scan of the next block: its rows are read once more
                sfx[K - 1] = *q;
                q += wpr;
#pragma unroll
                for (int d = K - 2; d >= 0; --d) sfx[d] = qb[d * wpr] | sfx[d + 1];
            }
        }
    }
    __syncthreads();
}

// 3x3-bounded element with compile-time row flags (bit0 centre, bit1 dx=-1, bit2 dx=+1): A -> B.
// out[r] = V_up(r-1) | V_mid(r) | V_dn(r+1); every input row streams once through registers.
template <int FU, int FM, int FD>
DEVI void small_pass(const uint32_t* A, uint32_t* B, const BandCtx& c, uint32_t flip) {
    constexpr bool NEED_L = ((FU | FM | FD) & 2) != 0, NEED_R = ((FU | FM | FD) & 4) != 0;
    uint32_t pend = 0, up_prev = 0;            // pend = V_up(x-2) | V_mid(x-1);  up_prev = V_up(x-1)
    const uint32_t* row = A + (c.ra - 1) * c.wpr;
    uint32_t* out = B + (c.ra - 1) * c.wpr + c.j;
    if (c.ra < c.rb)
        for (int x = c.ra - 1; x <= c.rb; ++x, row += c.wpr, out += c.wpr) {
            uint32_t v_up = 0, v_mid = 0, v_dn = 0;
            if (x >= c.r_lo && x < c.r_hi) {
                const uint32_t m = (row[c.j] ^ flip) & c.vm;
                const uint32_t cl = NEED_L ? __funnelshift_l((row[c.jp] ^ flip) & c.pm, m, 1) : 0u;
                const uint32_t cr = NEED_R ? __funnelshift_r(m, (row[c.jn] ^ flip) & c.nm, 1) : 0u;
                v_up = ((FU & 1) ? m : 0u) | ((FU & 2) ? cl : 0u) | ((FU & 4) ? cr : 0u);
                v_mid = ((FM & 1) ? m : 0u) | ((FM & 2) ? cl : 0u) | ((FM & 4) ? cr : 0u);
                v_dn = ((FD & 1) ? m : 0u) | ((FD & 2) ? cl : 0u) | ((FD & 4) ? cr : 0u);
            }
            if (x > c.ra) out[-c.wpr] = ((pend | v_dn) ^ flip) & c.vm;        // row x-1 in [ra, rb)
            pend = up_prev | v_mid;
            up_prev = v_up;
        }
    __syncthreads();
}

// MORPH_ELLIPSE (2, 2) = {(0,0), (-1,0), (0,-1)} applied twice with the same polarity (the two erosions in the middle of CLOSE, OPEN:
// the reference's mask clean-up, motion_compression_opt.py:89-90) is one pass with the Minkowski sum
// {(0,0), (-1,0), (-2,0), (0,-1), (-1,-1), (0,-2)}: out[r] = t[r] | l2[r] | t[r-1] | m[r-2] with t = m | l1, lk = the row shifted by k
// pixels.  Exact with cv2's ignored borders for the same reason as merged rectangles: all offsets point the same way, so the
// intermediate pixel of a two-step path lies between its end points.  A -> B, rows stream through registers once.
DEVI void ellipse2x2_pass(const uint32_t* A, uint32_t* B, const BandCtx& c, uint32_t flip) {
    uint32_t t1 = 0, m1 = 0, m2 = 0;            // t[x-1], m[x-1], m[x-2]
    const uint32_t* row = A + (c.ra - 2) * c.wpr;
    uint32_t* out = B + (c.ra - 2) * c.wpr + c.j;
    if (c.ra < c.rb)
        for (int x = c.ra - 2; x < c.rb; ++x, row += c.wpr, out += c.wpr) {
            uint32_t m = 0, l1 = 0, l2 = 0;
            if (x >= c.r_lo && x < c.r_hi) {
                m = (row[c.j] ^ flip) & c.vm;
                const uint32_t p = (row[c.jp] ^ flip) & c.pm;
                l1 = __funnelshift_l(p, m, 1);
                l2 = __funnelshift_l(p, m, 2);
            }
            const uint32_t t = m | l1;
            if (x >= c.ra) *out = ((t | l2 | t1 | m2) ^ flip) & c.vm;
            m2 = m1; m1 = m; t1 = t;
        }
    __syncthreads();
}

// grid: (bands, n_images); dynamic smem: 2 planes of ext_rows x wpr words + one mbarrier.
// Thread (g, j) owns word column j of a contiguous run of rows (row group g), so consecutive outputs of a
// thread reuse the rows it has just read (3x3-bounded elements stream each input row through registers
// once) and addressing is a pointer increment.
// Erosion runs as NOT dilate NOT: the complement is folded into the first read and the last write of the
// primitive.  Rows outside the image and bits beyond W are 'ignored' pixels: they read as 0 in the dilation
// domain of either polarity, so only rows [r_lo, r_hi) of the staged band are ever touched.
template <int MAXT>      // 256: several CTAs per SM (small halos); 1024: one CTA owns the SM's shared memory (large halos)
__global__ void __launch_bounds__(MAXT, MAXT == 256 ? 4 : 1)
k_morph_chain(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, int H, int W, int wpr, int band_rows,
              MorphChain ch) {
    extern __shared__ __align__(128) uint32_t smem[];
    const int ext_rows = band_rows + ch.halo_top + ch.halo_bot;
    const size_t plane = (size_t)(ext_rows + 2 * ch.pad) * wpr;          // words per staged plane, padding included
    uint32_t* A = smem + (size_t)ch.pad * wpr;                           // row 0 of the band
    uint32_t* B = A + plane;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + 2 * plane);
    const int y0 = blockIdx.x * band_rows;                    // first output row of this band
    const int ey0 = y0 - ch.halo_top;                         // image row of ext row 0
    const size_t plane_words = (size_t)H * wpr;
    const uint32_t* sp = src + (size_t)blockIdx.y * plane_words;
    uint32_t* dp = dst + (size_t)blockIdx.y * plane_words;
    const int tid = threadIdx.x, nt = blockDim.x;
    const int r_lo = max(0, -ey0), r_hi = min(ext_rows, H - ey0);     // ext rows that exist in the image

    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {       // stage rows [r_lo, r_hi): contiguous in the plane, one bulk (TMA) copy
        const uint32_t bytes = (uint32_t)(r_hi - r_lo) * wpr * 4u;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(A + (size_t)r_lo * wpr)), "l"(sp + (size_t)(ey0 + r_lo) * wpr), "r"(bytes),
                       "r"(smem_u32(bar)) : "memory");
    }
    // rows of either plane that no pass ever writes -- the padding and the band rows outside the image -- are zeroed once
    // (they are disjoint from the rows the bulk copy fills, so this overlaps the copy)
    {
        const int top = (ch.pad + r_lo) * wpr, bot0 = (ch.pad + r_hi) * wpr, total = (int)plane;
        for (int pl = 0; pl < 2; ++pl) {
            uint32_t* base = smem + pl * plane;
            for (int i = tid; i < top; i += nt) base[i] = 0u;
            for (int i = bot0 + tid; i < total; i += nt) base[i] = 0u;
        }
    }
    // thread -> (row group, word column)
    const int groups = nt / wpr;                              // >= 1 (host guarantees wpr <= blockDim)
    const int j = tid % wpr, g = tid / wpr;
    const int rows_img = r_hi - r_lo, chunk = (rows_img + groups - 1) / groups;
    const int ra = r_lo + g * chunk, rb = g < groups ? min(r_hi, ra + chunk) : ra;   // owned rows [ra, rb)
    const uint32_t vm = valid_mask(j, W);
    const uint32_t pm = j > 0 ? valid_mask(j - 1, W) : 0u, nm = j + 1 < wpr ? valid_mask(j + 1, W) : 0u;
    const int jp = j > 0 ? j - 1 : j, jn = j + 1 < wpr ? j + 1 : j;      // clamped neighbour columns (masked by pm / nm)
    if (tid == 0) {       // one waiter; everybody else parks at the barrier below instead of spinning
        uint32_t done = 0;
        while (!done) {
            asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n selp.u32 %0, 1, 0, p;\n}"
                         : "=r"(done) : "r"(smem_u32(bar)) : "memory");
        }
    }
    __syncthreads();

    BandCtx cx;
    cx.wpr = wpr; cx.j = j; cx.jp = jp; cx.jn = jn; cx.ra = ra; cx.rb = rb; cx.r_lo = r_lo; cx.r_hi = r_hi;
    cx.vm = vm; cx.pm = pm; cx.nm = nm;

    for (int pi = 0; pi < ch.n; ++pi) {
        const MorphPrim& P = ch.p[pi];
        const uint32_t flip = P.erode ? 0xffffffffu : 0u;
        // compile-time specialisations of the common elements
        if (P.kind != 0) {
            bool swap = true;
            switch (P.kind) {
                case 103: rect_pass<3>(A, B, cx, flip); swap = false; break;
                case 105: rect_pass<5>(A, B, cx, flip); swap = false; break;
                case 107: rect_pass<7>(A, B, cx, flip); swap = false; break;
                case 109: rect_pass<9>(A, B, cx, flip); swap = false; break;
                case 111: rect_pass<11>(A, B, cx, flip); swap = false; break;
                case 113: rect_pass<13>(A, B, cx, flip); swap = false; break;
                case 115: rect_pass<15>(A, B, cx, flip); swap = false; break;
                case 117: rect_pass<17>(A, B, cx, flip); swap = false; break;
                case 119: rect_pass<19>(A, B, cx, flip); swap = false; break;
                case 121: rect_pass<21>(A, B, cx, flip); swap = false; break;
                case 123: rect_pass<23>(A, B, cx, flip); swap = false; break;
                case 125: rect_pass<25>(A, B, cx, flip); swap = false; break;
                case 127: rect_pass<27>(A, B, cx, flip); swap = false; break;
                case 129: rect_pass<29>(A, B, cx, flip); swap = false; break;
                case 131: rect_pass<31>(A, B, cx, flip); swap = false; break;
                case 133: rect_pass<33>(A, B, cx, flip); swap = false; break;
                case 1: small_pass<1, 3, 0>(A, B, cx, flip); break;     // MORPH_ELLIPSE 2x2
                case 2: small_pass<1, 7, 1>(A, B, cx, flip); break;     // MORPH_ELLIPSE 3x3 (a cross)
                case 3: ellipse2x2_pass(A, B, cx, flip); break;         // MORPH_ELLIPSE 2x2, twice
                default: break;
            }
            if (swap) { uint32_t* t = A; A = B; B = t; }
            continue;
        }
        if (P.separable) {
            const HRun hr = make_hrun(P.lo[0], P.hi[0]);
            {                                                                   // horizontal: A -> B
                const uint32_t* row = A + ra * wpr;
                uint32_t* out = B + ra * wpr + j;
                for (int r = ra; r < rb; ++r, row += wpr, out += wpr) {
                    const uint32_t p = (row[jp] ^ flip) & pm, c = (row[j] ^ flip) & vm, n = (row[jn] ^ flip) & nm;
                    *out = (p | c | n) ? hrun_or(p, c, n, hr) & vm : 0u;
                }
            }
            __syncthreads();
            const int dy0 = P.dy[0], dy1 = P.dy[P.nrows - 1];
            for (int r = ra; r < rb; ++r) {                                     // vertical: B -> A
                const int a0 = max(r + dy0, r_lo), a1 = min(r + dy1, r_hi - 1);
                const uint32_t* q = B + a0 * wpr + j;
                uint32_t acc = 0;
#pragma unroll 4
                for (int rr = a0; rr <= a1; ++rr, q += wpr) acc |= *q;
                A[r * wpr + j] = (acc ^ flip) & vm;
            }
            __syncthreads();
        } else if (P.small) {
            // 3x3-bounded element (e.g. MORPH_ELLIPSE 2 or 3).  Row flags: bit0 centre, bit1 dx=-1, bit2 dx=+1.
            // out[r] = V_up(r-1) | V_mid(r) | V_dn(r+1); input rows stream once through registers.
            const int f_up = P.small_rows[0], f_mid = P.small_rows[1], f_dn = P.small_rows[2];
            const bool need_l = ((f_up | f_mid | f_dn) & 2) != 0, need_r = ((f_up | f_mid | f_dn) & 4) != 0;
            uint32_t pend = 0, up_prev = 0;            // pend = V_up(x-2) | V_mid(x-1);  up_prev = V_up(x-1)
            const uint32_t* row = A + (ra - 1) * wpr;
            uint32_t* out = B + (ra - 1) * wpr + j;    // out[x-1] is written at step x, so this trails by one row
            if (ra < rb)
                for (int x = ra - 1; x <= rb; ++x, row += wpr, out += wpr) {
                    uint32_t v_up = 0, v_mid = 0, v_dn = 0;
                    if (x >= r_lo && x < r_hi) {
                        const uint32_t c = (row[j] ^ flip) & vm;
                        const uint32_t cl = need_l ? __funnelshift_l((row[jp] ^ flip) & pm, c, 1) : 0u;
                        const uint32_t cr = need_r ? __funnelshift_r(c, (row[jn] ^ flip) & nm, 1) : 0u;
                        v_up = ((f_up & 1) ? c : 0u) | ((f_up & 2) ? cl : 0u) | ((f_up & 4) ? cr : 0u);
                        v_mid = ((f_mid & 1) ? c : 0u) | ((f_mid & 2) ? cl : 0u) | ((f_mid & 4) ? cr : 0u);
                        v_dn = ((f_dn & 1) ? c : 0u) | ((f_dn & 2) ? cl : 0u) | ((f_dn & 4) ? cr : 0u);
                    }
                    if (x > ra) out[-wpr] = ((pend | v_dn) ^ flip) & vm;       // row x-1 in [ra, rb)
                    pend = up_prev | v_mid;
                    up_prev = v_up;
                }
            __syncthreads();
            uint32_t* t = A; A = B; B = t;
        } else {
            const int nrows = P.nrows;
            for (int r = ra; r < rb; ++r) {                                     // generic: A -> B
                uint32_t acc = 0;
                for (int k = 0; k < nrows; ++k) {
                    const int rr = r + P.dy[k];
                    if (rr < r_lo || rr >= r_hi) continue;
                    const uint32_t* row = A + rr * wpr;
                    const uint32_t p = (row[jp] ^ flip) & pm, c = (row[j] ^ flip) & vm, n = (row[jn] ^ flip) & nm;
                    if (p | c | n) acc |= hrun_or(p, c, n, make_hrun(P.lo[k], P.hi[k]));
                }
                B[r * wpr + j] = (acc ^ flip) & vm;
            }
            __syncthreads();
            uint32_t* t = A; A = B; B = t;
        }
    }
    // write the band
    const int out_rows = min(band_rows, H - y0);
    for (int i = tid; i < out_rows * wpr; i += nt) dp[(size_t)y0 * wpr + i] = A[ch.halo_top * wpr + i];
}

// ------------------------------------------------------------------------------------------------
// structuring elements larger than MORPH_MAX_K: one primitive at a time, between global bit-planes
// ------------------------------------------------------------------------------------------------
// Horizontal runs of any length come from a doubling table: level p holds F_p(x) = OR of the dilation-domain bits
// [x, x + 2^p), and a run [x + lo, x + hi] of length L, 2^p <= L < 2^(p+1), is F_p(x + lo) | F_p(x + hi + 1 - 2^p): two
// funnel-shifted reads per output word whatever L is.  Runs are clipped to the frame on the host (|lo|, |hi| <= W - 1), so a
// level row needs wpr words of zeros on the left and wpr + 1 on the right: MLARGE_RS(wpr) words, image word 0 at offset wpr.
// Bits outside the image are 0 in the dilation domain, so erosion is NOT dilate NOT with cv2's ignored borders, as in
// k_morph_chain.
//   rect      rows of one run: the horizontal run at level p, then van Herk / Gil-Werman down the columns (k_mlarge_vscan
//             + k_mlarge_vcombine), whose cost does not depend on k
//   ellipse   not separable: out(y) = OR over the element rows dy of the run of row y + dy, one k_mlarge_rows launch per level
//             with the rows of that level
__host__ __device__ inline int mlarge_rs(int wpr) { return 3 * wpr + 1; }
struct LargeRow { int dy, lo, hi, pad; };   // one element row clipped to the frame: run [lo, hi] of row y + dy

// level 0: the input in the dilation domain, zeros in the padding.  grid: (words of H padded rows, planes)
__global__ void __launch_bounds__(256)
k_mlarge_level0(const uint32_t* __restrict__ src, uint32_t* __restrict__ F, int H, int W, int wpr, uint32_t flip) {
    const int rs = mlarge_rs(wpr);
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)H * rs) return;
    const int y = (int)(i / rs), w = (int)(i % rs) - wpr;
    uint32_t v = 0u;
    if (w >= 0 && w < wpr) v = (src[((size_t)blockIdx.y * H + y) * wpr + w] ^ flip) & valid_mask(w, W);
    F[(size_t)blockIdx.y * H * rs + i] = v;
}

// level q from level q - 1: F_q(x) = F_{q-1}(x) | F_{q-1}(x + s), s = 2^(q-1); words beyond the padding read as zero
__global__ void __launch_bounds__(256)
k_mlarge_double(const uint32_t* __restrict__ Fi, uint32_t* __restrict__ Fo, int H, int wpr, int s) {
    const int rs = mlarge_rs(wpr);
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)H * rs) return;
    const int c = (int)(i % rs), c0 = c + (s >> 5);
    const size_t base = (size_t)blockIdx.y * H * rs + i - c;
    const uint32_t a = c0 < rs ? Fi[base + c0] : 0u, b = c0 + 1 < rs ? Fi[base + c0 + 1] : 0u;
    Fo[base + c] = Fi[base + c] | __funnelshift_r(a, b, s & 31);
}

// out(y) |= OR over table rows [beg, end) (all at level p) of the run [x + lo, x + hi] of level row y + dy.  `first` starts
// from zero instead of the dilation-domain value already in dst; the result is stored as (acc ^ xor_out) & valid, so the
// last launch of a primitive passes its flip and the others 0.  grid: (words of H rows, planes)
__global__ void __launch_bounds__(256)
k_mlarge_rows(const uint32_t* __restrict__ F, uint32_t* __restrict__ dst, int H, int W, int wpr,
              const LargeRow* __restrict__ rows, int beg, int end, int p, int first, uint32_t xor_out) {
    const int rs = mlarge_rs(wpr);
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)H * wpr) return;
    const int y = (int)(i / wpr), j = (int)(i % wpr), x0 = j * 32, tail = 1 - (1 << p);
    const size_t o = (size_t)blockIdx.y * H * wpr + i;
    const uint32_t* Fp = F + (size_t)blockIdx.y * H * rs + wpr;
    uint32_t acc = first ? 0u : dst[o];
    for (int r = beg; r < end; ++r) {
        const LargeRow e = rows[r];
        const int yy = y + e.dy;
        if (yy < 0 || yy >= H) continue;
        const uint32_t* row = Fp + (size_t)yy * rs;
        const int pa = x0 + e.lo, pb = x0 + e.hi + tail;           // >= -(W - 1) and < 2 W: inside the padded row
        const int wa = pa >> 5, wb = pb >> 5;
        acc |= __funnelshift_r(row[wa], row[wa + 1], pa & 31) | __funnelshift_r(row[wb], row[wb + 1], pb & 31);
    }
    dst[o] = (acc ^ xor_out) & valid_mask(j, W);
}

// van Herk / Gil-Werman down the columns, blocks of B rows from row 0: g(y) = OR of rows [block start, y], h(y) = OR of rows
// [y, block end] (clipped to H).  One thread per (word column, block).  grid: (word columns x blocks, planes)
__global__ void __launch_bounds__(256)
k_mlarge_vscan(const uint32_t* __restrict__ in, uint32_t* __restrict__ g, uint32_t* __restrict__ h, int H, int wpr, int B) {
    const int nb = (H + B - 1) / B;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nb * wpr) return;
    const int j = i % wpr, y0 = (i / wpr) * B, y1 = min(H, y0 + B);
    const size_t off = (size_t)blockIdx.y * H * wpr + j;
    in += off; g += off; h += off;
    uint32_t a = 0u;
    for (int y = y0; y < y1; ++y) { a |= in[(size_t)y * wpr]; g[(size_t)y * wpr] = a; }
    a = 0u;
    for (int y = y1 - 1; y >= y0; --y) { a |= in[(size_t)y * wpr]; h[(size_t)y * wpr] = a; }
}

// out(y) = OR of rows [y + dy0, y + dy0 + B - 1] = h(s) | g(e), s = y + dy0 <= y, e = s + B - 1 >= y.  Rows outside the image
// are zero: h(s < 0) is the suffix of an all-outside block; g(e >= H) is g(H - 1) when row H - 1 is in e's block, else zero.
__global__ void __launch_bounds__(256)
k_mlarge_vcombine(const uint32_t* __restrict__ g, const uint32_t* __restrict__ h, uint32_t* __restrict__ dst, int H, int W,
                  int wpr, int B, int dy0, uint32_t flip) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)H * wpr) return;
    const int y = (int)(i / wpr), j = (int)(i % wpr);
    const size_t pl = (size_t)blockIdx.y * H * wpr;
    const int s = y + dy0, e = s + B - 1;
    uint32_t v = 0u;
    if (s >= 0) v |= h[pl + (size_t)s * wpr + j];
    if (e < H) v |= g[pl + (size_t)e * wpr + j];
    else if ((e / B) * B <= H - 1) v |= g[pl + (size_t)(H - 1) * wpr + j];
    dst[pl + i] = (v ^ flip) & valid_mask(j, W);
}

}  // namespace dvc
