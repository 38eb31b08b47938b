// K4 for block_size 4 (frame_differencing.py:110-111,115-130; arithmetic contract in k_degrade.cuh) and the 8x8 kernel.
// The arithmetic is built around what profiles/r1f measured on the first, scalar K4: it was issue-bound (70 % issue-slot
// utilisation, 860 warp instructions per 4x4 block), not HBM-bound.
//
//  * Blackwell's packed fp32 pipe (FADD2 / FMUL2 / FFMA2, PTX add/mul/fma.rn.f32x2) processes two IEEE
//    binary32 lanes per instruction with the same per-lane rounding as the scalar instructions.  A thread
//    owns two adjacent 4x4 blocks, so block A rides in the low lane and block B in the high lane of every
//    DCT / quantiser instruction: half the floating-point issue slots, bit-identical results.
//  * round(d / q): the IEEE quotient fl(d / q) is formed without a division by one Markstein correction step,
//        y0 = fl(d * r),  e = fma(-q, y0, d) (exact),  y = fma(e, r, y0),   r = fl(1 / q) (host, correctly rounded)
//    which is the correctly rounded quotient (Markstein 1990, Thm. 8; re-checked for this value range against the
//    hardware division on 3e9 samples, tests/test_oracle_vs_cv2.py::test_markstein_quotient for a sample).  Then
//    rint() is the usual magic-number add/sub.  No tie detection, no slow path, no second evaluation: the
//    quantiser is six packed instructions per coefficient pair.  The host takes this path for q in [0.01, 1e6],
//    where the step is exact and |d / q| < 2^22 keeps the magic-number rounding valid; other levels go to
//    k_degrade_generic.
//  * luma: Y << 14 = 1868 B + 9617 G + 4899 R + 8192 as two IDP.2A (u16 x u8 pairs) per pixel instead of
//    three-to-four IDP.4A + shift-add, and (s >> 14) | 0x4B000000 (the 2^23 + Y float pattern) is one funnel
//    shift.
#pragma once
#include "k_degrade.cuh"

namespace dvc {

struct QuantP {
    float rcp[3];    // fl(1 / (q * 2^NE)),  NE = number of even indices among (row, col) = pending scale 2^-NE
    float nqs[3];    // -(q * 2^NE)
    float o[3];      // q * 2^-NE: output scale with the inverse butterflies' x0.5 pre-applied
};

// forward / inverse 4-point DCT without the x0.5 of outputs 0 and 2 / inputs 0 and 2: those power-of-two scalings are
// folded into QuantP
template <typename T>
DEVI void dct4_fwd_t(T& x0, T& x1, T& x2, T& x3) {
    const T c1 = splat<T>(DVC_C1), c3 = splat<T>(DVC_C3), nc1 = splat<T>(-DVC_C1);
    const T s0 = add(x0, x3), s1 = add(x1, x2), d0 = sub(x0, x3), d1 = sub(x1, x2);
    x0 = add(s0, s1);
    x2 = sub(s0, s1);
    x1 = fma_(c3, d1, mul(c1, d0));
    x3 = fma_(c3, d0, mul(nc1, d1));          // -(c1 * d1) == (-c1) * d1 exactly
}
template <typename T>
DEVI void dct4_inv_t(T& x0, T& x1, T& x2, T& x3) {
    const T c1 = splat<T>(DVC_C1), c3 = splat<T>(DVC_C3), nc1 = splat<T>(-DVC_C1);
    const T e0 = add(x0, x2), e1 = sub(x0, x2);
    const T o0 = fma_(c3, x3, mul(c1, x1));
    const T o1 = fma_(c3, x1, mul(nc1, x3));
    x0 = add(e0, o0);
    x3 = sub(e0, o0);
    x1 = add(e1, o1);
    x2 = sub(e1, o1);
}

// n * o for a packed pair with two scalar multiplications.  ptxas 12.9 contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 in
// spite of the explicit rounding modifiers (it does not for scalar f32, and it sees through fma(n, o, -0.0)); the products of
// coefficient columns 0 and 2 feed the additions of the inverse row butterflies, and the fused form changed one result bit in
// ~1e-4 of the blocks at small q.  A scalar FMUL cannot be folded into a packed FADD2.
DEVI float dequant(float n, float o) { return __fmul_rn(n, o); }
DEVI P2 dequant(P2 n, float o) { float a, b; unp2(n, a, b); return p2(__fmul_rn(a, o), __fmul_rn(b, o)); }

// rint(fl(d_true / q)) * q, scalings folded: d arrives as d_true * 2^NE, leaves as value * 2^-NE.
// FEEDS_ADD: the result is an operand of an addition (see dequant).
template <int NE, bool FEEDS_ADD, typename T>
DEVI T quantise_t(T d, const QuantP& qp) {
    const T r = splat<T>(qp.rcp[NE]), nq = splat<T>(qp.nqs[NE]), magic = splat<T>(12582912.0f);   // 1.5 * 2^23
    const T y0 = mul(d, r);
    const T e = fma_(nq, y0, d);
    const T y = fma_(e, r, y0);                                // == fl(d / (q 2^NE)), correctly rounded
    const T n = sub(add(y, magic), magic);                     // round half to even
    if (FEEDS_ADD) return dequant(n, qp.o[NE]);
    return mul(n, splat<T>(qp.o[NE]));
}

template <typename T>
DEVI void degrade_block_t(T (&v)[4][4], const QuantP& qp) {
#pragma unroll
    for (int r = 0; r < 4; ++r) dct4_fwd_t(v[r][0], v[r][1], v[r][2], v[r][3]);
#pragma unroll
    for (int c = 0; c < 4; ++c) dct4_fwd_t(v[0][c], v[1][c], v[2][c], v[3][c]);
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        // columns 0 and 2 enter the inverse row butterflies through additions, columns 1 and 3 through multiplications
        if ((r & 1) == 0) {
            v[r][0] = quantise_t<2, true>(v[r][0], qp); v[r][1] = quantise_t<1, false>(v[r][1], qp);
            v[r][2] = quantise_t<2, true>(v[r][2], qp); v[r][3] = quantise_t<1, false>(v[r][3], qp);
        } else {
            v[r][0] = quantise_t<1, true>(v[r][0], qp); v[r][1] = quantise_t<0, false>(v[r][1], qp);
            v[r][2] = quantise_t<1, true>(v[r][2], qp); v[r][3] = quantise_t<0, false>(v[r][3], qp);
        }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) dct4_inv_t(v[r][0], v[r][1], v[r][2], v[r][3]);
#pragma unroll
    for (int c = 0; c < 4; ++c) dct4_inv_t(v[0][c], v[1][c], v[2][c], v[3][c]);
}

// float bit patterns of 2^23 + Y for the four pixels in three packed BGR words.
// dp2a.lo: a.lo16 * b.byte0 + a.hi16 * b.byte1; dp2a.hi: a.lo16 * b.byte2 + a.hi16 * b.byte3.
DEVI void luma4_bits(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t (&y)[4]) {
    const uint32_t cBG = 1868u | (9617u << 16), cR_ = 4899u, c_B = 1868u << 16, cGR = 9617u | (4899u << 16);
    const uint32_t s0 = __dp2a_hi(cR_, w0, __dp2a_lo(cBG, w0, 8192u));     // B G R .
    const uint32_t s1 = __dp2a_lo(cGR, w1, __dp2a_hi(c_B, w0, 8192u));     // . . . B | G R
    const uint32_t s2 = __dp2a_lo(cR_, w2, __dp2a_hi(cBG, w1, 8192u));     // . . B G | R
    const uint32_t s3 = __dp2a_hi(cGR, w2, __dp2a_lo(c_B, w2, 8192u));     // . B G R
    // (s >> 14) | 0x4B000000 in one funnel shift: 0x12C0 << 18 == 0x4B000000
    y[0] = __funnelshift_r(s0, 0x12C0u, 14); y[1] = __funnelshift_r(s1, 0x12C0u, 14);
    y[2] = __funnelshift_r(s2, 0x12C0u, 14); y[3] = __funnelshift_r(s3, 0x12C0u, 14);
}

// four grey output bytes -> the three BGR words of four grey pixels
DEVI void grey4_words(uint32_t y0, uint32_t y1, uint32_t y2, uint32_t y3, uint32_t& a, uint32_t& b, uint32_t& c) {
    a = __byte_perm(y0, y1, 0x4000);          // y0 y0 y0 y1
    b = __byte_perm(y1, y2, 0x4400);          // y1 y1 y2 y2
    c = __byte_perm(y2, y3, 0x4440);          // y2 y3 y3 y3
}

// The two 4x4 blocks of one thread, in place in the packed BGR words w[row][6] (block A = words 0..2, B = 3..5).
DEVI void k4_blocks(uint32_t (&w)[4][6], bool st_a, bool st_b, const QuantP& qp) {
    if (st_a && st_b) {
        // ---- both blocks static (97 % of threads on surveillance content): packed lanes A | B ----
        P2 v[4][4];
        const P2 bias = p2(8388736.0f, 8388736.0f);                  // 2^23 + 128
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            uint32_t ya[4], yb[4];
            luma4_bits(w[r][0], w[r][1], w[r][2], ya);
            luma4_bits(w[r][3], w[r][4], w[r][5], yb);
#pragma unroll
            for (int c = 0; c < 4; ++c) v[r][c] = sub(p2(__uint_as_float(ya[c]), __uint_as_float(yb[c])), bias);
        }
        degrade_block_t(v, qp);
        const P2 p128 = p2(128.0f, 128.0f);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            uint32_t ya[4], yb[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                float a, b;
                unp2(add(v[r][c], p128), a, b);
                asm("cvt.rzi.sat.u8.f32 %0, %1;" : "=r"(ya[c]) : "f"(a));
                asm("cvt.rzi.sat.u8.f32 %0, %1;" : "=r"(yb[c]) : "f"(b));
            }
            grey4_words(ya[0], ya[1], ya[2], ya[3], w[r][0], w[r][1], w[r][2]);
            grey4_words(yb[0], yb[1], yb[2], yb[3], w[r][3], w[r][4], w[r][5]);
        }
    } else {
        // ---- a block with motion in this thread: per block, scalar lanes ----
#pragma unroll
        for (int b = 0; b < 2; ++b) {
            if (b == 0 ? st_a : st_b) {
                float v[4][4];
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    uint32_t y[4];
                    luma4_bits(w[r][3 * b], w[r][3 * b + 1], w[r][3 * b + 2], y);
#pragma unroll
                    for (int c = 0; c < 4; ++c) v[r][c] = __fsub_rn(__uint_as_float(y[c]), 8388736.0f);
                }
                degrade_block_t(v, qp);
#pragma unroll
                for (int r = 0; r < 4; ++r)
                    grey4_words(out_byte_bits(v[r][0]), out_byte_bits(v[r][1]), out_byte_bits(v[r][2]),
                                out_byte_bits(v[r][3]), w[r][3 * b], w[r][3 * b + 1], w[r][3 * b + 2]);
            } else {
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    uint32_t o[3] = {0, 0, 0};
#pragma unroll
                    for (int p = 0; p < 4; ++p) {
                        const int i = 12 * b + 3 * p;
                        int bb = byte_at(w[r], i), gg = byte_at(w[r], i + 1), rr = byte_at(w[r], i + 2);
                        ycc_roundtrip(bb, gg, rr);
                        const int j = 3 * p;
                        o[j >> 2] |= (uint32_t)bb << ((j & 3) * 8);
                        o[(j + 1) >> 2] |= (uint32_t)gg << (((j + 1) & 3) * 8);
                        o[(j + 2) >> 2] |= (uint32_t)rr << (((j + 2) & 3) * 8);
                    }
                    w[r][3 * b] = o[0]; w[r][3 * b + 1] = o[1]; w[r][3 * b + 2] = o[2];
                }
            }
        }
    }
}

// One thread per pair of 4x4 blocks (8 px x 4 rows, 8-byte loads and stores: pointers must be 8-byte aligned).  The fallback
// for shapes and pointers the ring kernel below cannot take.
__global__ void __launch_bounds__(256, 4)
k_degrade4p(const uint8_t* __restrict__ frames, const uint32_t* __restrict__ over127,
            const uint32_t* __restrict__ nonzero, uint8_t* __restrict__ compressed, uint8_t* __restrict__ overlay,
            int H, int W, int wpr, QuantP qp, Counters* __restrict__ counters) {
    const int gpr = W >> 3, nbr = H >> 2;
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned n_motion = 0, n_static = 0;
    if (gid < gpr * nbr) {
        const int br = gid / gpr, gx = gid - br * gpr;
        const size_t frame_off = (size_t)blockIdx.y * H * W * 3;
        const size_t plane_off = (size_t)blockIdx.y * H * wpr;
        const size_t base = frame_off + ((size_t)(br * 4) * W + (size_t)gx * 8) * 3;
        const size_t pitch = (size_t)W * 3;
        uint32_t w[4][6];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const uint2 t = __ldcs(reinterpret_cast<const uint2*>(frames + base + r * pitch + 8 * i));
                w[r][2 * i] = t.x; w[r][2 * i + 1] = t.y;
            }
        uint32_t hi[4], nz = 0;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const size_t wo = plane_off + (size_t)(br * 4 + r) * wpr;
            hi[r] = reinterpret_cast<const uint8_t*>(over127 + wo)[gx];
            nz |= reinterpret_cast<const uint8_t*>(nonzero + wo)[gx];
        }
        // ---- overlay: paint (B,G,R) = (0,0,255) where acc > 127 ----
        if (overlay) {
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                uint32_t o[6];
#pragma unroll
                for (int i = 0; i < 6; ++i) o[i] = w[r][i];
                if (hi[r] != 0u) {
#pragma unroll
                    for (int b = 0; b < 2; ++b) {
                        const uint32_t m = hi[r] >> (4 * b);
                        if (m & 1u) { o[3 * b] = (o[3 * b] & 0xff000000u) | 0x00ff0000u; }
                        if (m & 2u) { o[3 * b] &= 0x00ffffffu; o[3 * b + 1] = (o[3 * b + 1] & 0xffff0000u) | 0x0000ff00u; }
                        if (m & 4u) { o[3 * b + 1] &= 0x0000ffffu; o[3 * b + 2] = (o[3 * b + 2] & 0xffffff00u) | 0x000000ffu; }
                        if (m & 8u) { o[3 * b + 2] = (o[3 * b + 2] & 0x000000ffu) | 0xff000000u; }
                    }
                }
#pragma unroll
                for (int i = 0; i < 3; ++i)
                    __stcs(reinterpret_cast<uint2*>(overlay + base + r * pitch + 8 * i), make_uint2(o[2 * i], o[2 * i + 1]));
            }
        }
        n_motion = __popc(hi[0]) + __popc(hi[1]) + __popc(hi[2]) + __popc(hi[3]);
        const bool st_a = (nz & 0xfu) == 0u, st_b = (nz >> 4) == 0u;
        n_static = (st_a ? 1u : 0u) + (st_b ? 1u : 0u);
        if (compressed) {
            k4_blocks(w, st_a, st_b, qp);
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int i = 0; i < 3; ++i)
                    __stcs(reinterpret_cast<uint2*>(compressed + base + r * pitch + 8 * i), make_uint2(w[r][2 * i], w[r][2 * i + 1]));
        }
    }
    // ---- statistics: warp shuffle reduction, one atomic pair per warp ----
    if (counters) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            n_motion += __shfl_xor_sync(0xffffffffu, n_motion, o);
            n_static += __shfl_xor_sync(0xffffffffu, n_static, o);
        }
        if ((threadIdx.x & 31) == 0) {
            if (n_motion) atomicAdd(&counters->motion_pixels, (unsigned long long)n_motion);
            if (n_static) atomicAdd(&counters->static_blocks, (unsigned long long)n_static);
        }
    }
}

DEVI void sts64(uint32_t saddr, uint32_t a, uint32_t b) {
    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(saddr), "r"(a), "r"(b) : "memory");
}
DEVI void lds64(uint32_t saddr, uint32_t& a, uint32_t& b) {
    asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(a), "=r"(b) : "r"(saddr));
}
DEVI uint32_t lds_u8(uint32_t saddr) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}
DEVI void bulk_load(uint32_t sdst, const void* gsrc, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(sdst), "l"(gsrc), "r"(bytes), "r"(bar) : "memory");
}

DEVI void bulk_store(const void* gdst, uint32_t ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(ssrc), "r"(bytes) : "memory");
}

// ------------------------------------------------------------------------------------------------
// block_size 8 (frame_differencing.py:203 main config; motion_compression_opt.py:152-183): one thread per 8x8 block,
// 8 rows x 24 bytes moved with 8-byte vector loads / stores (a warp covers 768 contiguous bytes per row), the pixels
// stay packed in registers.  FLAVOUR 0 = FD (luma quantised, chroma 128), 1 = MCO (Y, Cr and Cb quantised, then
// YCrCb -> BGR -> gray, replicated).  The quotient d / q is the exact IEEE one (quantise_t, Markstein step); the 8x8
// transform pair is the exact restatement of cv2's 2-D routine (k_dct8.cuh).
// ------------------------------------------------------------------------------------------------
// The 8x8 transform pair of one plane with the block staged in shared memory and every pass a ROLLED loop (two rows or two
// columns per trip on the packed pipe).  Fully unrolled in registers the kernel was 7 800 instructions (124 KB) of straight-line
// code and spent most of its time waiting for instruction fetch (ncu: "no_instructions" 60 % of all stall samples, 34 % FP pipe);
// rolled, the hot code is a few hundred instructions and the 64 floats no longer pin 128 registers.
//   sBlk   shared-memory address of this thread's float block: element (r, c) at 4 * (r * 8 + c); threads are K8_BLK_STRIDE
//          bytes apart (66 words: 64-bit accesses of a half-warp touch all 32 banks once)
//   sPl    shared-memory address of row 0 of the byte plane (in: pixels, out: result), rows K8_ROW_STRIDE bytes apart
constexpr int K8_THREADS = 128;
constexpr uint32_t K8_BLK_STRIDE = 66 * 4, K8_ROW_STRIDE = K8_THREADS * 8;
template <int FLAVOUR> constexpr int k8_smem_bytes() { return K8_THREADS * (66 * 4 + (FLAVOUR == 1 ? 3 : 1) * 64); }

DEVI P2 lds_p2(uint32_t saddr) { P2 r; asm volatile("ld.shared.b64 %0, [%1];" : "=l"(r.v) : "r"(saddr)); return r; }
DEVI void sts_p2(uint32_t saddr, P2 v) { asm volatile("st.shared.b64 [%0], %1;" ::"r"(saddr), "l"(v.v) : "memory"); }
DEVI void sts_u16(uint32_t saddr, uint32_t v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(saddr), "h"((unsigned short)v) : "memory"); }

DEVI void degrade_plane8_smem(uint32_t sBlk, uint32_t sPl, const QuantP& qp) {
    // forward rows: bytes -> (value - 128) -> row transform, rows 2i and 2i + 1 in the two lanes
#pragma unroll 1
    for (int i = 0; i < 4; ++i) {
        uint32_t x0[2], x1[2];
        lds64(sPl + (2 * i) * K8_ROW_STRIDE, x0[0], x0[1]);
        lds64(sPl + (2 * i + 1) * K8_ROW_STRIDE, x1[0], x1[1]);
        P2 rp[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) rp[c] = p2((float)((int)byte_at(x0, c) - 128), (float)((int)byte_at(x1, c) - 128));
        dct8x8_row_fwd_t(rp);
        float lo[8], hi[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) unp2(rp[c], lo[c], hi[c]);
#pragma unroll
        for (int c = 0; c < 8; c += 2) {
            sts_p2(sBlk + 4 * ((2 * i) * 8 + c), p2(lo[c], lo[c + 1]));
            sts_p2(sBlk + 4 * ((2 * i + 1) * 8 + c), p2(hi[c], hi[c + 1]));
        }
    }
    // forward columns (2j, 2j + 1 in the two lanes), quantiser, the inverse's row scale
#pragma unroll 1
    for (int j = 0; j < 4; ++j) {
        P2 cp[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) cp[r] = lds_p2(sBlk + 4 * (r * 8 + 2 * j));
        dct8x8_col_fwd_t(cp[0], cp[1], cp[2], cp[3], cp[4], cp[5], cp[6], cp[7]);
#pragma unroll
        for (int r = 0; r < 8; ++r) sts_p2(sBlk + 4 * (r * 8 + 2 * j), mul(quantise_t<0, false>(cp[r], qp), splat<P2>(dct8_rowscale(r))));
    }
    // inverse rows
#pragma unroll 1
    for (int i = 0; i < 4; ++i) {
        float a[8], b[8];
#pragma unroll
        for (int c = 0; c < 8; c += 2) {
            unp2(lds_p2(sBlk + 4 * ((2 * i) * 8 + c)), a[c], a[c + 1]);
            unp2(lds_p2(sBlk + 4 * ((2 * i + 1) * 8 + c)), b[c], b[c + 1]);
        }
        P2 rp[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) rp[c] = p2(a[c], b[c]);
        dct8x8_row_inv_t(rp);
#pragma unroll
        for (int c = 0; c < 8; ++c) unp2(rp[c], a[c], b[c]);
#pragma unroll
        for (int c = 0; c < 8; c += 2) {
            sts_p2(sBlk + 4 * ((2 * i) * 8 + c), p2(a[c], a[c + 1]));
            sts_p2(sBlk + 4 * ((2 * i + 1) * 8 + c), p2(b[c], b[c + 1]));
        }
    }
    // inverse columns, + 128, clip, truncate: two result bytes per row go back into the byte plane
#pragma unroll 1
    for (int j = 0; j < 4; ++j) {
        P2 cp[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) cp[r] = lds_p2(sBlk + 4 * (r * 8 + 2 * j));
        dct8x8_col_inv_t(cp[0], cp[1], cp[2], cp[3], cp[4], cp[5], cp[6], cp[7]);
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            float lo, hi;
            unp2(cp[r], lo, hi);
            sts_u16(sPl + r * K8_ROW_STRIDE + 2 * j, out_byte_bits(lo) | (out_byte_bits(hi) << 8));
        }
    }
}

template <int FLAVOUR>
__global__ void __launch_bounds__(K8_THREADS)
k_degrade8(const uint8_t* __restrict__ frames, const uint32_t* __restrict__ over127, const uint32_t* __restrict__ nonzero,
           uint8_t* __restrict__ compressed, uint8_t* __restrict__ overlay, int H, int W, int wpr, QuantP qp,
           Counters* __restrict__ counters) {
    const int nbx = W >> 3, nby = H >> 3;
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned n_motion = 0, n_static = 0;
    if (gid < nbx * nby) {
        const int by = gid / nbx, bx = gid - by * nbx;
        const size_t pitch = (size_t)W * 3;
        const size_t base = (size_t)blockIdx.y * H * pitch + (size_t)(by * 8) * pitch + (size_t)bx * 24;
        const size_t plane_off = (size_t)blockIdx.y * H * wpr + (size_t)(by * 8) * wpr;
        uint32_t w[8][6];
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const uint2 t = __ldcs(reinterpret_cast<const uint2*>(frames + base + r * pitch + 8 * i));
                w[r][2 * i] = t.x; w[r][2 * i + 1] = t.y;
            }
        uint32_t nz = 0;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const uint32_t hb = reinterpret_cast<const uint8_t*>(over127 + plane_off + (size_t)r * wpr)[bx];
            nz |= reinterpret_cast<const uint8_t*>(nonzero + plane_off + (size_t)r * wpr)[bx];
            n_motion += __popc(hb);
            if (overlay) {
                uint32_t o[6];
#pragma unroll
                for (int i = 0; i < 6; ++i) o[i] = w[r][i];
                if (hb) {
#pragma unroll
                    for (int b = 0; b < 2; ++b) {
                        const uint32_t m = hb >> (4 * b);
                        if (m & 1u) { o[3 * b] = (o[3 * b] & 0xff000000u) | 0x00ff0000u; }
                        if (m & 2u) { o[3 * b] &= 0x00ffffffu; o[3 * b + 1] = (o[3 * b + 1] & 0xffff0000u) | 0x0000ff00u; }
                        if (m & 4u) { o[3 * b + 1] &= 0x0000ffffu; o[3 * b + 2] = (o[3 * b + 2] & 0xffffff00u) | 0x000000ffu; }
                        if (m & 8u) { o[3 * b + 2] = (o[3 * b + 2] & 0x000000ffu) | 0xff000000u; }
                    }
                }
#pragma unroll
                for (int i = 0; i < 3; ++i)
                    __stcs(reinterpret_cast<uint2*>(overlay + base + r * pitch + 8 * i), make_uint2(o[2 * i], o[2 * i + 1]));
            }
        }
        const bool is_static = nz == 0u;
        n_static = is_static ? 1u : 0u;
        if (compressed) {
            if (!is_static) {
#pragma unroll
                for (int r = 0; r < 8; ++r) {
                    uint32_t o[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll
                    for (int p = 0; p < 8; ++p) {
                        int bb = byte_at(w[r], 3 * p), gg = byte_at(w[r], 3 * p + 1), rr = byte_at(w[r], 3 * p + 2);
                        ycc_roundtrip(bb, gg, rr);
                        const int j = 3 * p;
                        o[j >> 2] |= (uint32_t)bb << ((j & 3) * 8);
                        o[(j + 1) >> 2] |= (uint32_t)gg << (((j + 1) & 3) * 8);
                        o[(j + 2) >> 2] |= (uint32_t)rr << (((j + 2) & 3) * 8);
                    }
#pragma unroll
                    for (int i = 0; i < 6; ++i) w[r][i] = o[i];
                }
            } else {
                // Static block.  Every stage is a rolled loop over rows (the pixel words are parked in this thread's float-block
                // area, which the transform only needs afterwards), so the hot code stays small enough for the instruction cache.
                extern __shared__ __align__(16) uint8_t k8_smem[];
                const uint32_t sBlk = (uint32_t)__cvta_generic_to_shared(k8_smem) + threadIdx.x * K8_BLK_STRIDE;
                const uint32_t sQ = (uint32_t)__cvta_generic_to_shared(k8_smem) + K8_THREADS * K8_BLK_STRIDE + threadIdx.x * 8u;   // + (plane * 8 + row) * K8_ROW_STRIDE
#pragma unroll
                for (int r = 0; r < 8; ++r)
#pragma unroll
                    for (int i = 0; i < 3; ++i) sts64(sBlk + r * 24 + 8 * i, w[r][2 * i], w[r][2 * i + 1]);
                // pixels -> byte planes: Y (fd:115-116), and Cr, Cb for the MCO flavour (mco:152-153)
#pragma unroll 1
                for (int r = 0; r < 8; ++r) {
                    uint32_t x[6], ya[4], yb[4];
#pragma unroll
                    for (int i = 0; i < 3; ++i) lds64(sBlk + r * 24 + 8 * i, x[2 * i], x[2 * i + 1]);
                    luma4_bits(x[0], x[1], x[2], ya);
                    luma4_bits(x[3], x[4], x[5], yb);
                    sts64(sQ + r * K8_ROW_STRIDE,
                          (ya[0] & 0xffu) | ((ya[1] & 0xffu) << 8) | ((ya[2] & 0xffu) << 16) | (ya[3] << 24),
                          (yb[0] & 0xffu) | ((yb[1] & 0xffu) << 8) | ((yb[2] & 0xffu) << 16) | (yb[3] << 24));
                    if (FLAVOUR == 1) {
                        uint32_t crw[2] = {0u, 0u}, cbw[2] = {0u, 0u};
#pragma unroll
                        for (int c = 0; c < 8; ++c) {
                            const int y = (int)((c < 4 ? ya[c] : yb[c - 4]) & 0xffu);
                            const int cr = sat8((((int)byte_at(x, 3 * c + 2) - y) * 11682 + (128 << 14) + 8192) >> 14);
                            const int cb = sat8((((int)byte_at(x, 3 * c) - y) * 9241 + (128 << 14) + 8192) >> 14);
                            crw[c >> 2] |= (uint32_t)cr << ((c & 3) * 8);
                            cbw[c >> 2] |= (uint32_t)cb << ((c & 3) * 8);
                        }
                        sts64(sQ + (8 + r) * K8_ROW_STRIDE, crw[0], crw[1]);
                        sts64(sQ + (16 + r) * K8_ROW_STRIDE, cbw[0], cbw[1]);
                    }
                }
                // quantise the plane(s): motion_compression_opt.py:162-168 does Y, Cr and Cb, frame_differencing.py:121-125 only Y
#pragma unroll 1
                for (int k = 0; k < (FLAVOUR == 1 ? 3 : 1); ++k) degrade_plane8_smem(sBlk, sQ + (k * 8) * K8_ROW_STRIDE, qp);
                // planes -> output pixels, stored row by row: grey Y' (fd: chroma 128, :126-130) or YCrCb -> BGR -> gray (mco:171,181-183)
#pragma unroll 1
                for (int r = 0; r < 8; ++r) {
                    uint32_t qy[2], gy[8], o[6];
                    lds64(sQ + r * K8_ROW_STRIDE, qy[0], qy[1]);
                    if (FLAVOUR == 1) {
                        uint32_t qr[2], qb[2];
                        lds64(sQ + (8 + r) * K8_ROW_STRIDE, qr[0], qr[1]);
                        lds64(sQ + (16 + r) * K8_ROW_STRIDE, qb[0], qb[1]);
#pragma unroll
                        for (int c = 0; c < 8; ++c) {
                            const int y = (int)byte_at(qy, c), cr = (int)byte_at(qr, c) - 128, cb = (int)byte_at(qb, c) - 128;
                            const int b = sat8(y + ((29049 * cb + 8192) >> 14));
                            const int gg = sat8(y + ((-5636 * cb - 11698 * cr + 8192) >> 14));
                            const int rr = sat8(y + ((22987 * cr + 8192) >> 14));
                            gy[c] = gray_of(b, gg, rr);
                        }
                    } else {
#pragma unroll
                        for (int c = 0; c < 8; ++c) gy[c] = byte_at(qy, c);
                    }
                    grey4_words(gy[0], gy[1], gy[2], gy[3], o[0], o[1], o[2]);
                    grey4_words(gy[4], gy[5], gy[6], gy[7], o[3], o[4], o[5]);
#pragma unroll
                    for (int i = 0; i < 3; ++i)
                        __stcs(reinterpret_cast<uint2*>(compressed + base + r * pitch + 8 * i), make_uint2(o[2 * i], o[2 * i + 1]));
                }
            }
            if (!is_static) {
#pragma unroll
                for (int r = 0; r < 8; ++r)
#pragma unroll
                    for (int i = 0; i < 3; ++i)
                        __stcs(reinterpret_cast<uint2*>(compressed + base + r * pitch + 8 * i), make_uint2(w[r][2 * i], w[r][2 * i + 1]));
            }
        }
    }
    if (counters) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            n_motion += __shfl_xor_sync(0xffffffffu, n_motion, o);
            n_static += __shfl_xor_sync(0xffffffffu, n_static, o);
        }
        if ((threadIdx.x & 31) == 0) {
            if (n_motion) atomicAdd(&counters->motion_pixels, (unsigned long long)n_motion);
            if (n_static) atomicAdd(&counters->static_blocks, (unsigned long long)n_static);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Tile geometry of the ring kernel below: a tile is a span of whole 4-pixel-high block rows (contiguous in the frame), or
// an exact part of one block row for W > 2048.  (A one-shot CTA-per-span kernel built on the same geometry was measured
// and dropped: profiles/r1l_k4_experiments.txt section 2.)
// ------------------------------------------------------------------------------------------------
struct K4Geom {
    int gp;          // pixel groups (8 px) per CTA row piece
    int parts;       // CTAs per block row (1 = whole block rows per CTA)
    int nb;          // block rows per CTA when parts == 1
    int sp;          // shared-memory row pitch in bytes (= W * 3 when parts == 1, gp * 24 otherwise)
    int span_bytes;  // bytes of one span buffer
    int mask_bytes;  // bytes of one mask-plane row group buffer (4 * nb rows of wpr words)
};

// ------------------------------------------------------------------------------------------------
// Persistent, warp-specialised K4 (block_size 4): one CTA per SM walks tiles t = blockIdx.x, blockIdx.x + gridDim.x, ...
// over all frames of the launch.  A tile is the K4Geom span (whole block rows, or part of one for W > 2048).
//   loader (lane 0 of the       waits for "free[s]", then cp.async.bulk loads of span + mask rows into stage s of a
//   last warp)                  ring of `stages` input buffers, completing on "full[s]" (mbarrier expect_tx).  Its
//                               per-tile instruction chain is a barrier wait and a handful of copies, nothing else.
//   2 consumer groups of 256    wait for "full", LDS.64 their 8 px x 4 rows, paint the overlay in place in the
//   threads                     input buffer, run k4_blocks, STS.64 the compressed pixels into the group's output
//                               buffer, fence.proxy.async, group barrier; then the group's two issuer lanes send the
//                               tile out with cp.async.bulk stores (lane 0 the overlay from the input stage, lane 1
//                               the compressed pixels from the output buffer) and, one tile later, after
//                               cp.async.bulk.wait_group.read, hand the stage back to the loader ("free") and the
//                               output buffer back to the group.
// A contiguous span is at most 256 pixel groups x 96 B = 24 KB and moves as one bulk operation per buffer (smaller pieces
// were measured from 1.4 KB up without a gain: profiles/README.md, r1l); a part of a block row moves as its four rows.
// Shared memory: `stages` x (span + 2 mask row groups) + 2 x span (6 x 25 KB + 2 x 23 KB at 1080p).
// HBM sees a steady stream of bulk operations whose depth is `stages`, independent of CTA launch / drain behaviour;
// consumers never touch global memory (statistics: one atomic pair per warp per launch).
// ------------------------------------------------------------------------------------------------
struct K4SGeom {
    K4Geom g;
    int stages;            // input ring depth (more than K4S_GROUPS)
    int tiles_per_frame;
    int n_tiles;           // tiles_per_frame * frames
    int stage_bytes;       // span_bytes + 2 * mask_bytes, rounded up to 128
    int ybuf_bytes;        // span_bytes rounded up to 128
};

constexpr int K4S_GROUPS = 2;                               // consumer groups of 256 threads
constexpr int K4S_THREADS = K4S_GROUPS * 256 + 32;          // + the loader warp
constexpr int K4S_ISSUERS = 2;                              // lanes 0 and 1 of a consumer group issue its stores

DEVI void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    }
}
DEVI void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
DEVI void group_sync(int id) { asm volatile("bar.sync %0, 256;" ::"r"(id) : "memory"); }

// tile walker: (frame, tile-in-frame) advanced by a fixed number of tiles without divisions
struct K4Walk {
    int f, l, df, dl, tpf;
    DEVI void init(int t0, int step, int tiles_per_frame) {
        tpf = tiles_per_frame; f = t0 / tpf; l = t0 - f * tpf; df = step / tpf; dl = step - df * tpf;
    }
    DEVI void next() { f += df; l += dl; if (l >= tpf) { l -= tpf; ++f; } }
};
struct K4Tile { size_t span_off, mask_off; int nbv, g0, ng; };
DEVI K4Tile k4_tile(const K4Walk& wk, const K4Geom& g, int H, int W, int wpr) {
    const int gpr = W >> 3, nbr = H >> 2;
    K4Tile r;
    int br0;
    if (g.parts == 1) { br0 = wk.l * g.nb; r.nbv = min(g.nb, nbr - br0); r.g0 = 0; r.ng = gpr; }
    else { br0 = wk.l / g.parts; r.nbv = 1; r.g0 = (wk.l - br0 * g.parts) * g.gp; r.ng = min(g.gp, gpr - r.g0); }
    r.span_off = ((size_t)wk.f * H + (size_t)(br0 * 4)) * W * 3 + (size_t)r.g0 * 24;
    r.mask_off = ((size_t)wk.f * H + (size_t)(br0 * 4)) * wpr;
    return r;
}

__global__ void __launch_bounds__(K4S_THREADS, 1)
k_degrade4s(const uint8_t* __restrict__ frames, const uint32_t* __restrict__ over127,
            const uint32_t* __restrict__ nonzero, uint8_t* __restrict__ compressed, uint8_t* __restrict__ overlay,
            int H, int W, int wpr, QuantP qp, Counters* __restrict__ counters, K4SGeom sg) {
    extern __shared__ __align__(128) uint8_t k4_smem[];
    const K4Geom& g = sg.g;
    const uint32_t s0 = (uint32_t)__cvta_generic_to_shared(k4_smem);
    const int S = sg.stages;
    const uint32_t ybufs = s0 + (uint32_t)S * (uint32_t)sg.stage_bytes;              // K4S_GROUPS output buffers
    const uint32_t bars = ybufs + (uint32_t)K4S_GROUPS * (uint32_t)sg.ybuf_bytes;    // full[S], free[S]
    const uint32_t desc = (bars + 8u * (uint32_t)(2 * S) + 15u) & ~15u;              // per stage: {nbv, g0, ng, -}
    const int tid = threadIdx.x;
    const int first = blockIdx.x, stride = gridDim.x;
    const int nj = first < sg.n_tiles ? (sg.n_tiles - first + stride - 1) / stride : 0;
    const uint32_t pitch = (uint32_t)W * 3u;
    const uint32_t mrow_bytes = (uint32_t)wpr * 4u;
    const bool contiguous = g.parts == 1;

    if (tid == 0) {
        for (int s = 0; s < S; ++s) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bars + 8u * s));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bars + 8u * (S + s)), "r"(K4S_ISSUERS));
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (tid >= K4S_GROUPS * 256) {
        // ------------------------------ loader ------------------------------
        if (tid > K4S_GROUPS * 256) return;
        K4Walk wl;
        wl.init(first, stride, sg.tiles_per_frame);
        for (int j = 0; j < nj; ++j) {
            const int s = j % S;
            const K4Tile t = k4_tile(wl, g, H, W, wpr);
            wl.next();
            const uint32_t sX = s0 + (uint32_t)s * (uint32_t)sg.stage_bytes;
            const uint32_t sMh = sX + g.span_bytes, sMn = sMh + g.mask_bytes;
            const uint32_t full = bars + 8u * s;
            const uint32_t mbytes = (uint32_t)(4 * t.nbv) * mrow_bytes;
            const uint32_t rows = contiguous ? (uint32_t)(4 * t.nbv) : 4u;
            const uint32_t rbytes = contiguous ? pitch : (uint32_t)t.ng * 24u;
            if (j >= S) mbar_wait(bars + 8u * (S + s), (uint32_t)(j / S - 1) & 1u);       // the stage's previous tile has left
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(desc + 16u * s), "r"(t.nbv), "r"(t.g0), "r"(t.ng), "r"(0) : "memory");
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full), "r"(rows * rbytes + 2u * mbytes) : "memory");
            if (contiguous) bulk_load(sX, frames + t.span_off, rows * rbytes, full);
            else
                for (uint32_t r = 0; r < rows; ++r) bulk_load(sX + r * g.sp, frames + t.span_off + (size_t)r * pitch, rbytes, full);
            bulk_load(sMh, over127 + t.mask_off, mbytes, full);
            bulk_load(sMn, nonzero + t.mask_off, mbytes, full);
        }
        return;
    }

    // ------------------------------ consumers ------------------------------
    const int grp = tid >> 8, t = tid & 255;
    const bool issuer = t < K4S_ISSUERS;
    const int gpr = W >> 3;
    int brl = 0, gxl = t;
    if (contiguous) { brl = t / gpr; gxl = t - brl * gpr; }
    const uint32_t toff = (uint32_t)(brl * 4) * (uint32_t)g.sp + (uint32_t)gxl * 24u;
    const uint32_t sY = ybufs + (uint32_t)grp * (uint32_t)sg.ybuf_bytes;
    unsigned n_motion = 0, n_static = 0;
    K4Walk ws;                              // this group's tiles, for the store addresses
    ws.init(first + grp * stride, K4S_GROUPS * stride, sg.tiles_per_frame);
    int s_prev = -1;
    for (int j = grp; j < nj; j += K4S_GROUPS) {
        const int s = j % S;
        const uint32_t sX = s0 + (uint32_t)s * (uint32_t)sg.stage_bytes;
        const uint32_t sMh = sX + g.span_bytes, sMn = sMh + g.mask_bytes;
        mbar_wait(bars + 8u * s, (uint32_t)(j / S) & 1u);
        uint32_t nbv, tg0, tng, unused;
        asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(nbv), "=r"(tg0), "=r"(tng), "=r"(unused) : "r"(desc + 16u * s));
        const bool active = brl < (int)nbv && gxl < (int)tng;
        uint32_t w[4][6];
        if (active) {
            const uint32_t moff = (uint32_t)(brl * 4) * mrow_bytes + tg0 + (uint32_t)gxl;
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int i = 0; i < 3; ++i) lds64(sX + toff + r * g.sp + 8 * i, w[r][2 * i], w[r][2 * i + 1]);
            uint32_t hi[4], nz = 0;
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                hi[r] = lds_u8(sMh + moff + r * mrow_bytes);
                nz |= lds_u8(sMn + moff + r * mrow_bytes);
            }
            if (overlay) {
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    if (hi[r] == 0u) continue;
                    uint32_t o[6];
#pragma unroll
                    for (int i = 0; i < 6; ++i) o[i] = w[r][i];
#pragma unroll
                    for (int b = 0; b < 2; ++b) {
                        const uint32_t m = hi[r] >> (4 * b);
                        if (m & 1u) { o[3 * b] = (o[3 * b] & 0xff000000u) | 0x00ff0000u; }
                        if (m & 2u) { o[3 * b] &= 0x00ffffffu; o[3 * b + 1] = (o[3 * b + 1] & 0xffff0000u) | 0x0000ff00u; }
                        if (m & 4u) { o[3 * b + 1] &= 0x0000ffffu; o[3 * b + 2] = (o[3 * b + 2] & 0xffffff00u) | 0x000000ffu; }
                        if (m & 8u) { o[3 * b + 2] = (o[3 * b + 2] & 0x000000ffu) | 0xff000000u; }
                    }
#pragma unroll
                    for (int i = 0; i < 3; ++i) sts64(sX + toff + r * g.sp + 8 * i, o[2 * i], o[2 * i + 1]);
                }
            }
            n_motion += __popc(hi[0]) + __popc(hi[1]) + __popc(hi[2]) + __popc(hi[3]);
            const bool st_a = (nz & 0xfu) == 0u, st_b = (nz >> 4) == 0u;
            n_static += (st_a ? 1u : 0u) + (st_b ? 1u : 0u);
            if (compressed) k4_blocks(w, st_a, st_b, qp);
        }
        // the previous tile's stores have read their shared-memory sources: its input stage goes back to the loader,
        // the output buffer back to the group
        if (issuer && s_prev >= 0) {
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            mbar_arrive(bars + 8u * (S + s_prev));
        }
        group_sync(1 + grp);
        if (compressed && active) {
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int i = 0; i < 3; ++i) sts64(sY + toff + r * g.sp + 8 * i, w[r][2 * i], w[r][2 * i + 1]);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        group_sync(1 + grp);
        if (issuer) {
            uint8_t* dst = t == 0 ? overlay : compressed;
            if (dst) {
                const K4Tile tl = k4_tile(ws, g, H, W, wpr);
                const uint32_t src = t == 0 ? sX : sY;
                if (contiguous) bulk_store(dst + tl.span_off, src, 4u * nbv * pitch);
                else
                    for (uint32_t r = 0; r < 4; ++r) bulk_store(dst + tl.span_off + (size_t)r * pitch, src + r * g.sp, tng * 24u);
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            s_prev = s;
        }
        ws.next();
    }
    if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");        // shared memory must outlive the reads
    if (counters) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            n_motion += __shfl_xor_sync(0xffffffffu, n_motion, o);
            n_static += __shfl_xor_sync(0xffffffffu, n_static, o);
        }
        if ((tid & 31) == 0) {
            if (n_motion) atomicAdd(&counters->motion_pixels, (unsigned long long)n_motion);
            if (n_static) atomicAdd(&counters->static_blocks, (unsigned long long)n_static);
        }
    }
}

}  // namespace dvc
