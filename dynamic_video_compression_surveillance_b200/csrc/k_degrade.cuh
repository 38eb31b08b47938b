// K4: overlay paint + BGR->YCrCb + block-DCT degrade of static blocks + YCrCb->BGR, and the
// statistics, in one pass over the frame (frame_differencing.py:110-111,115-130;
// motion_compression_opt.py:152-183).
//
// Inputs are the BGR frame and two bit-planes of the accumulated mask: over127 (acc > 127, the
// overlay test, frame_differencing.py:111) and nonzero (acc != 0; a block is static when its
// nonzero bits are all clear, which is what `.mean() == 0` says, :120).
//
// Arithmetic contract (SURVEY.md section 2.1, re-verified in tests/test_oracle_vs_cv2.py):
//   BGR->YCrCb   Y  = (1868 B + 9617 G + 4899 R + 8192) >> 14
//                Cr = sat(((R - Y) * 11682 + (128 << 14) + 8192) >> 14),  Cb likewise with B, 9241
//   YCrCb->BGR   B = sat(Y + ((29049 Cb' + 8192) >> 14)),  R = sat(Y + ((22987 Cr' + 8192) >> 14)),
//                G = sat(Y + ((-5636 Cb' - 11698 Cr' + 8192) >> 14)),  ' = minus 128
//   static block Y' = trunc(clip(idct(rint(dct(Y - 128) / q) * q) + 128, 0, 255)), chroma 128 => B=G=R=Y'
// The 4-point DCT below reproduces cv2.dct / cv2.idct (IPP build, float32) bit for bit: the operation
// order and the two FMAs were recovered by search against cv2 on 200 000 random vectors (DESIGN.md).
#pragma once
#include "k_dct8.cuh"

namespace dvc {

// np.round(d / q) * q in float32: IEEE division, round half to even, exact product
DEVI float quantise(float d, float q) { return __fmul_rn(rintf(__fdiv_rn(d, q)), q); }

DEVI uint32_t clip_trunc_u8(float v) {   // np.clip(v, 0, 255) stored into a uint8 array
    return (uint32_t)__float2int_rz(fminf(fmaxf(v, 0.0f), 255.0f));
}

DEVI int luma_of(int b, int g, int r) { return (1868 * b + 9617 * g + 4899 * r + 8192) >> 14; }
DEVI int sat8(int v) { return min(255, max(0, v)); }

// BGR -> YCrCb -> BGR of one pixel (the non-static path: pure integer round trip)
DEVI void ycc_roundtrip(int& b, int& g, int& r) {
    const int y = luma_of(b, g, r);
    const int cr = sat8(((r - y) * 11682 + (128 << 14) + 8192) >> 14) - 128;
    const int cb = sat8(((b - y) * 9241 + (128 << 14) + 8192) >> 14) - 128;
    b = sat8(y + ((29049 * cb + 8192) >> 14));
    g = sat8(y + ((-5636 * cb - 11698 * cr + 8192) >> 14));
    r = sat8(y + ((22987 * cr + 8192) >> 14));
}

// 4x4 block, full 2-D transform pair on luma (rows first, then columns, as cv2 does)
DEVI void degrade_block4(float (&v)[4][4], float q) {
#pragma unroll
    for (int r = 0; r < 4; ++r) dct4_fwd(v[r][0], v[r][1], v[r][2], v[r][3]);
#pragma unroll
    for (int c = 0; c < 4; ++c) dct4_fwd(v[0][c], v[1][c], v[2][c], v[3][c]);
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) v[r][c] = quantise(v[r][c], q);
#pragma unroll
    for (int r = 0; r < 4; ++r) dct4_inv(v[r][0], v[r][1], v[r][2], v[r][3]);
#pragma unroll
    for (int c = 0; c < 4; ++c) dct4_inv(v[0][c], v[1][c], v[2][c], v[3][c]);
}

struct Counters { unsigned long long frames, pixels, motion_pixels, blocks, static_blocks; };

__global__ void k_counters_add(Counters* c, unsigned long long frames, unsigned long long pixels, unsigned long long blocks) {
    atomicAdd(&c->frames, frames);
    atomicAdd(&c->pixels, pixels);
    atomicAdd(&c->blocks, blocks);
}

// np.clip(v + 128, 0, 255) stored to uint8 (truncation): one saturating round-toward-zero conversion
DEVI uint32_t out_byte_bits(float v) {
    uint32_t r;
    asm("cvt.rzi.sat.u8.f32 %0, %1;" : "=r"(r) : "f"(__fadd_rn(v, 128.0f)));
    return r;
}

// ------------------------------------------------------------------------------------------------
// General path: block_size 4 or 8, any W, H that are multiples of block_size, both flavours.
// One thread per block, bytewise access, IEEE division in the quantiser: exact for every q and any
// pointer alignment.  The fallback of the packed kernels (k_degrade4p.cuh) for W % 8 != 0, q outside
// [0.01, 1e6] and pointers that are not 8-byte aligned.  8x8 blocks use the exact restatement of cv2's
// 2-D routine in k_dct8.cuh.
// ------------------------------------------------------------------------------------------------
template <int BS>
DEVI void degrade_plane(float (&v)[BS][BS], float q) {
    if constexpr (BS == 4) degrade_block4(v, q);
    else degrade_block8_exact(v, [q](float d) { return quantise(d, q); });
}

template <int BS, int FLAVOUR>   // FLAVOUR 0 = FD, 1 = MCO
__global__ void __launch_bounds__(128)
k_degrade_generic(const uint8_t* __restrict__ frames, const uint32_t* __restrict__ over127,
                  const uint32_t* __restrict__ nonzero, uint8_t* __restrict__ compressed,
                  uint8_t* __restrict__ overlay, int H, int W, int wpr, float q, Counters* __restrict__ counters) {
    const int nbx = W / BS, nby = H / BS;
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned n_motion = 0, n_static = 0;
    if (gid < nbx * nby) {
        const int by = gid / nbx, bx = gid - by * nbx;
        const int x0 = bx * BS, y0 = by * BS;
        const uint8_t* fr = frames + (size_t)blockIdx.y * H * W * 3;
        const size_t plane_off = (size_t)blockIdx.y * H * wpr;
        uint32_t nz = 0;
        for (int r = 0; r < BS; ++r) {
            const size_t wo = plane_off + (size_t)(y0 + r) * wpr;
            const uint32_t hb = (over127[wo + (x0 >> 5)] >> (x0 & 31)) & ((1u << BS) - 1u);
            nz |= (nonzero[wo + (x0 >> 5)] >> (x0 & 31)) & ((1u << BS) - 1u);
            n_motion += __popc(hb);
            if (overlay) {
                uint8_t* orow = overlay + (size_t)blockIdx.y * H * W * 3 + ((size_t)(y0 + r) * W + x0) * 3;
                const uint8_t* irow = fr + ((size_t)(y0 + r) * W + x0) * 3;
                for (int c = 0; c < BS; ++c) {
                    const bool m = (hb >> c) & 1u;
                    orow[3 * c] = m ? 0 : irow[3 * c];
                    orow[3 * c + 1] = m ? 0 : irow[3 * c + 1];
                    orow[3 * c + 2] = m ? 255 : irow[3 * c + 2];
                }
            }
        }
        const bool is_static = nz == 0u;
        if (is_static) ++n_static;
        if (compressed) {
            uint8_t* out = compressed + (size_t)blockIdx.y * H * W * 3;
            if (!is_static) {
                for (int r = 0; r < BS; ++r)
                    for (int c = 0; c < BS; ++c) {
                        const size_t o = ((size_t)(y0 + r) * W + x0 + c) * 3;
                        int b = fr[o], g = fr[o + 1], rr = fr[o + 2];
                        ycc_roundtrip(b, g, rr);
                        out[o] = (uint8_t)b; out[o + 1] = (uint8_t)g; out[o + 2] = (uint8_t)rr;
                    }
            } else if (FLAVOUR == 0) {
                float v[BS][BS];
#pragma unroll
                for (int r = 0; r < BS; ++r)
#pragma unroll
                    for (int c = 0; c < BS; ++c) {
                        const size_t o = ((size_t)(y0 + r) * W + x0 + c) * 3;
                        v[r][c] = (float)(luma_of(fr[o], fr[o + 1], fr[o + 2]) - 128);
                    }
                degrade_plane<BS>(v, q);
#pragma unroll
                for (int r = 0; r < BS; ++r)
#pragma unroll
                    for (int c = 0; c < BS; ++c) {
                        const size_t o = ((size_t)(y0 + r) * W + x0 + c) * 3;
                        const uint8_t y = (uint8_t)clip_trunc_u8(__fadd_rn(v[r][c], 128.0f));
                        out[o] = y; out[o + 1] = y; out[o + 2] = y;
                    }
            } else {
                // MCO: quantise Y, Cr, Cb; YCrCb->BGR; BGR->gray; replicate (motion_compression_opt.py:162-183)
                float v[BS][BS];
                uint8_t ch[3][BS][BS];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
#pragma unroll
                    for (int r = 0; r < BS; ++r)
#pragma unroll
                        for (int c = 0; c < BS; ++c) {
                            const size_t o = ((size_t)(y0 + r) * W + x0 + c) * 3;
                            const int b = fr[o], g = fr[o + 1], rr = fr[o + 2];
                            const int y = luma_of(b, g, rr);
                            int val = y;
                            if (k == 1) val = sat8(((rr - y) * 11682 + (128 << 14) + 8192) >> 14);
                            if (k == 2) val = sat8(((b - y) * 9241 + (128 << 14) + 8192) >> 14);
                            v[r][c] = (float)(val - 128);
                        }
                    degrade_plane<BS>(v, q);
#pragma unroll
                    for (int r = 0; r < BS; ++r)
#pragma unroll
                        for (int c = 0; c < BS; ++c) ch[k][r][c] = (uint8_t)clip_trunc_u8(__fadd_rn(v[r][c], 128.0f));
                }
#pragma unroll
                for (int r = 0; r < BS; ++r)
#pragma unroll
                    for (int c = 0; c < BS; ++c) {
                        const int y = ch[0][r][c], cr = ch[1][r][c] - 128, cb = ch[2][r][c] - 128;
                        const int b = sat8(y + ((29049 * cb + 8192) >> 14));
                        const int g = sat8(y + ((-5636 * cb - 11698 * cr + 8192) >> 14));
                        const int rr = sat8(y + ((22987 * cr + 8192) >> 14));
                        const uint8_t gy = (uint8_t)gray_of(b, g, rr);
                        const size_t o = ((size_t)(y0 + r) * W + x0 + c) * 3;
                        out[o] = gy; out[o + 1] = gy; out[o + 2] = gy;
                    }
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
// Clipped edge blocks: frames whose size is not a multiple of block_size (frame_differencing.py:117-121 slices the last
// block of a row / column shorter; motion_compression_opt.py:159 skips partial blocks).  One thread per edge block: the right
// column of partial blocks (all block rows) and the bottom row (all full block columns).  Clipped blocks are bit-exact
// through the 1-D routines of k_dct8.cuh (every length 1..8).
// A frame has at most W / bs + H / bs + 1 such blocks, so this launch costs microseconds.
// ------------------------------------------------------------------------------------------------
template <int FLAVOUR>
__global__ void __launch_bounds__(64)
k_degrade_edges(const uint8_t* __restrict__ frames, const uint32_t* __restrict__ over127, const uint32_t* __restrict__ nonzero,
                uint8_t* __restrict__ compressed, uint8_t* __restrict__ overlay, int H, int W, int wpr, int bs, float q,
                Counters* __restrict__ counters, int all_blocks) {
    const int nbx = W / bs, nbx_c = (W + bs - 1) / bs, nby_c = (H + bs - 1) / bs;
    const int n_right = W % bs ? nby_c : 0, n_bottom = H % bs ? nbx : 0;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    // all_blocks: every block of the frame goes through this general path (block sizes other than 4 and 8)
    if (e >= (all_blocks ? nbx_c * nby_c : n_right + n_bottom)) return;
    const int bx = all_blocks ? e % nbx_c : (e < n_right ? nbx_c - 1 : e - n_right);
    const int by = all_blocks ? e / nbx_c : (e < n_right ? e : nby_c - 1);
    const int x0 = bx * bs, y0 = by * bs, bw = min(bs, W - x0), bh = min(bs, H - y0);
    const uint8_t* fr = frames + (size_t)blockIdx.y * H * W * 3;
    const size_t plane_off = (size_t)blockIdx.y * H * wpr;
    unsigned n_motion = 0;
    bool any_nz = false;
    for (int r = 0; r < bh; ++r) {
        const size_t wo = plane_off + (size_t)(y0 + r) * wpr;
        for (int c = 0; c < bw; ++c) {
            const int x = x0 + c;
            const bool hi = (over127[wo + (x >> 5)] >> (x & 31)) & 1u;
            any_nz |= ((nonzero[wo + (x >> 5)] >> (x & 31)) & 1u) != 0;
            n_motion += hi ? 1u : 0u;
            if (overlay) {
                const size_t o = (size_t)blockIdx.y * H * W * 3 + ((size_t)(y0 + r) * W + x) * 3;
                overlay[o] = hi ? 0 : frames[o]; overlay[o + 1] = hi ? 0 : frames[o + 1]; overlay[o + 2] = hi ? 255 : frames[o + 2];
            }
        }
    }
    const bool is_static = FLAVOUR == 0 && !any_nz;
    if (compressed) {
        uint8_t* out = compressed + (size_t)blockIdx.y * H * W * 3;
        if (!is_static) {
            for (int r = 0; r < bh; ++r)
                for (int c = 0; c < bw; ++c) {
                    const size_t o = ((size_t)(y0 + r) * W + x0 + c) * 3;
                    int b = fr[o], g = fr[o + 1], rr = fr[o + 2];
                    ycc_roundtrip(b, g, rr);
                    out[o] = (uint8_t)b; out[o + 1] = (uint8_t)g; out[o + 2] = (uint8_t)rr;
                }
        } else {
            float v[8][8];
            for (int r = 0; r < bh; ++r)
                for (int c = 0; c < bw; ++c) {
                    const size_t o = ((size_t)(y0 + r) * W + x0 + c) * 3;
                    v[r][c] = (float)(luma_of(fr[o], fr[o + 1], fr[o + 2]) - 128);
                }
            // cv2.dct on a clipped block: rows, then columns, forward and inverse alike, each through the 1-D routine of
            // its length (k_dct8.cuh, exact for every length 1..8).
            for (int r = 0; r < bh; ++r) dct1d(&v[r][0], bw, 1, false);
            for (int c = 0; c < bw; ++c) dct1d(&v[0][c], bh, 8, false);
            for (int r = 0; r < bh; ++r)
                for (int c = 0; c < bw; ++c) v[r][c] = quantise(v[r][c], q);
            for (int r = 0; r < bh; ++r) dct1d(&v[r][0], bw, 1, true);
            for (int c = 0; c < bw; ++c) dct1d(&v[0][c], bh, 8, true);
            for (int r = 0; r < bh; ++r)
                for (int n = 0; n < bw; ++n) {
                    const uint8_t y = (uint8_t)clip_trunc_u8(__fadd_rn(v[r][n], 128.0f));
                    const size_t o = ((size_t)(y0 + r) * W + x0 + n) * 3;
                    out[o] = y; out[o + 1] = y; out[o + 2] = y;
                }
        }
    }
    if (counters) {
        if (n_motion) atomicAdd(&counters->motion_pixels, (unsigned long long)n_motion);
        if (is_static) atomicAdd(&counters->static_blocks, 1ull);
    }
}

// cv2.dct / cv2.idct on a stack of float32 blocks (dvc_dct_blocks_f32): one thread per block.
__global__ void __launch_bounds__(128)
k_dct_blocks(const float* __restrict__ src, float* __restrict__ dst, long long n, int bh, int bw, int inverse) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const float* s = src + b * bh * bw;
    float* d = dst + b * bh * bw;
    float v[8][8];
    for (int r = 0; r < bh; ++r)
        for (int c = 0; c < bw; ++c) v[r][c] = s[r * bw + c];
    if (bh == 8 && bw == 8) {
        if (!inverse) {
            for (int r = 0; r < 8; ++r) dct8x8_row_fwd(v[r]);
            for (int c = 0; c < 8; ++c) dct8x8_col_fwd(v[0][c], v[1][c], v[2][c], v[3][c], v[4][c], v[5][c], v[6][c], v[7][c]);
        } else {
            for (int r = 0; r < 8; ++r) {
                for (int c = 0; c < 8; ++c) v[r][c] = __fmul_rn(v[r][c], dct8_rowscale(r));
                dct8x8_row_inv(v[r]);
            }
            for (int c = 0; c < 8; ++c) dct8x8_col_inv(v[0][c], v[1][c], v[2][c], v[3][c], v[4][c], v[5][c], v[6][c], v[7][c]);
        }
    } else {
        for (int r = 0; r < bh; ++r) dct1d(&v[r][0], bw, 1, inverse != 0);
        for (int c = 0; c < bw; ++c) dct1d(&v[0][c], bh, 8, inverse != 0);
    }
    for (int r = 0; r < bh; ++r)
        for (int c = 0; c < bw; ++c) d[r * bw + c] = v[r][c];
}

}  // namespace dvc
