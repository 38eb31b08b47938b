// dvc_b200.cu -- host side of the C ABI declared in include/dvc_b200.h: per-stream state, the batch
// loop (kernel sequencing for both loop flavours), the double-buffered host pipeline, and the
// stage-level entry points.  Kernels live in the k_*.cuh headers next to this file.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "../../include/dvc_b200.h"
#include "k_ccl.cuh"
#include "k_ccl_sweep.cuh"
#include "k_degrade.cuh"
#include "k_degrade4p.cuh"
#include "k_flow.cuh"
#include "k_front.cuh"
#include "k_mask.cuh"

using namespace dvc;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int set_err(char* dst, int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    if (dst) { strncpy(dst, g_err, 511); dst[511] = 0; }
    return code;
}

#define CU(expr)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (expr);                                                                         \
        if (e_ != cudaSuccess)                                                                           \
            return set_err(ERRBUF, e_ == cudaErrorMemoryAllocation ? DVC_ERR_NOMEM : DVC_ERR_CUDA,       \
                           "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__);  \
    } while (0)
#define CHECK_LAUNCH() CU(cudaGetLastError())

static inline unsigned cdiv(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

static int pack_to_bits(const uint8_t* src, uint32_t* dst, int n, int H, int W, cudaStream_t st);
static int unpack_from_bits(const uint32_t* src, uint8_t* dst, int n, int H, int W, cudaStream_t st);

// ------------------------------------------------------------------------------------------------
// structuring elements -> MorphChain
// ------------------------------------------------------------------------------------------------
// Row runs of np.ones((k,k)) or cv2.getStructuringElement(MORPH_ELLIPSE,(k,k)) relative to the default
// anchor (k/2, k/2).  The ellipse restates OpenCV's morph code: row i spans |dx| <= rint(c*sqrt(r^2-dy^2)/r).
static bool make_prim(int shape, int k, bool erode, MorphPrim& p) {
    if (k < 1 || k > MORPH_MAX_K) return false;
    memset(&p, 0, sizeof(p));
    p.erode = erode;
    const int a = k / 2;
    int n = 0;
    for (int i = 0; i < k; ++i) {
        int j1 = 0, j2 = k;
        if (shape == DVC_SHAPE_ELLIPSE) {
            const int r = k / 2, c = k / 2;
            const double inv_r2 = r ? 1.0 / ((double)r * r) : 0.0;
            const int dy = i - r;
            j1 = j2 = 0;
            if (std::abs(dy) <= r) {
                const int dx = (int)std::nearbyint(c * std::sqrt((r * r - dy * dy) * inv_r2));
                j1 = std::max(c - dx, 0);
                j2 = std::min(c + dx + 1, k);
            }
        }
        if (j2 <= j1) continue;
        p.dy[n] = (int8_t)(i - a);
        p.lo[n] = (int8_t)(j1 - a);
        p.hi[n] = (int8_t)(j2 - 1 - a);
        ++n;
    }
    p.nrows = (int8_t)n;
    if (n == 0) return false;
    bool sep = true;
    for (int i = 1; i < n; ++i)
        if (p.lo[i] != p.lo[0] || p.hi[i] != p.hi[0] || p.dy[i] != p.dy[i - 1] + 1) sep = false;
    p.separable = sep;
    // 3x3-bounded, non-separable elements get the unrolled path
    bool small = !sep;
    for (int i = 0; i < n; ++i)
        if (p.dy[i] < -1 || p.dy[i] > 1 || p.lo[i] < -1 || p.hi[i] > 1 || p.lo[i] > 0 || p.hi[i] < 0) small = false;
    p.small = small;
    if (small)
        for (int i = 0; i < n; ++i)
            p.small_rows[p.dy[i] + 1] = (int8_t)(1 | (p.lo[i] == -1 ? 2 : 0) | (p.hi[i] == 1 ? 4 : 0));
    // kernels specialised at compile time (k_mask.cuh: rect_pass<K>, small_pass<FU,FM,FD>)
    p.kind = 0;
    if (sep && shape == DVC_SHAPE_RECT && (k & 1) && k >= 3) p.kind = (int16_t)(100 + k);      // every odd k up to MORPH_MAX_K
    if (small && p.small_rows[0] == 1 && p.small_rows[1] == 3 && p.small_rows[2] == 0) p.kind = 1;
    if (small && p.small_rows[0] == 1 && p.small_rows[1] == 7 && p.small_rows[2] == 1) p.kind = 2;
    return true;
}

static bool chain_push(MorphChain& ch, int op, int shape, int k) {
    auto push = [&](bool erode) {
        // Two consecutive odd rectangles of the same polarity are one rectangle: the Minkowski sum (k1 + k2 - 1), which is
        // exact with cv2's "ignore what is outside the image" borders because the intermediate pixel of any two-step path
        // lies between its end points, inside the image.  CLOSE, OPEN, DILATE with one k x k element (BASELINE config 3)
        // is D E E D D = D(k) E(2k-1) D(2k-1): three passes instead of five, and a pass costs the same for any k.
        if (ch.n > 0 && shape == DVC_SHAPE_RECT && (k & 1) && k >= 3) {
            MorphPrim& q = ch.p[ch.n - 1];
            const int kq = q.kind - 100;
            if (q.kind >= 103 && (bool)q.erode == erode && kq + k - 1 <= MORPH_MAX_K) {
                if (!make_prim(DVC_SHAPE_RECT, kq + k - 1, erode, q)) return false;
                ch.halo_top += k / 2;
                ch.halo_bot += k / 2;
                ch.pad = std::max<int>(ch.pad, (kq + k - 1) / 2);
                return true;
            }
        }
        // Likewise MORPH_ELLIPSE (2, 2) twice (the E E in the middle of CLOSE, OPEN): one pass with the summed element (kind 3)
        if (ch.n > 0 && shape == DVC_SHAPE_ELLIPSE && k == 2) {
            MorphPrim& q = ch.p[ch.n - 1];
            if (q.kind == 1 && (bool)q.erode == erode) {
                q.kind = 3;
                ch.halo_top += 1;           // the element reaches one more row up; nothing below the anchor
                return true;
            }
        }
        if (ch.n >= MORPH_MAX_PRIMS) return false;
        MorphPrim& p = ch.p[ch.n];
        if (!make_prim(shape, k, erode, p)) return false;
        ch.halo_top += -std::min<int>(p.dy[0], 0);
        ch.halo_bot += std::max<int>(p.dy[p.nrows - 1], 0);
        if (p.kind >= 100) ch.pad = std::max<int>(ch.pad, (p.kind - 100) / 2);       // rect_pass<K> reads K / 2 rows beyond its run
        ++ch.n;
        return true;
    };
    switch (op) {
        case DVC_MORPH_ERODE: return push(true);
        case DVC_MORPH_DILATE: return push(false);
        case DVC_MORPH_OPEN: return push(true) && push(false);
        case DVC_MORPH_CLOSE: return push(false) && push(true);
    }
    return false;
}

// python: smallest c with c*255 >= alpha*L*255, evaluated in doubles exactly as motion_compression_opt.py:86
static void window_min_counts(double alpha, int K, MinCounts& mc) {
    memset(&mc, 0, sizeof(mc));
    for (int L = 1; L <= K; ++L) {
        const double rhs = alpha * L * 255;
        int c = 0;
        while (!((double)(c * 255) >= rhs) && c <= L) ++c;
        mc.v[L - 1] = (uint8_t)std::min(c, 255);
    }
}

// ------------------------------------------------------------------------------------------------
// launch helpers (all asynchronous on `st`)
// ------------------------------------------------------------------------------------------------
// Function attributes and __constant__ uploads are per device: one-time set-up is tracked per CUDA device ordinal so that
// handles on several GPUs in one process all get it.
// Measurement switches (kernel generations, band and chunk sizes, copy-only probes: DESIGN.md section 6a) exist only in the
// -DDVC_MEASURE flavour of the library that tools/ build for A/B runs.  The product build ignores the environment, so a
// stray variable can never change what the loop computes.
#ifdef DVC_MEASURE
static int measure_env(const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; }
#else
static constexpr int measure_env(const char*, int dflt) { return dflt; }
#endif

struct PerDeviceOnce {
    std::mutex mu;
    bool done[64] = {};
    struct Guard {
        PerDeviceOnce* o; int d;
        explicit operator bool() const { return o != nullptr; }
        void commit() { o->done[d] = true; }              // not reached when the set-up bails out: it is retried next time
        ~Guard() { if (o) o->mu.unlock(); }
    };
    // `if (auto g = once.begin()) { set-up; g.commit(); }`: the lock is held while the first caller sets up, so a second thread
    // cannot launch before the attributes / tables are in place
    Guard begin() {
        int d = 0;
        cudaGetDevice(&d);
        d &= 63;
        mu.lock();
        if (done[d]) { mu.unlock(); return Guard{nullptr, d}; }
        return Guard{this, d};
    }
};

static int g_morph_smem_limit = 0;
static PerDeviceOnce g_morph_once;

static int launch_morph_chain(char* ERRBUF, const uint32_t* src, uint32_t* dst, int n, int H, int W,
                              const MorphChain& ch, cudaStream_t st) {
    const int wpr = words_per_row(W);
    if (ch.n == 0) {
        if (src != dst) CU(cudaMemcpyAsync(dst, src, (size_t)n * H * wpr * 4, cudaMemcpyDeviceToDevice, st));
        return DVC_OK;
    }
    if (auto once = g_morph_once.begin()) {
        int dev = 0, lim = 0;
        CU(cudaGetDevice(&dev));
        CU(cudaDeviceGetAttribute(&lim, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        CU(cudaFuncSetAttribute(k_morph_chain<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CU(cudaFuncSetAttribute(k_morph_chain<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        g_morph_smem_limit = lim;
        once.commit();
    }
    const int halo = ch.halo_top + ch.halo_bot;
    for (int i = 0; i < ch.n; ++i)
        for (int k = 0; k < ch.p[i].nrows; ++k)
            if (ch.p[i].lo[k] > 0 || ch.p[i].hi[k] < 0)
                return set_err(ERRBUF, DVC_ERR_UNSUPPORTED, "structuring element row that does not span its anchor column");
    if (wpr > 256) return set_err(ERRBUF, DVC_ERR_UNSUPPORTED, "frames wider than 8192 pixels are not supported by the morphology kernel");
    // Band height: ~36 KB of shared memory per CTA (two planes) keeps ~6 CTAs of 256 threads resident per SM.  Chains with a
    // large halo (BASELINE config 3: five 15x15 primitives = 35 rows on each side) would recompute most of such a band, so
    // they take the whole shared memory of an SM for one band (halo rows under ~40 % of the staged rows) and make up the
    // occupancy with 1024 threads in that one CTA.
    const size_t row_bytes = 2 * (size_t)wpr * 4;
    const size_t limit = (size_t)g_morph_smem_limit - 64;
    static const int target_kb = std::max(4, measure_env("DVC_MORPH_SMEM_KB", 36));
    const int pad = 2 * ch.pad;                          // zero rows above and below each staged plane (not counted in the target)
    int band = (int)((size_t)target_kb * 1024 / row_bytes) - halo;
    if (band < 2 * halo) band = (int)(limit / row_bytes) - halo - pad;
    band = std::max(band, 16);
    band = std::min<int>(band, (int)(limit / row_bytes) - halo - pad);
    if (band < 1) return set_err(ERRBUF, DVC_ERR_UNSUPPORTED, "morphology chain halo %d rows x %d words does not fit in shared memory", halo, wpr);
    band = std::min(band, H);
    const int nbands = (H + band - 1) / band;
    band = (H + nbands - 1) / nbands;
    const size_t smem = 2 * (size_t)(band + halo + pad) * wpr * 4 + 16;
    const int threads = smem > 110 * 1024 ? 1024 : smem > 72 * 1024 ? 512 : 256;     // CTAs per SM: 1, 2, 3+
    dim3 grid(nbands, n);
    if (threads == 256) k_morph_chain<256><<<grid, 256, smem, st>>>(src, dst, H, W, wpr, band, ch);
    else k_morph_chain<1024><<<grid, threads, smem, st>>>(src, dst, H, W, wpr, band, ch);
    CHECK_LAUNCH();
    return DVC_OK;
}

struct CclScratch {
    // first generation (k_ccl.cuh; frames wider than 8192 pixels and the measure flavour's A/B switch): union-find storage per
    // frame, dense slot-0 arrays [plane_words + 1] and overflow arrays [plane_words * 15], for the phase A parents, the phase B
    // parents and the phase B areas
    int *pa0 = nullptr, *paov = nullptr, *pb0 = nullptr, *pbov = nullptr, *ar0 = nullptr, *arov = nullptr;
    uint8_t* rowflag = nullptr;   // [frames][H]: the row holds foreground (written by the first kernel, read by the other six)
    uint32_t* filled = nullptr;  // [frames] planes: F of the first generation
    // sweep kernel (k_ccl_sweep.cuh): node arrays of frames with more than SW_CAP row runs, [frames][g_stride] each
    int *gp = nullptr, *ga = nullptr;
    size_t g_stride = 0;
    bool sweep = false;
    int frames = 0;
};

static PerDeviceOnce g_sweep_once;
static int g_sweep_smem_limit = 0;

// the sweep kernel takes rows of up to 4 x 2048 pixels and needs (H + 1) row bases in shared memory
static bool ccl_sweep_usable(int H, int W) {
    static const bool on = measure_env("DVC_CCL_SWEEP", 1) != 0;
    return on && W <= 8192 && ccl_sweep_smem_bytes(H, W) <= 200 * 1024;
}

static int launch_contour_sweep(char* ERRBUF, const uint32_t* raw, uint32_t* out, int n, int H, int W, int thr,
                                const CclScratch& sc, cudaStream_t st) {
    if (auto once = g_sweep_once.begin()) {
        int dev = 0, lim = 0;
        CU(cudaGetDevice(&dev));
        CU(cudaDeviceGetAttribute(&lim, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        CU(cudaFuncSetAttribute(k_ccl_sweep<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim - 1024));
        CU(cudaFuncSetAttribute(k_ccl_sweep<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim - 1024));
        CU(cudaFuncSetAttribute(k_ccl_sweep<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim - 1024));
        g_sweep_smem_limit = lim;
        once.commit();
    }
    const int wpr = words_per_row(W);
    const size_t pw = (size_t)H * wpr, smem = ccl_sweep_smem_bytes(H, W);
    static const int chunk_rows = std::max(1, measure_env("DVC_CCL_ROWS", 16));     // consecutive rows a warp sweeps in one go
    if (smem + 2048 > (size_t)g_sweep_smem_limit) return set_err(ERRBUF, DVC_ERR_UNSUPPORTED, "contour filter: %d rows do not fit in shared memory", H);
    for (int i0 = 0; i0 < n; i0 += sc.frames) {
        const int m = std::min(sc.frames, n - i0);
        const uint32_t* r = raw + (size_t)i0 * pw;
        uint32_t* o = out + (size_t)i0 * pw;
        if (W <= 2048) k_ccl_sweep<1><<<m, SW_THREADS, smem, st>>>(r, o, sc.gp, sc.ga, sc.g_stride, H, W, wpr, thr, chunk_rows);
        else if (W <= 4096) k_ccl_sweep<2><<<m, SW_THREADS, smem, st>>>(r, o, sc.gp, sc.ga, sc.g_stride, H, W, wpr, thr, chunk_rows);
        else k_ccl_sweep<4><<<m, SW_THREADS, smem, st>>>(r, o, sc.gp, sc.ga, sc.g_stride, H, W, wpr, thr, chunk_rows);
        CHECK_LAUNCH();
    }
    return DVC_OK;
}

static int launch_contour_filter(char* ERRBUF, const uint32_t* raw, uint32_t* out, int n, int H, int W,
                                 double min_area, const CclScratch& sc, cudaStream_t st) {
    const int wpr = words_per_row(W);
    const size_t pw = (size_t)H * wpr;
    const double t2 = std::floor(2.0 * min_area);
    const int thr = t2 >= 2147483647.0 ? 2147483647 : (t2 < -1.0 ? -1 : (int)t2);
    if (sc.sweep) return launch_contour_sweep(ERRBUF, raw, out, n, H, W, thr, sc, st);
    for (int i0 = 0; i0 < n; i0 += sc.frames) {
        const int m = std::min(sc.frames, n - i0);
        dim3 grid(cdiv(pw, 256), m);
        dim3 grow((H + 7) / 8, m);
        const uint32_t* r = raw + (size_t)i0 * pw;
        static const bool row_skip = measure_env("DVC_CCL_ROWSKIP", 1) != 0;
        uint8_t* rf = row_skip ? sc.rowflag : nullptr;
        k_ccl_rowlink<true, true><<<grow, 256, 0, st>>>(r, sc.pa0, sc.paov, nullptr, nullptr, H, W, wpr, rf);
        const dim3 gpos = CCL_GRID(wpr, H, m);
        k_ccl_union<true, 4><<<gpos, 256, 0, st>>>(r, sc.pa0, sc.paov, H, W, wpr, rf);
        k_ccl_fill<<<gpos, 256, 0, st>>>(r, sc.pa0, sc.paov, sc.filled, H, W, wpr, rf);
        k_ccl_rowlink<false, false><<<grow, 256, 0, st>>>(sc.filled, sc.pb0, sc.pbov, sc.ar0, sc.arov, H, W, wpr, rf);
        k_ccl_union<false, 8><<<gpos, 256, 0, st>>>(sc.filled, sc.pb0, sc.pbov, H, W, wpr, rf);
        k_ccl_area<<<gpos, 256, 0, st>>>(sc.filled, sc.pb0, sc.pbov, sc.ar0, sc.arov, H, W, wpr, rf);
        k_ccl_select<<<gpos, 256, 0, st>>>(sc.filled, sc.pb0, sc.pbov, sc.ar0, sc.arov, out + (size_t)i0 * pw, H, W, wpr, thr, rf);
        CHECK_LAUNCH();
    }
    return DVC_OK;
}

static size_t ccl_dense_ints(int H, int W) { return (size_t)H * words_per_row(W) + 1; }
static size_t ccl_overflow_ints(int H, int W) { return (size_t)H * words_per_row(W) * 15; }

// A dense + overflow pair shares one allocation (uf_addr reaches the overflow part through a 32-bit offset from the dense one).
static int ccl_scratch_alloc(char* ERRBUF, CclScratch& sc, int frames, int H, int W) {
    const size_t pw = (size_t)H * words_per_row(W);
    sc.frames = frames;
    sc.sweep = ccl_sweep_usable(H, W);
    if (!sc.sweep) CU(cudaMalloc(&sc.filled, pw * 4 * frames));
    if (sc.sweep) {
        sc.g_stride = ccl_sweep_max_nodes(H, W);
        if (sc.g_stride >= 0x7fffffffull) return set_err(ERRBUF, DVC_ERR_UNSUPPORTED, "contour filter scratch exceeds 2^31 nodes");
        CU(cudaMalloc(&sc.gp, sc.g_stride * sizeof(int) * frames));
        CU(cudaMalloc(&sc.ga, sc.g_stride * sizeof(int) * frames));
        return DVC_OK;
    }
    const size_t d = ccl_dense_ints(H, W) * sizeof(int) * frames, o = ccl_overflow_ints(H, W) * sizeof(int) * frames;
    if ((d + o) / sizeof(int) >= 0x7fffffffull) return set_err(ERRBUF, DVC_ERR_UNSUPPORTED, "contour filter scratch exceeds 2^31 nodes");
    CU(cudaMalloc(&sc.pa0, d + o)); sc.paov = sc.pa0 + d / sizeof(int);
    CU(cudaMalloc(&sc.pb0, d + o)); sc.pbov = sc.pb0 + d / sizeof(int);
    CU(cudaMalloc(&sc.ar0, d + o)); sc.arov = sc.ar0 + d / sizeof(int);
    CU(cudaMalloc(&sc.rowflag, (size_t)frames * H));
    return DVC_OK;
}
static void ccl_scratch_free(CclScratch& sc) {
    cudaFree(sc.pa0); cudaFree(sc.pb0); cudaFree(sc.ar0);
    cudaFree(sc.filled); cudaFree(sc.rowflag);
    cudaFree(sc.gp); cudaFree(sc.ga);
    sc = CclScratch();
}

// ------------------------------------------------------------------------------------------------
// cv2.resize INTER_LINEAR tables (OpenCV resize(): scale = 1 / ((double)dst / src); fx = (float)((d + 0.5) * scale - 0.5);
// sx = floor(fx); fx -= sx; columns clamp (sx, fx) at the image border, rows keep fx and clip the row index instead;
// coefficients = cvRound(float * 2048))
// ------------------------------------------------------------------------------------------------
struct ResizeHostTables { std::vector<int> xofs, yofs; std::vector<short> xa, yb; };
static void make_resize_tables(int sH, int sW, int dH, int dW, ResizeHostTables& t) {
    auto fill = [](int sn, int dn, bool clamp, std::vector<int>& ofs, std::vector<short>& co) {
        ofs.resize(dn); co.resize(2 * (size_t)dn);
        const double inv = (double)dn / sn, scale = 1.0 / inv;
        for (int d = 0; d < dn; ++d) {
            float f = (float)((d + 0.5) * scale - 0.5);
            int i = (int)std::floor(f);
            f -= (float)i;
            if (clamp) {
                if (i < 0) { i = 0; f = 0.0f; }
                if (i >= sn - 1) { i = sn - 1; f = 0.0f; }
            }
            ofs[d] = i;
            co[2 * d] = (short)lrintf((1.0f - f) * 2048.0f);
            co[2 * d + 1] = (short)lrintf(f * 2048.0f);
        }
    };
    fill(sW, dW, true, t.xofs, t.xa);
    fill(sH, dH, false, t.yofs, t.yb);
}
// device copy of the tables in one allocation: [xofs dW ints][yofs dH ints][xa dW short2][yb dH short2]
static size_t resize_tables_bytes(int dH, int dW) { return (size_t)(dW + dH) * (sizeof(int) + sizeof(short2)); }
static ResizeTables resize_tables_view(void* dev, int dH, int dW) {
    ResizeTables v;
    char* p = (char*)dev;
    v.xofs = (const int*)p; p += (size_t)dW * sizeof(int);
    v.yofs = (const int*)p; p += (size_t)dH * sizeof(int);
    v.xa = (const short2*)p; p += (size_t)dW * sizeof(short2);
    v.yb = (const short2*)p;
    return v;
}
static void resize_tables_pack(const ResizeHostTables& t, int dH, int dW, std::vector<char>& blob) {
    blob.resize(resize_tables_bytes(dH, dW));
    char* p = blob.data();
    memcpy(p, t.xofs.data(), (size_t)dW * sizeof(int)); p += (size_t)dW * sizeof(int);
    memcpy(p, t.yofs.data(), (size_t)dH * sizeof(int)); p += (size_t)dH * sizeof(int);
    memcpy(p, t.xa.data(), (size_t)dW * sizeof(short2)); p += (size_t)dW * sizeof(short2);
    memcpy(p, t.yb.data(), (size_t)dH * sizeof(short2));
}
static int launch_resize(char* ERRBUF, const uint8_t* src, uint8_t* dst, int n, int sH, int sW, int dH, int dW, int cn,
                         const ResizeTables& t, cudaStream_t st) {
    dim3 grid(cdiv((size_t)dW * dH, 256), n);
    if (cn == 3) k_resize_linear<3><<<grid, 256, 0, st>>>(src, dst, sH, sW, dH, dW, t);
    else if (cn == 1) k_resize_linear<1><<<grid, 256, 0, st>>>(src, dst, sH, sW, dH, dW, t);
    else return set_err(ERRBUF, DVC_ERR_UNSUPPORTED, "resize: %d channels (1 or 3 supported)", cn);
    CHECK_LAUNCH();
    return DVC_OK;
}

// OpenCV's fixed-point Gaussian kernel for uint8 images (getGaussianKernelBitExact + getGaussianKernelFixedPoint_ED):
// the double-precision kernel, normalised to sum 1, is rounded to 8 fractional bits from the ends towards the middle
// with the rounding error carried along, so the taps sum to exactly 256.  sigma <= 0 uses cv2's rule (and its table of
// small kernels for ksize <= 7).
static bool gaussian_taps_fixed(int n, double sigma, GaussTaps& tp) {
    if (n < 1 || n > 33 || !(n & 1)) return false;
    tp.n = n;
    double k[33];
    static const double small_tab[4][7] = {{1.0}, {0.25, 0.5, 0.25}, {0.0625, 0.25, 0.375, 0.25, 0.0625},
                                           {0.03125, 0.109375, 0.21875, 0.28125, 0.21875, 0.109375, 0.03125}};
    if (sigma <= 0 && n <= 7) {
        for (int i = 0; i < n; ++i) k[i] = small_tab[n >> 1][i];
    } else {
        const double sg = sigma > 0 ? sigma : ((n - 1) * 0.5 - 1) * 0.3 + 0.8;
        const double scale2x = -0.5 / (sg * sg), c = (n - 1) * 0.5;
        double sum = 0;
        for (int i = 0; i < n; ++i) { k[i] = std::exp(scale2x * (i - c) * (i - c)); sum += k[i]; }
        for (int i = 0; i < n; ++i) k[i] /= sum;
    }
    double err = 0;
    const int h = n / 2;
    for (int i = 0; i < h; ++i) {
        const double adj = k[i] * 256.0 + err;
        const double v = std::nearbyint(adj);
        err = adj - v;
        tp.k[i] = tp.k[n - 1 - i] = (uint16_t)v;
    }
    tp.k[h] = (uint16_t)std::nearbyint(k[h] * 256.0 + err);
    return true;
}

static int launch_gaussian(char* ERRBUF, const uint8_t* src, uint8_t* dst, uint16_t* tmp, int n, int H, int W, int ksize, double sigma,
                           cudaStream_t st) {
    GaussTaps tp;
    if (!gaussian_taps_fixed(ksize, sigma, tp))
        return set_err(ERRBUF, DVC_ERR_UNSUPPORTED, "GaussianBlur ksize %d: odd sizes 1..33 are implemented", ksize);
    dim3 grid(cdiv((size_t)H * W, 256), n);
    k_gauss_h<<<grid, 256, 0, st>>>(src, tmp, H, W, tp);
    k_gauss_v<<<grid, 256, 0, st>>>(tmp, dst, H, W, tp);
    CHECK_LAUNCH();
    return DVC_OK;
}

// partial blocks at the right / bottom edge of frames whose size is not a multiple of the block size
static int launch_degrade_edges(char* ERRBUF, const uint8_t* frames, const uint32_t* over127, const uint32_t* nonzero,
                                uint8_t* compressed, uint8_t* overlay, int n, int H, int W, int bs, float q, int flavour,
                                Counters* counters, cudaStream_t st, bool all_blocks = false) {
    if (!all_blocks && H % bs == 0 && W % bs == 0) return DVC_OK;
    const int n_edge = all_blocks ? ((W + bs - 1) / bs) * ((H + bs - 1) / bs) : (W % bs ? (H + bs - 1) / bs : 0) + (H % bs ? W / bs : 0);
    dim3 grid(cdiv(n_edge, 64), n);
    const int wpr = words_per_row(W);
    if (flavour == DVC_DEGRADE_FD) k_degrade_edges<0><<<grid, 64, 0, st>>>(frames, over127, nonzero, compressed, overlay, H, W, wpr, bs, q, counters, all_blocks);
    else k_degrade_edges<1><<<grid, 64, 0, st>>>(frames, over127, nonzero, compressed, overlay, H, W, wpr, bs, q, counters, all_blocks);
    CHECK_LAUNCH();
    return DVC_OK;
}

// The kernel that degrades the whole blocks of a frame (partial blocks at the right / bottom edge: launch_degrade_edges).
// `addr_bits` is the OR of the frame and output addresses.  4x4 blocks are FD only (MCO takes 8x8, checked by the caller).
enum class DegradeKernel { edges, ring4, packed4, generic4, packed8, generic8 };

static DegradeKernel degrade_kernel(int bs, int H, int W, float q, uintptr_t addr_bits) {
    if (bs != 4 && bs != 8) return DegradeKernel::edges;      // rare block sizes: every block through the exact general path
    // packed kernels (k_degrade4p.cuh): 8-byte vector access, Markstein quotient (exact for q in [0.01, 1e6]); otherwise the
    // one-thread-per-block kernels, bytewise and with the IEEE division
    const bool packed = W % 8 == 0 && q >= 0.01f && q <= 1.0e6f && addr_bits % 8 == 0;
    if (bs == 8) return packed ? DegradeKernel::packed8 : DegradeKernel::generic8;
    if (!packed) return DegradeKernel::generic4;
    // the ring's bulk copies need every frame of the batch 16-byte aligned, and 16-byte row pieces when a block row is split
    // over several tiles (W > 2048)
    const bool ring = addr_bits % 16 == 0 && (size_t)H * W * 3 % 16 == 0 && (W / 8 <= 256 || W % 16 == 0);
    return ring ? DegradeKernel::ring4 : DegradeKernel::packed4;
}

// Tiles and shared-memory ring of k_degrade4s for n frames, and the dynamic shared memory it needs; false if that does not fit.
static bool k4_ring_geometry(int n, int H, int W, K4SGeom& sg, size_t& smem) {
    const int wpr = words_per_row(W), gpr = W / 8, nbr = H / 4;
    K4Geom& g = sg.g;
    if (gpr <= 256) {
        g.parts = 1; g.gp = gpr; g.nb = std::max(1, std::min(nbr, std::min(256 / gpr, 256 / wpr))); g.sp = W * 3;
        g.span_bytes = g.nb * 4 * W * 3;
    } else {
        g.parts = (gpr + 255) / 256;
        g.gp = (((gpr + g.parts - 1) / g.parts) + 15) & ~15;
        g.parts = (gpr + g.gp - 1) / g.gp;
        g.nb = 1; g.sp = g.gp * 24; g.span_bytes = 4 * g.sp;
    }
    g.mask_bytes = 4 * g.nb * wpr * 4;
    sg.tiles_per_frame = g.parts == 1 ? (int)cdiv(nbr, g.nb) : nbr * g.parts;
    sg.n_tiles = sg.tiles_per_frame * n;
    sg.stage_bytes = (g.span_bytes + 2 * g.mask_bytes + 127) & ~127;
    sg.ybuf_bytes = (g.span_bytes + 127) & ~127;
    const size_t smem_cap = 224 * 1024;
    auto smem_need = [&](int stages) {
        return (size_t)stages * sg.stage_bytes + (size_t)K4S_GROUPS * sg.ybuf_bytes + 8 * (2 * stages) + 16 + 16 * stages;
    };
    int S = 6;
    while (smem_need(S) > smem_cap && S > 2) --S;
    sg.stages = S;
    smem = smem_need(S);
    // A group hands a stage back only while it works on its next tile, so every group needs a second stage to move on to:
    // with stages <= groups the ring would wait on itself.
    return S > K4S_GROUPS && smem <= smem_cap;
}

static int launch_degrade(char* ERRBUF, const uint8_t* frames, const uint32_t* over127, const uint32_t* nonzero,
                          uint8_t* compressed, uint8_t* overlay, int n, int H, int W, int bs, float q, int flavour,
                          Counters* counters, cudaStream_t st) {
    if (bs < 1 || bs > 8)
        return set_err(ERRBUF, DVC_ERR_UNSUPPORTED, "block_size %d: the GPU path implements 1..8 (cv2's DCT routines for longer blocks are not restated)", bs);
    if (flavour == DVC_DEGRADE_MCO && bs != 8) return set_err(ERRBUF, DVC_ERR_INVALID, "MCO flavour uses 8x8 blocks");
    if (!(q > 0.0f)) return set_err(ERRBUF, DVC_ERR_INVALID, "quantization_level must be > 0");
    if (n <= 0) return DVC_OK;

    const DegradeKernel kern = degrade_kernel(bs, H, W, q, (uintptr_t)frames | (uintptr_t)compressed | (uintptr_t)overlay);
    if (kern == DegradeKernel::edges)
        return launch_degrade_edges(ERRBUF, frames, over127, nonzero, compressed, overlay, n, H, W, bs, q, flavour, counters, st, true);
    if (H % bs || W % bs) {
        // full blocks by the kernels below (they floor H and W to whole blocks), partial edge blocks by a small second launch
        int rc = launch_degrade_edges(ERRBUF, frames, over127, nonzero, compressed, overlay, n, H, W, bs, q, flavour, counters, st);
        if (rc) return rc;
        if (H < bs || W < bs) return DVC_OK;
    }

    static PerDeviceOnce attr_once;
    if (auto once = attr_once.begin()) {
        CU(cudaFuncSetAttribute(k_degrade4s, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        CU(cudaFuncSetAttribute(k_degrade8<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, k8_smem_bytes<0>()));
        CU(cudaFuncSetAttribute(k_degrade8<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, k8_smem_bytes<1>()));
        once.commit();
    }
    const int wpr = words_per_row(W);
    const bool fd = flavour == DVC_DEGRADE_FD;
    // quotient constants of the packed kernels; the 4x4 ones carry the DCT butterflies' folded power-of-two scalings
    QuantP qp;
    for (int ne = 0; ne < 3; ++ne) {
        const float scale = bs == 4 ? (float)(1 << ne) : 1.0f;
        qp.rcp[ne] = 1.0f / (q * scale);
        qp.nqs[ne] = -(q * scale);
        qp.o[ne] = q / scale;
    }
    const dim3 grid_generic(cdiv((size_t)(W / bs) * (H / bs), 128), n);
    switch (kern) {
        case DegradeKernel::ring4: {
            K4SGeom sg;
            size_t smem = 0;
            if (!k4_ring_geometry(n, H, W, sg, smem))
                return set_err(ERRBUF, DVC_ERR_UNSUPPORTED, "K4 ring: %d stages for %d consumer groups do not fit (%zu bytes of shared memory)",
                               sg.stages, K4S_GROUPS, smem);
            int dev = 0, sms = 0;
            CU(cudaGetDevice(&dev));
            CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
            k_degrade4s<<<(unsigned)std::min(sg.n_tiles, sms), K4S_THREADS, smem, st>>>(frames, over127, nonzero, compressed, overlay,
                                                                                        H, W, wpr, qp, counters, sg);
            break;
        }
        case DegradeKernel::packed4:
            k_degrade4p<<<dim3(cdiv((size_t)(W / 8) * (H / 4), 256), n), 256, 0, st>>>(frames, over127, nonzero, compressed, overlay,
                                                                                        H, W, wpr, qp, counters);
            break;
        case DegradeKernel::generic4:
            k_degrade_generic<4, 0><<<grid_generic, 128, 0, st>>>(frames, over127, nonzero, compressed, overlay, H, W, wpr, q, counters);
            break;
        case DegradeKernel::packed8: {
            const dim3 g8(cdiv((size_t)(W / 8) * (H / 8), K8_THREADS), n);
            if (fd) k_degrade8<0><<<g8, K8_THREADS, k8_smem_bytes<0>(), st>>>(frames, over127, nonzero, compressed, overlay, H, W, wpr, qp, counters);
            else k_degrade8<1><<<g8, K8_THREADS, k8_smem_bytes<1>(), st>>>(frames, over127, nonzero, compressed, overlay, H, W, wpr, qp, counters);
            break;
        }
        case DegradeKernel::generic8:
            if (fd) k_degrade_generic<8, 0><<<grid_generic, 128, 0, st>>>(frames, over127, nonzero, compressed, overlay, H, W, wpr, q, counters);
            else k_degrade_generic<8, 1><<<grid_generic, 128, 0, st>>>(frames, over127, nonzero, compressed, overlay, H, W, wpr, q, counters);
            break;
        case DegradeKernel::edges:
            break;
    }
    CHECK_LAUNCH();
    return DVC_OK;
}

// ------------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------------
struct ProfRec { int kid; int launches; cudaEvent_t a, b; };

struct dvc_handle {
    dvc_config cfg;
    int H, W, wpr;
    int S;                        // streams of this handle (cfg.n_streams, >= 1): a lock-step group shares every launch
    size_t plane_words, plane_bytes, frame_bytes;
    bool aligned;                 // W % 16 == 0: vector paths
    long long n_masks;            // masks produced so far in this stream
    int seg_len;
    int gray_impl;                // DVC_GRAY_IMPL: 0 = PRMT + IMAD, 1 = IDP.4A, 2 = IDP.2A (default) gray conversion in K1
    // state
    uint8_t* prev_gray[2];
    int cur;
    uint8_t* acc;                 // FD: accumulated_mask
    uint32_t* ring;               // WINDOW: raw-mask ring, ring_cap planes
    int ring_cap;
    MinCounts min_counts;
    // scratch (max_batch planes each)
    uint32_t* bits[2][3];         // two sets (software pipelining across batches) of three bit-plane arrays
    uint8_t* blurred;             // FD: [max_batch] gray planes
    CclScratch ccl;
    MorphChain chain;
    Counters* counters_dev;
    dvc_counters counters_host;   // frames / pixels / blocks are counted on the host
    // two-stream software pipeline: mask kernels of batch c+1 overlap the degrade kernel of batch c
    bool overlap;                 // dvc_set_overlap: applies to dvc_process_batch (dvc_process_host always pipelines)
    int pp;                       // scratch set / event parity of the next batch
    cudaStream_t s_front, s_mask, s_k4;      // pipelined mode: front kernel | mask kernels | degrade kernel, each a batch apart
    cudaEvent_t ev_in, ev_front[2], ev_mask[2], ev_k4[2];
    bool ev_used[2];
    cudaEvent_t ev_user;          // end of the last batch issued on a caller's stream (strict-order mode)
    bool ev_user_used;
    // host pipeline
    cudaStream_t s_h2d, s_d2h;
    cudaEvent_t ev_h2d[2], ev_d2h[2];
    uint8_t *st_in[2], *st_ov[2], *st_cp[2], *st_mask[2];
    uint8_t* st_src[2];           // source-size upload buffers when the handle resizes (cfg.src_width / src_height)
    void* resize_tables;          // device copy of the cv2.resize tables
    bool resizing;
    size_t src_frame_bytes;
    bool staging;
    // profiling: CUDA events around each kernel group, on the launching stream
    bool prof;
    std::vector<ProfRec>* prof_recs;
    long long launches;           // kernels launched by the loop so far
    char err[512];
};

// Frames per stream in one chunk of dvc_process_host's copy pipeline: small enough that the first upload and the last
// download (the only copies nothing overlaps) are short against the PCIe-bound steady state, large enough for full-size
// kernels: about 8 frames per chunk over all streams of the handle.
static int host_chunk_frames(const dvc_handle* h) {
    const int total = std::max(1, measure_env("DVC_HOST_CHUNK", 8));
    return std::max(1, std::min(h->cfg.max_batch, (total + h->S - 1) / h->S));
}

static int alloc_staging(dvc_handle* h) {
    char* ERRBUF = h->err;
    if (h->staging) return DVC_OK;
    const size_t nst = (size_t)h->S * host_chunk_frames(h);
    const size_t fb = h->frame_bytes * nst;
    for (int b = 0; b < 2; ++b) {
        CU(cudaMalloc(&h->st_in[b], fb));
        CU(cudaMalloc(&h->st_ov[b], fb));
        CU(cudaMalloc(&h->st_cp[b], fb));
        CU(cudaMalloc(&h->st_mask[b], h->plane_bytes * nst));
        if (h->resizing) CU(cudaMalloc(&h->st_src[b], h->src_frame_bytes * nst));
        CU(cudaEventCreateWithFlags(&h->ev_h2d[b], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&h->ev_d2h[b], cudaEventDisableTiming));
    }
    CU(cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&h->s_d2h, cudaStreamNonBlocking));
    h->staging = true;
    return DVC_OK;
}

// Wait for everything this handle has in flight -- its own streams and the last batch issued on a caller's stream --
// without a device-wide synchronisation: handles of other streams on the same GPU keep running.
static cudaError_t handle_join(dvc_handle* h) {
    cudaError_t e;
    if (h->ev_user_used && (e = cudaEventSynchronize(h->ev_user)) != cudaSuccess) return e;
    if (h->s_front && (e = cudaStreamSynchronize(h->s_front)) != cudaSuccess) return e;
    if (h->s_mask && (e = cudaStreamSynchronize(h->s_mask)) != cudaSuccess) return e;
    if (h->s_k4 && (e = cudaStreamSynchronize(h->s_k4)) != cudaSuccess) return e;
    if (h->staging) {
        if ((e = cudaStreamSynchronize(h->s_h2d)) != cudaSuccess) return e;
        if ((e = cudaStreamSynchronize(h->s_d2h)) != cudaSuccess) return e;
    }
    return cudaSuccess;
}
// synchronous copies / fills on the handle's own stream (the legacy default stream would serialise all handles)
static cudaError_t h_copy(dvc_handle* h, void* dst, const void* src, size_t bytes, cudaMemcpyKind kind) {
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, kind, h->s_mask);
    return e != cudaSuccess ? e : cudaStreamSynchronize(h->s_mask);
}
static cudaError_t h_fill0(dvc_handle* h, void* dst, size_t bytes) {
    cudaError_t e = cudaMemsetAsync(dst, 0, bytes, h->s_mask);
    return e != cudaSuccess ? e : cudaStreamSynchronize(h->s_mask);
}

extern "C" int dvc_abi_version(void) { return DVC_ABI_VERSION; }
extern "C" int dvc_measure_build(void) {
#ifdef DVC_MEASURE
    return 1;
#else
    return 0;
#endif
}

extern "C" const char* dvc_last_error(const dvc_handle* h) { return h ? h->err : g_err; }

extern "C" void dvc_default_config(dvc_config* c) {
    memset(c, 0, sizeof(*c));
    c->mode = DVC_MODE_FD;
    c->block_size = 4;
    c->motion_threshold = 0.5f;
    c->min_area = 500.0;
    c->kernel_size = 7;
    c->release_factor = 0.5;
    c->quantization_level = 100.0f;
    c->window_size = 30;
    c->alpha_fraction = 0.2;
    c->morph_kernel = 2;
    c->morph_shape = DVC_SHAPE_ELLIPSE;
    c->max_batch = 16;
    c->device = 0;
    c->n_streams = 1;
}

static int create_impl(const dvc_config* cfg, dvc_handle* h) {
    char* ERRBUF = h->err;
    h->cfg = *cfg;
    h->W = cfg->width; h->H = cfg->height;
    h->cfg.n_streams = h->S = std::max(1, cfg->n_streams);
    h->wpr = words_per_row(h->W);
    h->plane_words = (size_t)h->H * h->wpr;
    h->plane_bytes = (size_t)h->H * h->W;
    h->frame_bytes = h->plane_bytes * 3;
    h->aligned = (h->W % 16) == 0;
    const int S = h->S;
    const int T = cfg->max_batch * S;          // planes of scratch per set: max_batch frames of every stream
    h->seg_len = std::max(1, measure_env("DVC_SEG_LEN", 8));
    h->gray_impl = measure_env("DVC_GRAY_IMPL", 2);
    CU(cudaSetDevice(cfg->device));
    h->resizing = cfg->src_width > 0 && cfg->src_height > 0 && (cfg->src_width != cfg->width || cfg->src_height != cfg->height);
    h->src_frame_bytes = h->resizing ? (size_t)cfg->src_width * cfg->src_height * 3 : h->frame_bytes;
    h->resize_tables = nullptr;
    if (h->resizing) {
        ResizeHostTables ht;
        make_resize_tables(cfg->src_height, cfg->src_width, h->H, h->W, ht);
        std::vector<char> blob;
        resize_tables_pack(ht, h->H, h->W, blob);
        CU(cudaMalloc(&h->resize_tables, blob.size()));
        CU(cudaMemcpy(h->resize_tables, blob.data(), blob.size(), cudaMemcpyHostToDevice));
    }
    for (int i = 0; i < 2; ++i) { CU(cudaMalloc(&h->prev_gray[i], h->plane_bytes * S)); CU(cudaMemset(h->prev_gray[i], 0, h->plane_bytes * S)); }
    for (int s = 0; s < 2; ++s)
        for (int k = 0; k < 3; ++k) {
            CU(cudaMalloc(&h->bits[s][k], h->plane_words * 4 * T));
            CU(cudaMemset(h->bits[s][k], 0, h->plane_words * 4 * T));
        }
    CU(cudaStreamCreateWithFlags(&h->s_front, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&h->s_mask, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&h->s_k4, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->ev_user, cudaEventDisableTiming));
    for (int s = 0; s < 2; ++s) {
        CU(cudaEventCreateWithFlags(&h->ev_front[s], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&h->ev_mask[s], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&h->ev_k4[s], cudaEventDisableTiming));
    }
    CU(cudaMalloc(&h->counters_dev, sizeof(Counters)));
    CU(cudaMemset(h->counters_dev, 0, sizeof(Counters)));
    h->chain.n = 0; h->chain.pad = 0; h->chain.halo_top = h->chain.halo_bot = 0;
    if (cfg->mode == DVC_MODE_FD) {
        CU(cudaMalloc(&h->acc, h->plane_bytes * S));
        CU(cudaMemset(h->acc, 0, h->plane_bytes * S));
        int rc = ccl_scratch_alloc(h->err, h->ccl, std::min(T, std::max(1, measure_env("DVC_CCL_CHUNK", 256))), h->H, h->W);
        if (rc) return rc;
        if (cfg->kernel_size > 0 && !chain_push(h->chain, DVC_MORPH_DILATE, DVC_SHAPE_RECT, cfg->kernel_size))
            return set_err(h->err, DVC_ERR_UNSUPPORTED, "kernel_size %d: supported range is 1..%d", cfg->kernel_size, MORPH_MAX_K);
    } else {
        if (cfg->window_size < 1 || cfg->window_size > WINDOW_MAX)
            return set_err(h->err, DVC_ERR_UNSUPPORTED, "window_size %d: supported range is 1..%d", cfg->window_size, WINDOW_MAX);
        h->ring_cap = cfg->max_batch + cfg->window_size + 1;
        CU(cudaMalloc(&h->ring, h->plane_words * 4 * h->ring_cap * S));
        CU(cudaMemset(h->ring, 0, h->plane_words * 4 * h->ring_cap * S));
        window_min_counts(cfg->alpha_fraction, cfg->window_size, h->min_counts);
        if (cfg->morph_kernel > 0) {
            if (!chain_push(h->chain, DVC_MORPH_CLOSE, cfg->morph_shape, cfg->morph_kernel) ||
                !chain_push(h->chain, DVC_MORPH_OPEN, cfg->morph_shape, cfg->morph_kernel))
                return set_err(h->err, DVC_ERR_UNSUPPORTED, "morph_kernel %d: supported range is 1..%d", cfg->morph_kernel, MORPH_MAX_K);
        }
        if (cfg->kernel_size > 0 && !chain_push(h->chain, DVC_MORPH_DILATE, DVC_SHAPE_RECT, cfg->kernel_size))
            return set_err(h->err, DVC_ERR_UNSUPPORTED, "kernel_size %d: supported range is 1..%d", cfg->kernel_size, MORPH_MAX_K);
    }
    return DVC_OK;
}

extern "C" int dvc_destroy(dvc_handle* h) {
    if (!h) return DVC_OK;
    cudaSetDevice(h->cfg.device);
    handle_join(h);
    cudaFree(h->prev_gray[0]); cudaFree(h->prev_gray[1]); cudaFree(h->acc); cudaFree(h->ring);
    for (int s = 0; s < 2; ++s) for (int k = 0; k < 3; ++k) cudaFree(h->bits[s][k]);
    cudaFree(h->blurred); cudaFree(h->counters_dev); cudaFree(h->resize_tables);
    if (h->s_front) cudaStreamDestroy(h->s_front);
    if (h->s_mask) cudaStreamDestroy(h->s_mask);
    if (h->s_k4) cudaStreamDestroy(h->s_k4);
    if (h->ev_in) cudaEventDestroy(h->ev_in);
    if (h->ev_user) cudaEventDestroy(h->ev_user);
    for (int s = 0; s < 2; ++s) { if (h->ev_front[s]) cudaEventDestroy(h->ev_front[s]); if (h->ev_mask[s]) cudaEventDestroy(h->ev_mask[s]); if (h->ev_k4[s]) cudaEventDestroy(h->ev_k4[s]); }
    ccl_scratch_free(h->ccl);
    if (h->staging) {
        for (int b = 0; b < 2; ++b) {
            cudaFree(h->st_in[b]); cudaFree(h->st_ov[b]); cudaFree(h->st_cp[b]); cudaFree(h->st_mask[b]);
            if (h->resizing) cudaFree(h->st_src[b]);
            cudaEventDestroy(h->ev_h2d[b]); cudaEventDestroy(h->ev_d2h[b]);
        }
        cudaStreamDestroy(h->s_h2d); cudaStreamDestroy(h->s_d2h);
    }
    if (h->prof_recs) { for (ProfRec& r : *h->prof_recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); } delete h->prof_recs; }
    delete h;
    return DVC_OK;
}

extern "C" int dvc_create(const dvc_config* cfg, dvc_handle** out) {
    if (!cfg || !out) return set_err(nullptr, DVC_ERR_INVALID, "dvc_create: null argument");
    *out = nullptr;
    if (cfg->width < 1 || cfg->height < 1 || cfg->max_batch < 1)
        return set_err(nullptr, DVC_ERR_INVALID, "dvc_create: width, height and max_batch must be >= 1");
    if (cfg->mode != DVC_MODE_FD && cfg->mode != DVC_MODE_WINDOW) return set_err(nullptr, DVC_ERR_INVALID, "dvc_create: unknown mode %d", cfg->mode);
    if (cfg->block_size < 1 || cfg->block_size > 8)
        return set_err(nullptr, DVC_ERR_UNSUPPORTED, "block_size %d: the GPU path implements 1..8 (cv2's DCT routines for longer blocks are not restated)", cfg->block_size);
    if (!(cfg->quantization_level > 0.0f)) return set_err(nullptr, DVC_ERR_INVALID, "quantization_level must be > 0");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return set_err(nullptr, DVC_ERR_CUDA, "no CUDA device: this library has no CPU fallback");
    dvc_handle* h = new dvc_handle();
    memset(h, 0, sizeof(*h));
    new (&h->ccl) CclScratch();
    h->prof_recs = new std::vector<ProfRec>();
    int rc = create_impl(cfg, h);
    if (rc) {
        char msg[512];
        strncpy(msg, h->err, 511); msg[511] = 0;
        dvc_destroy(h);
        set_err(nullptr, rc, "%s", msg);
        return rc;
    }
    *out = h;
    return DVC_OK;
}

extern "C" int dvc_begin_stream(dvc_handle* h, const uint8_t* prev_gray_host) {
    char* ERRBUF = h ? h->err : nullptr;
    if (!h || !prev_gray_host) return set_err(h ? h->err : nullptr, DVC_ERR_INVALID, "dvc_begin_stream: null argument");
    CU(cudaSetDevice(h->cfg.device));
    CU(handle_join(h));
    CU(h_copy(h, h->prev_gray[h->cur], prev_gray_host, h->plane_bytes * h->S, cudaMemcpyHostToDevice));
    if (h->acc) CU(h_fill0(h, h->acc, h->plane_bytes * h->S));
    if (h->ring) CU(h_fill0(h, h->ring, h->plane_words * 4 * h->ring_cap * h->S));
    h->n_masks = 0;
    return DVC_OK;
}

// ---- state blob: header | prev_gray | acc (FD)  or  K raw planes oldest..newest (WINDOW) ----------
struct StateHeader { uint32_t magic, mode, W, H, K, reserved; int64_t n_masks; };
static const uint32_t STATE_MAGIC = 0x31435644u;   // "DVC1"

extern "C" size_t dvc_state_bytes(const dvc_handle* h) {
    if (!h) return 0;
    size_t n = h->plane_bytes;
    n += h->cfg.mode == DVC_MODE_FD ? h->plane_bytes : (size_t)h->cfg.window_size * h->plane_words * 4;
    return sizeof(StateHeader) + n * h->S;      // header | per stream: prev_gray | acc or K raw planes
}

extern "C" int dvc_get_state(dvc_handle* h, void* buf, size_t bytes) {
    char* ERRBUF = h ? h->err : nullptr;
    if (!h || !buf || bytes < dvc_state_bytes(h)) return set_err(h ? h->err : nullptr, DVC_ERR_INVALID, "dvc_get_state: buffer too small");
    CU(cudaSetDevice(h->cfg.device));
    CU(handle_join(h));
    StateHeader hd = {STATE_MAGIC, (uint32_t)h->cfg.mode, (uint32_t)h->W, (uint32_t)h->H, (uint32_t)h->cfg.window_size, (uint32_t)h->S, h->n_masks};
    uint8_t* p = (uint8_t*)buf;
    memcpy(p, &hd, sizeof(hd)); p += sizeof(hd);
    for (int st = 0; st < h->S; ++st) {
        CU(h_copy(h, p, h->prev_gray[h->cur] + (size_t)st * h->plane_bytes, h->plane_bytes, cudaMemcpyDeviceToHost)); p += h->plane_bytes;
        if (h->cfg.mode == DVC_MODE_FD) {
            CU(h_copy(h, p, h->acc + (size_t)st * h->plane_bytes, h->plane_bytes, cudaMemcpyDeviceToHost)); p += h->plane_bytes;
        } else {
            const int K = h->cfg.window_size;
            const uint32_t* ring = h->ring + (size_t)st * h->ring_cap * h->plane_words;
            for (int i = 0; i < K; ++i) {       // slot i holds mask n_masks-K+i (zeros if before the stream start)
                const long long f = h->n_masks - K + i;
                if (f >= 0) CU(h_copy(h, p, ring + (size_t)(f % h->ring_cap) * h->plane_words, h->plane_words * 4, cudaMemcpyDeviceToHost));
                else memset(p, 0, h->plane_words * 4);
                p += h->plane_words * 4;
            }
        }
    }
    return DVC_OK;
}

extern "C" int dvc_set_state(dvc_handle* h, const void* buf, size_t bytes) {
    char* ERRBUF = h ? h->err : nullptr;
    if (!h || !buf || bytes < dvc_state_bytes(h)) return set_err(h ? h->err : nullptr, DVC_ERR_INVALID, "dvc_set_state: buffer too small");
    StateHeader hd;
    const uint8_t* p = (const uint8_t*)buf;
    memcpy(&hd, p, sizeof(hd)); p += sizeof(hd);
    if (hd.magic != STATE_MAGIC || hd.mode != (uint32_t)h->cfg.mode || hd.W != (uint32_t)h->W || hd.H != (uint32_t)h->H ||
        (h->cfg.mode == DVC_MODE_WINDOW && hd.K != (uint32_t)h->cfg.window_size) || std::max(1u, hd.reserved) != (uint32_t)h->S)
        return set_err(h->err, DVC_ERR_INVALID, "dvc_set_state: blob does not match this handle's configuration");
    CU(cudaSetDevice(h->cfg.device));
    CU(handle_join(h));
    h->n_masks = hd.n_masks;
    for (int st = 0; st < h->S; ++st) {
        CU(h_copy(h, h->prev_gray[h->cur] + (size_t)st * h->plane_bytes, p, h->plane_bytes, cudaMemcpyHostToDevice)); p += h->plane_bytes;
        if (h->cfg.mode == DVC_MODE_FD) {
            CU(h_copy(h, h->acc + (size_t)st * h->plane_bytes, p, h->plane_bytes, cudaMemcpyHostToDevice)); p += h->plane_bytes;
        } else {
            const int K = h->cfg.window_size;
            uint32_t* ring = h->ring + (size_t)st * h->ring_cap * h->plane_words;
            for (int i = 0; i < K; ++i) {
                const long long f = h->n_masks - K + i;
                if (f >= 0) CU(h_copy(h, ring + (size_t)(f % h->ring_cap) * h->plane_words, p, h->plane_words * 4, cudaMemcpyHostToDevice));
                p += h->plane_words * 4;
            }
        }
    }
    return DVC_OK;
}

extern "C" int dvc_get_counters(dvc_handle* h, dvc_counters* out) {
    char* ERRBUF = h ? h->err : nullptr;
    if (!h || !out) return set_err(h ? h->err : nullptr, DVC_ERR_INVALID, "dvc_get_counters: null argument");
    CU(cudaSetDevice(h->cfg.device));
    CU(handle_join(h));
    Counters c;
    CU(h_copy(h, &c, h->counters_dev, sizeof(c), cudaMemcpyDeviceToHost));
    *out = h->counters_host;
    out->motion_pixels = c.motion_pixels;
    out->static_blocks = c.static_blocks;
    return DVC_OK;
}

extern "C" int dvc_reset_counters(dvc_handle* h) {
    char* ERRBUF = h ? h->err : nullptr;
    if (!h) return set_err(nullptr, DVC_ERR_INVALID, "dvc_reset_counters: null handle");
    CU(cudaSetDevice(h->cfg.device));
    CU(handle_join(h));
    CU(h_fill0(h, h->counters_dev, sizeof(Counters)));
    memset(&h->counters_host, 0, sizeof(h->counters_host));
    return DVC_OK;
}

// ------------------------------------------------------------------------------------------------
// profiling hooks (dvc_profile_*): per kernel group, CUDA-event time on the launching stream
// ------------------------------------------------------------------------------------------------
struct ProfScope {
    dvc_handle* h; cudaStream_t st; int idx;
    ProfScope(dvc_handle* h_, int kid, int launches, cudaStream_t st_) : h(h_), st(st_), idx(-1) {
        h->launches += launches;
        if (!h->prof) return;
        ProfRec r; r.kid = kid; r.launches = launches;
        if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
        cudaEventRecord(r.a, st);
        h->prof_recs->push_back(r);
        idx = (int)h->prof_recs->size() - 1;
    }
    ~ProfScope() { if (idx >= 0) cudaEventRecord((*h->prof_recs)[idx].b, st); }
};

extern "C" int dvc_profile_enable(dvc_handle* h, int32_t on) {
    if (!h) return set_err(nullptr, DVC_ERR_INVALID, "dvc_profile_enable: null handle");
    h->prof = on != 0;
    return DVC_OK;
}

extern "C" int dvc_profile_read(dvc_handle* h, double* ms_by_kernel, int64_t* launches_by_kernel, int32_t n_kernels) {
    char* ERRBUF = h ? h->err : nullptr;
    if (!h || !ms_by_kernel || !launches_by_kernel || n_kernels < DVC_PROF_KERNELS)
        return set_err(ERRBUF, DVC_ERR_INVALID, "dvc_profile_read: need arrays of %d entries", DVC_PROF_KERNELS);
    CU(cudaSetDevice(h->cfg.device));
    CU(handle_join(h));
    for (int i = 0; i < n_kernels; ++i) { ms_by_kernel[i] = 0.0; launches_by_kernel[i] = 0; }
    for (ProfRec& r : *h->prof_recs) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) { ms_by_kernel[r.kid] += ms; launches_by_kernel[r.kid] += r.launches; }
        cudaEventDestroy(r.a); cudaEventDestroy(r.b);
    }
    h->prof_recs->clear();
    return DVC_OK;
}

extern "C" int64_t dvc_launch_count(const dvc_handle* h) { return h ? h->launches : 0; }

// ------------------------------------------------------------------------------------------------
// the loop body for one device-resident batch
// ------------------------------------------------------------------------------------------------
// Mask kernels run on `st`, the degrade kernel on `st_k4` (the same stream, or a second one so that it overlaps
// the mask kernels of the next batch); `set` selects the scratch bit-planes.
// st_front / st / st_k4: streams of the front kernel, of the other mask kernels and of the degrade kernel.  In pipelined mode they
// differ: the front kernel of batch n + 1 (issue- or HBM-bound, touches only the frames, its own state and scratch set (n + 1) % 2)
// runs beside the contour filter / morphology / EMA of batch n (latency-bound, a few hundred CTAs), which run beside the degrade
// kernel of batch n - 1.
static int process_batch_impl(dvc_handle* h, const uint8_t* frames, int T, uint8_t* overlay, uint8_t* compressed,
                              uint8_t* mask_out, cudaStream_t st_front, cudaStream_t st, cudaStream_t st_k4, int set) {
    char* ERRBUF = h->err;
    uint32_t* const bits_a = h->bits[set][0];
    uint32_t* const bits_b = h->bits[set][1];
    uint32_t* const bits_c = h->bits[set][2];
    const int H = h->H, W = h->W, wpr = h->wpr;
    const int S = h->S, ST = S * T;          // T frames of each of the S streams: buffers are [S][T] (stream-major)
    const uint32_t thr = (uint32_t)std::max(0.0f, std::floor(h->cfg.motion_threshold));
    const uint32_t* over127 = nullptr;
    const uint32_t* nonzero = nullptr;
    const unsigned g16 = cdiv((size_t)((W + 15) / 16) * H, 256);
    if (h->cfg.mode == DVC_MODE_WINDOW) {
        uint8_t* pg_in = h->prev_gray[h->cur];
        uint8_t* pg_out = h->prev_gray[h->cur ^ 1];
        const int K = h->cfg.window_size;
        static const bool fuse_env = measure_env("DVC_FUSE_VOTE", 1) != 0;
        if (h->aligned && K <= 8 && h->gray_impl == 2 && fuse_env) {
            // K1 + K2 in one kernel (k_gray_diff_vote): long segments, each rebuilding its K - 1 frames of history
            const int seg = std::max(K, std::max(8, measure_env("DVC_FUSE_SEG", 64))), nsegf = (T + seg - 1) / seg;
            dim3 gf(g16, nsegf, S);
            {
            ProfScope ps(h, DVC_PROF_FRONT, 1, st_front);
#define DVC_VOTE_CASE(KK) case KK: k_gray_diff_vote<KK><<<gf, 256, 0, st_front>>>(frames, T, H, W, pg_in, pg_out, h->ring, wpr, h->ring_cap, h->n_masks, thr, seg, h->min_counts, bits_a); break;
            switch (K) {
                DVC_VOTE_CASE(1) DVC_VOTE_CASE(2) DVC_VOTE_CASE(3) DVC_VOTE_CASE(4)
                DVC_VOTE_CASE(5) DVC_VOTE_CASE(6) DVC_VOTE_CASE(7) DVC_VOTE_CASE(8)
            }
#undef DVC_VOTE_CASE
            }
            CHECK_LAUNCH();
            if (st_front != st) { CU(cudaEventRecord(h->ev_front[set], st_front)); CU(cudaStreamWaitEvent(st, h->ev_front[set], 0)); }
            h->cur ^= 1;
        } else {
        const int nseg = (T + h->seg_len - 1) / h->seg_len;
        dim3 g1(g16, nseg, S);
        { ProfScope ps(h, DVC_PROF_FRONT, 1, st);
        if (h->aligned && h->gray_impl == 2)
            k_gray_diff_thresh<true, 2><<<g1, 256, 0, st>>>(frames, T, H, W, pg_in, pg_out, nullptr, h->ring, wpr, h->ring_cap, h->n_masks, thr, h->seg_len);
        else if (h->aligned && h->gray_impl == 1)
            k_gray_diff_thresh<true, 1><<<g1, 256, 0, st>>>(frames, T, H, W, pg_in, pg_out, nullptr, h->ring, wpr, h->ring_cap, h->n_masks, thr, h->seg_len);
        else if (h->aligned)
            k_gray_diff_thresh<true><<<g1, 256, 0, st>>>(frames, T, H, W, pg_in, pg_out, nullptr, h->ring, wpr, h->ring_cap, h->n_masks, thr, h->seg_len);
        else
            k_gray_diff_thresh<false><<<g1, 256, 0, st>>>(frames, T, H, W, pg_in, pg_out, nullptr, h->ring, wpr, h->ring_cap, h->n_masks, thr, h->seg_len);
        }
        CHECK_LAUNCH();
        h->cur ^= 1;
        dim3 g2(cdiv(h->plane_words, 256), nseg, S);
        { ProfScope ps(h, DVC_PROF_VOTE, 1, st);
        if (K <= 31) k_window_vote<5><<<g2, 256, 0, st>>>(h->ring, h->ring_cap, H, W, wpr, h->n_masks, (int)(h->n_masks % h->ring_cap), T, K, h->min_counts, bits_a, h->seg_len);
        else k_window_vote<7><<<g2, 256, 0, st>>>(h->ring, h->ring_cap, H, W, wpr, h->n_masks, (int)(h->n_masks % h->ring_cap), T, K, h->min_counts, bits_a, h->seg_len);
        }
        CHECK_LAUNCH();
        }
        const uint32_t* fin = bits_a;
        if (h->chain.n) {
            ProfScope ps(h, DVC_PROF_MORPH, 1, st);
            int rc = launch_morph_chain(h->err, bits_a, bits_b, ST, H, W, h->chain, st);
            if (rc) return rc;
            fin = bits_b;
        }
        over127 = nonzero = fin;
        if (mask_out) {
            ProfScope ps(h, DVC_PROF_MISC, 1, st);
            int rc = unpack_from_bits(fin, mask_out, ST, H, W, st);
            if (rc) return rc;
        }
    } else {
        // gray -> blur5 -> absdiff -> threshold fused and walking the frames of a segment: the blurred planes stay in registers
        const int tiles = (wpr / 4) * ((H + FF_TH - 1) / FF_TH);
        const int want_segs = std::max(1, (1500 + tiles * S - 1) / (tiles * S));          // enough CTAs for a few waves
        static const int seg_env = measure_env("DVC_FD_SEG", 0);                          // > 0: frames a CTA walks
        const int seg0 = seg_env > 0 ? seg_env : std::min(32, std::max(4, (T + want_segs - 1) / want_segs));
        const int nseg = (T + seg0 - 1) / seg0;
        const int seg = (T + nseg - 1) / nseg;                                              // balanced: no short last segment
        dim3 gf(wpr / 4, (H + FF_TH - 1) / FF_TH, S * nseg);
        { ProfScope ps(h, DVC_PROF_FRONT, 1, st_front);
        if (h->aligned) k_fd_front<true><<<gf, 256, 0, st_front>>>(frames, T, H, W, h->prev_gray[h->cur], h->prev_gray[h->cur ^ 1], bits_a, wpr, thr, seg, nseg);
        else k_fd_front<false><<<gf, 256, 0, st_front>>>(frames, T, H, W, h->prev_gray[h->cur], h->prev_gray[h->cur ^ 1], bits_a, wpr, thr, seg, nseg);
        }
        CHECK_LAUNCH();
        if (st_front != st) { CU(cudaEventRecord(h->ev_front[set], st_front)); CU(cudaStreamWaitEvent(st, h->ev_front[set], 0)); }
        h->cur ^= 1;
        int rc;
        { ProfScope ps(h, DVC_PROF_CCL, (h->ccl.sweep ? 1 : 7) * ((ST + h->ccl.frames - 1) / h->ccl.frames), st);
        rc = launch_contour_filter(h->err, bits_a, bits_b, ST, H, W, h->cfg.min_area, h->ccl, st);
        }
        if (rc) return rc;
        { ProfScope ps(h, DVC_PROF_MORPH, 1, st);
        rc = launch_morph_chain(h->err, bits_b, bits_a, ST, H, W, h->chain, st);      // dilate -> bits_a
        }
        if (rc) return rc;
        const float alpha = (float)h->cfg.release_factor, beta = (float)(1.0 - h->cfg.release_factor);
        { ProfScope ps(h, DVC_PROF_EMA, 1, st);
        static const int ema_px = measure_env("DVC_EMA_PX", 8);
        if (h->aligned && ema_px == 8)
            k_ema<true, 8><<<dim3(cdiv((size_t)(W / 8) * H, 256), S), 256, 0, st>>>(h->acc, bits_a, bits_b, bits_c, mask_out, T, H, W, wpr, alpha, beta);
        else if (h->aligned) k_ema<true><<<dim3(g16, S), 256, 0, st>>>(h->acc, bits_a, bits_b, bits_c, mask_out, T, H, W, wpr, alpha, beta);
        else k_ema<false><<<dim3(g16, S), 256, 0, st>>>(h->acc, bits_a, bits_b, bits_c, mask_out, T, H, W, wpr, alpha, beta);
        }
        CHECK_LAUNCH();
        over127 = bits_b;
        nonzero = bits_c;
    }
    if (st_k4 != st) {
        CU(cudaEventRecord(h->ev_mask[set], st));
        CU(cudaStreamWaitEvent(st_k4, h->ev_mask[set], 0));
    }
    if (overlay || compressed) {
        ProfScope ps(h, DVC_PROF_DEGRADE, 1, st_k4);
        int rc = launch_degrade(h->err, frames, over127, nonzero, compressed, overlay, ST, H, W, h->cfg.block_size,
                                h->cfg.quantization_level, DVC_DEGRADE_FD, h->counters_dev, st_k4);
        if (rc) return rc;
    }
    if (st_k4 != st) {
        CU(cudaEventRecord(h->ev_k4[set], st_k4));
        h->ev_used[set] = true;
    }
    h->n_masks += T;
    h->counters_host.frames += ST;
    h->counters_host.pixels += (uint64_t)ST * H * W;
    h->counters_host.blocks += (uint64_t)ST * ((H + h->cfg.block_size - 1) / h->cfg.block_size) * ((W + h->cfg.block_size - 1) / h->cfg.block_size);   // clipped edge blocks count (frame_differencing.py:117-118)
    return DVC_OK;
}

// fd mode: the front kernel (issue-bound) gets its own stream and runs a batch ahead of the contour filter / EMA (latency-bound):
// 129 k -> 143 k frames/s at 1080p.  Window mode: its front kernel is HBM-bound like the degrade kernel it would run beside
// (201 k -> 194 k frames/s with its own stream), so it stays on the mask stream.
static cudaStream_t front_stream_of(dvc_handle* h) {
    static const int sel = measure_env("DVC_FRONT_STREAM", -1);       // -1: by mode, 0: never, 1: always
    const bool own = sel < 0 ? h->cfg.mode == DVC_MODE_FD : sel != 0;
    return own ? h->s_front : h->s_mask;
}

extern "C" int dvc_process_batch(dvc_handle* h, const uint8_t* frames_dev, int32_t n_frames, uint8_t* overlay_dev,
                                 uint8_t* compressed_dev, uint8_t* mask_dev, void* stream) {
    char* ERRBUF = h ? h->err : nullptr;
    if (!h) return set_err(nullptr, DVC_ERR_INVALID, "dvc_process_batch: null handle");
    if (n_frames < 0 || n_frames > h->cfg.max_batch) return set_err(h->err, DVC_ERR_INVALID, "dvc_process_batch: n_frames %d outside 0..max_batch (%d)", n_frames, h->cfg.max_batch);
    if (n_frames == 0) return DVC_OK;
    if (!frames_dev) return set_err(h->err, DVC_ERR_INVALID, "dvc_process_batch: null frames");
    CU(cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    if (!h->overlap) {
        int rc = process_batch_impl(h, frames_dev, n_frames, overlay_dev, compressed_dev, mask_dev, st, st, st, 0);
        if (rc == DVC_OK) { CU(cudaEventRecord(h->ev_user, st)); h->ev_user_used = true; }
        return rc;
    }
    // pipelined: the batch is ordered after the work already in `stream`, but `stream` is only re-joined by dvc_flush
    const int set = h->pp;
    h->pp ^= 1;
    cudaStream_t sf = front_stream_of(h);
    CU(cudaEventRecord(h->ev_in, st));
    CU(cudaStreamWaitEvent(h->s_mask, h->ev_in, 0));
    if (h->ev_used[set]) CU(cudaStreamWaitEvent(h->s_mask, h->ev_k4[set], 0));      // scratch set free again
    if (sf != h->s_mask) {
        CU(cudaStreamWaitEvent(sf, h->ev_in, 0));
        if (h->ev_used[set]) CU(cudaStreamWaitEvent(sf, h->ev_k4[set], 0));
    }
    return process_batch_impl(h, frames_dev, n_frames, overlay_dev, compressed_dev, mask_dev, sf, h->s_mask, h->s_k4, set);
}

extern "C" int dvc_set_overlap(dvc_handle* h, int32_t on) {
    char* ERRBUF = h ? h->err : nullptr;
    if (!h) return set_err(nullptr, DVC_ERR_INVALID, "dvc_set_overlap: null handle");
    CU(cudaSetDevice(h->cfg.device));
    CU(handle_join(h));
    h->overlap = on != 0;
    return DVC_OK;
}

extern "C" int dvc_flush(dvc_handle* h, void* stream) {
    char* ERRBUF = h ? h->err : nullptr;
    if (!h) return set_err(nullptr, DVC_ERR_INVALID, "dvc_flush: null handle");
    CU(cudaSetDevice(h->cfg.device));
    for (int s = 0; s < 2; ++s)
        if (h->ev_used[s]) {
            CU(cudaStreamWaitEvent((cudaStream_t)stream, h->ev_mask[s], 0));
            CU(cudaStreamWaitEvent((cudaStream_t)stream, h->ev_k4[s], 0));
        }
    return DVC_OK;
}

extern "C" int dvc_process_host(dvc_handle* h, const uint8_t* frames_host, int64_t n_frames, uint8_t* overlay_host,
                                uint8_t* compressed_host, uint8_t* mask_host) {
    char* ERRBUF = h ? h->err : nullptr;
    if (!h) return set_err(nullptr, DVC_ERR_INVALID, "dvc_process_host: null handle");
    if (n_frames < 0) return set_err(h->err, DVC_ERR_INVALID, "dvc_process_host: negative n_frames");
    if (n_frames == 0) return DVC_OK;
    if (!frames_host) return set_err(h->err, DVC_ERR_INVALID, "dvc_process_host: null frames");
    CU(cudaSetDevice(h->cfg.device));
    int rc = alloc_staging(h);
    if (rc) return rc;
    const int Tc = host_chunk_frames(h);
    const int S = h->S;
    const int64_t nchunks = (n_frames + Tc - 1) / Tc;
    CU(handle_join(h));                   // join whatever dvc_process_batch left in flight (this handle only)
    for (int64_t c = 0; c < nchunks; ++c) {
        const int b = (int)(c & 1);       // staging buffers, scratch set and events all alternate with the chunk
        const int64_t f0 = c * Tc;
        const int T = (int)std::min<int64_t>(Tc, n_frames - f0);
        // the input buffer is free once the degrade kernel that read it (chunk c-2) is done
        if (c >= 2) CU(cudaStreamWaitEvent(h->s_h2d, h->ev_k4[b], 0));
        // host buffers are [S][n_frames] (stream-major), the device staging of a chunk is [S][T]: one copy per stream
        if (h->resizing) {
            // frames arrive at the capture's size: upload, then the reference's cv2.resize (frame_differencing.py:91) on the GPU
            for (int sidx = 0; sidx < S; ++sidx)
                CU(cudaMemcpyAsync(h->st_src[b] + (size_t)sidx * T * h->src_frame_bytes,
                                   frames_host + ((size_t)sidx * n_frames + f0) * h->src_frame_bytes, (size_t)T * h->src_frame_bytes,
                                   cudaMemcpyHostToDevice, h->s_h2d));
            rc = launch_resize(h->err, h->st_src[b], h->st_in[b], S * T, h->cfg.src_height, h->cfg.src_width, h->H, h->W, 3,
                               resize_tables_view(h->resize_tables, h->H, h->W), h->s_h2d);
            if (rc) { handle_join(h); return rc; }
            h->launches += 1;
        } else
        for (int sidx = 0; sidx < S; ++sidx)
            CU(cudaMemcpyAsync(h->st_in[b] + (size_t)sidx * T * h->frame_bytes, frames_host + ((size_t)sidx * n_frames + f0) * h->frame_bytes,
                               (size_t)T * h->frame_bytes, cudaMemcpyHostToDevice, h->s_h2d));
        CU(cudaEventRecord(h->ev_h2d[b], h->s_h2d));
        CU(cudaStreamWaitEvent(h->s_mask, h->ev_h2d[b], 0));
        cudaStream_t sf = front_stream_of(h);
        if (sf != h->s_mask) CU(cudaStreamWaitEvent(sf, h->ev_h2d[b], 0));
        if (c >= 2) {
            CU(cudaStreamWaitEvent(h->s_mask, h->ev_k4[b], 0));      // scratch set b free
            if (sf != h->s_mask) CU(cudaStreamWaitEvent(sf, h->ev_k4[b], 0));
            CU(cudaStreamWaitEvent(h->s_mask, h->ev_d2h[b], 0));     // output staging of chunk c-2 downloaded
            CU(cudaStreamWaitEvent(h->s_k4, h->ev_d2h[b], 0));
        }
        static const bool no_kernels = measure_env("DVC_HOST_NOKERNEL", 0) != 0;   // copy-pipeline probe
        if (no_kernels) { CU(cudaEventRecord(h->ev_k4[b], h->s_k4)); h->ev_used[b] = true; rc = DVC_OK; } else
        rc = process_batch_impl(h, h->st_in[b], T, overlay_host ? h->st_ov[b] : nullptr, compressed_host ? h->st_cp[b] : nullptr,
                                mask_host ? h->st_mask[b] : nullptr, sf, h->s_mask, h->s_k4, b);
        if (rc) { handle_join(h); return rc; }
        CU(cudaStreamWaitEvent(h->s_d2h, h->ev_k4[b], 0));
        for (int sidx = 0; sidx < S; ++sidx) {
            const size_t ho = (size_t)sidx * n_frames + f0, so = (size_t)sidx * T;
            if (overlay_host) CU(cudaMemcpyAsync(overlay_host + ho * h->frame_bytes, h->st_ov[b] + so * h->frame_bytes, (size_t)T * h->frame_bytes, cudaMemcpyDeviceToHost, h->s_d2h));
            if (compressed_host) CU(cudaMemcpyAsync(compressed_host + ho * h->frame_bytes, h->st_cp[b] + so * h->frame_bytes, (size_t)T * h->frame_bytes, cudaMemcpyDeviceToHost, h->s_d2h));
            if (mask_host) CU(cudaMemcpyAsync(mask_host + ho * h->plane_bytes, h->st_mask[b] + so * h->plane_bytes, (size_t)T * h->plane_bytes, cudaMemcpyDeviceToHost, h->s_d2h));
        }
        CU(cudaEventRecord(h->ev_d2h[b], h->s_d2h));
    }
    CU(cudaStreamSynchronize(h->s_d2h));
    CU(cudaStreamSynchronize(h->s_k4));
    CU(cudaStreamSynchronize(h->s_mask));
    CU(cudaStreamSynchronize(h->s_front));
    h->ev_used[0] = h->ev_used[1] = false;
    h->pp = 0;
    return DVC_OK;
}

// ------------------------------------------------------------------------------------------------
// stage-level entry points (stateless; scratch from the stream-ordered allocator)
// ------------------------------------------------------------------------------------------------
// The stream-ordered allocator's default pool gives memory back to the driver at every synchronisation point (release threshold
// 0), which turns the scratch of a stage-level call into a fresh driver allocation each time (about 0.5 ms per call measured on
// dvc_degrade_blend_u8).  Keep it cached: set once per device.
static PerDeviceOnce g_pool_once;
static void keep_async_pool_cached() {
    if (auto once = g_pool_once.begin()) {
        int dev = 0;
        cudaMemPool_t pool;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
            unsigned long long keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        once.commit();
    }
}

struct ScopedAsyncBuf {
    void* p = nullptr;
    cudaStream_t st;
    explicit ScopedAsyncBuf(cudaStream_t s) : st(s) {}
    cudaError_t alloc(size_t n) { keep_async_pool_cached(); return cudaMallocAsync(&p, n ? n : 1, st); }
    ~ScopedAsyncBuf() { if (p) cudaFreeAsync(p, st); }
};

static int check_dims(int n, int H, int W, const char* who) {
    if (n < 0 || H < 1 || W < 1) return set_err(nullptr, DVC_ERR_INVALID, "%s: bad dimensions n=%d H=%d W=%d", who, n, H, W);
    return DVC_OK;
}

extern "C" int dvc_bgr2gray_u8(const uint8_t* bgr, uint8_t* gray, int32_t n, int32_t H, int32_t W, void* stream) {
    char* ERRBUF = nullptr;
    int rc = check_dims(n, H, W, "dvc_bgr2gray_u8");
    if (rc || n == 0) return rc;
    if (!bgr || !gray) return set_err(nullptr, DVC_ERR_INVALID, "dvc_bgr2gray_u8: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    dim3 g(cdiv((size_t)((W + 15) / 16) * H, 256), n);
    if (W % 16 == 0) k_bgr2gray<true><<<g, 256, 0, st>>>(bgr, gray, H, W);
    else k_bgr2gray<false><<<g, 256, 0, st>>>(bgr, gray, H, W);
    CHECK_LAUNCH();
    return DVC_OK;
}

extern "C" int dvc_gray_absdiff_thresh_u8(const uint8_t* bgr, const uint8_t* prev_gray, uint8_t* gray_out, uint8_t* mask_out,
                                          int32_t n, int32_t H, int32_t W, float motion_threshold, int32_t blur5, void* stream) {
    char* ERRBUF = nullptr;
    int rc = check_dims(n, H, W, "dvc_gray_absdiff_thresh_u8");
    if (rc || n == 0) return rc;
    if (!bgr || !prev_gray) return set_err(nullptr, DVC_ERR_INVALID, "dvc_gray_absdiff_thresh_u8: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const int wpr = words_per_row(W);
    const size_t pw = (size_t)H * wpr, pb = (size_t)H * W;
    const uint32_t thr = (uint32_t)std::max(0.0f, std::floor(motion_threshold));
    const bool al = W % 16 == 0;
    ScopedAsyncBuf bits(st), gray_tmp(st);
    CU(bits.alloc(pw * 4 * n));
    CU(cudaMemsetAsync(bits.p, 0, pw * 4 * n, st));
    const unsigned g16 = cdiv((size_t)((W + 15) / 16) * H, 256);
    if (!blur5) {
        const int seg = 8, nseg = (n + seg - 1) / seg;
        dim3 g1(g16, nseg);
        if (al) k_gray_diff_thresh<true><<<g1, 256, 0, st>>>(bgr, n, H, W, prev_gray, nullptr, gray_out, (uint32_t*)bits.p, wpr, n, 0, thr, seg);
        else k_gray_diff_thresh<false><<<g1, 256, 0, st>>>(bgr, n, H, W, prev_gray, nullptr, gray_out, (uint32_t*)bits.p, wpr, n, 0, thr, seg);
        CHECK_LAUNCH();
    } else {
        uint8_t* bl = gray_out;
        if (!bl) { CU(gray_tmp.alloc(pb * n)); bl = (uint8_t*)gray_tmp.p; }
        dim3 gb((W + BL_TW - 1) / BL_TW, (H + BL_TH - 1) / BL_TH, n);
        if (al) k_gray_blur5<true><<<gb, 256, 0, st>>>(bgr, bl, H, W);
        else k_gray_blur5<false><<<gb, 256, 0, st>>>(bgr, bl, H, W);
        CHECK_LAUNCH();
        dim3 gd(g16, n);
        if (al) k_diff_thresh_planes<true><<<gd, 256, 0, st>>>(bl, prev_gray, H, W, (uint32_t*)bits.p, wpr, thr);
        else k_diff_thresh_planes<false><<<gd, 256, 0, st>>>(bl, prev_gray, H, W, (uint32_t*)bits.p, wpr, thr);
        CHECK_LAUNCH();
    }
    if (mask_out) return unpack_from_bits((const uint32_t*)bits.p, mask_out, n, H, W, st);
    return DVC_OK;
}

static int pack_to_bits(const uint8_t* src, uint32_t* dst, int n, int H, int W, cudaStream_t st) {
    char* ERRBUF = nullptr;
    const int wpr = words_per_row(W);
    dim3 g(cdiv((size_t)((W + 15) / 16) * H, 256), n);
    CU(cudaMemsetAsync(dst, 0, (size_t)n * H * wpr * 4, st));           // padding words of each row stay zero
    if (W % 16 == 0) k_pack_bits<true, false><<<g, 256, 0, st>>>(src, dst, nullptr, H, W, wpr);
    else k_pack_bits<false, false><<<g, 256, 0, st>>>(src, dst, nullptr, H, W, wpr);
    CHECK_LAUNCH();
    return DVC_OK;
}
static int unpack_from_bits(const uint32_t* src, uint8_t* dst, int n, int H, int W, cudaStream_t st) {
    char* ERRBUF = nullptr;
    const int wpr = words_per_row(W);
    dim3 g(cdiv((size_t)((W + 15) / 16) * H, 256), n);
    if (W % 16 == 0) k_unpack_bits<true><<<g, 256, 0, st>>>(src, dst, H, W, wpr);
    else k_unpack_bits<false><<<g, 256, 0, st>>>(src, dst, H, W, wpr);
    CHECK_LAUNCH();
    return DVC_OK;
}

extern "C" int dvc_temporal_ring_u8(const uint8_t* masks, uint8_t* smoothed, int32_t n, int32_t H, int32_t W,
                                    int32_t window_size, double alpha_fraction, void* stream) {
    char* ERRBUF = nullptr;
    int rc = check_dims(n, H, W, "dvc_temporal_ring_u8");
    if (rc || n == 0) return rc;
    if (!masks || !smoothed) return set_err(nullptr, DVC_ERR_INVALID, "dvc_temporal_ring_u8: null pointer");
    if (window_size < 1 || window_size > WINDOW_MAX) return set_err(nullptr, DVC_ERR_UNSUPPORTED, "window_size %d: supported range is 1..%d", window_size, WINDOW_MAX);
    cudaStream_t st = (cudaStream_t)stream;
    const int wpr = words_per_row(W);
    const size_t pw = (size_t)H * wpr;
    ScopedAsyncBuf ring(st), voted(st);
    CU(ring.alloc(pw * 4 * n));
    CU(voted.alloc(pw * 4 * n));
    rc = pack_to_bits(masks, (uint32_t*)ring.p, n, H, W, st);
    if (rc) return rc;
    MinCounts mc;
    window_min_counts(alpha_fraction, window_size, mc);
    const int seg = 8, nseg = (n + seg - 1) / seg;
    dim3 g(cdiv(pw, 256), nseg);
    if (window_size <= 31) k_window_vote<5><<<g, 256, 0, st>>>((const uint32_t*)ring.p, n, H, W, wpr, 0, 0, n, window_size, mc, (uint32_t*)voted.p, seg);
    else k_window_vote<7><<<g, 256, 0, st>>>((const uint32_t*)ring.p, n, H, W, wpr, 0, 0, n, window_size, mc, (uint32_t*)voted.p, seg);
    CHECK_LAUNCH();
    return unpack_from_bits((const uint32_t*)voted.p, smoothed, n, H, W, st);
}

extern "C" int dvc_temporal_ema_u8(uint8_t* acc, const uint8_t* dilated, uint8_t* acc_all, int32_t n, int32_t H, int32_t W,
                                   double release_factor, void* stream) {
    char* ERRBUF = nullptr;
    int rc = check_dims(n, H, W, "dvc_temporal_ema_u8");
    if (rc || n == 0) return rc;
    if (!acc || !dilated) return set_err(nullptr, DVC_ERR_INVALID, "dvc_temporal_ema_u8: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const int wpr = words_per_row(W);
    const size_t pw = (size_t)H * wpr;
    ScopedAsyncBuf bits(st), f1(st), f2(st);
    CU(bits.alloc(pw * 4 * n));
    CU(f1.alloc(pw * 4 * n));
    CU(f2.alloc(pw * 4 * n));
    rc = pack_to_bits(dilated, (uint32_t*)bits.p, n, H, W, st);
    if (rc) return rc;
    const float alpha = (float)release_factor, beta = (float)(1.0 - release_factor);
    const unsigned g16 = cdiv((size_t)((W + 15) / 16) * H, 256);
    if (W % 16 == 0) k_ema<true><<<g16, 256, 0, st>>>(acc, (const uint32_t*)bits.p, (uint32_t*)f1.p, (uint32_t*)f2.p, acc_all, n, H, W, wpr, alpha, beta);
    else k_ema<false><<<g16, 256, 0, st>>>(acc, (const uint32_t*)bits.p, (uint32_t*)f1.p, (uint32_t*)f2.p, acc_all, n, H, W, wpr, alpha, beta);
    CHECK_LAUNCH();
    return DVC_OK;
}

extern "C" int dvc_morph_u8(const uint8_t* src, uint8_t* dst, int32_t n, int32_t H, int32_t W, int32_t op, int32_t shape,
                            int32_t k, void* stream) {
    char* ERRBUF = nullptr;
    int rc = check_dims(n, H, W, "dvc_morph_u8");
    if (rc || n == 0) return rc;
    if (!src || !dst) return set_err(nullptr, DVC_ERR_INVALID, "dvc_morph_u8: null pointer");
    if (op < DVC_MORPH_ERODE || op > DVC_MORPH_CLOSE || (shape != DVC_SHAPE_RECT && shape != DVC_SHAPE_ELLIPSE))
        return set_err(nullptr, DVC_ERR_INVALID, "dvc_morph_u8: bad op/shape");
    MorphChain ch;
    ch.n = 0; ch.pad = 0; ch.halo_top = ch.halo_bot = 0;
    if (!chain_push(ch, op, shape, k)) return set_err(nullptr, DVC_ERR_UNSUPPORTED, "dvc_morph_u8: kernel size %d outside 1..%d", k, MORPH_MAX_K);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t pw = (size_t)H * words_per_row(W);
    ScopedAsyncBuf a(st), b(st);
    CU(a.alloc(pw * 4 * n));
    CU(b.alloc(pw * 4 * n));
    rc = pack_to_bits(src, (uint32_t*)a.p, n, H, W, st);
    if (rc) return rc;
    rc = launch_morph_chain(nullptr, (const uint32_t*)a.p, (uint32_t*)b.p, n, H, W, ch, st);
    if (rc) return rc;
    return unpack_from_bits((const uint32_t*)b.p, dst, n, H, W, st);
}

extern "C" int dvc_contour_filter_u8(const uint8_t* src, uint8_t* dst, int32_t n, int32_t H, int32_t W, double min_area,
                                     void* stream) {
    char* ERRBUF = nullptr;
    int rc = check_dims(n, H, W, "dvc_contour_filter_u8");
    if (rc || n == 0) return rc;
    if (!src || !dst) return set_err(nullptr, DVC_ERR_INVALID, "dvc_contour_filter_u8: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t pw = (size_t)H * words_per_row(W);
    CclScratch sc;
    sc.sweep = ccl_sweep_usable(H, W);
    const int fr = std::min(n, sc.sweep ? 32 : 8);
    const size_t d = ccl_dense_ints(H, W) * sizeof(int) * fr, o = ccl_overflow_ints(H, W) * sizeof(int) * fr;
    ScopedAsyncBuf a(st), b(st), pa(st), pb(st), ar(st), fl(st), rfl(st);
    CU(a.alloc(pw * 4 * n));
    CU(b.alloc(pw * 4 * n));
    sc.frames = fr;
    if (!sc.sweep) { CU(fl.alloc(pw * 4 * fr)); sc.filled = (uint32_t*)fl.p; }
    if (sc.sweep) {
        sc.g_stride = ccl_sweep_max_nodes(H, W);
        CU(pa.alloc(sc.g_stride * sizeof(int) * fr)); CU(pb.alloc(sc.g_stride * sizeof(int) * fr));
        sc.gp = (int*)pa.p; sc.ga = (int*)pb.p;
    } else {
        CU(pa.alloc(d + o)); CU(pb.alloc(d + o)); CU(ar.alloc(d + o));      // dense + overflow pairs, one allocation each
        CU(rfl.alloc((size_t)fr * H));
        sc.rowflag = (uint8_t*)rfl.p;
        sc.pa0 = (int*)pa.p; sc.paov = sc.pa0 + d / sizeof(int); sc.pb0 = (int*)pb.p; sc.pbov = sc.pb0 + d / sizeof(int);
        sc.ar0 = (int*)ar.p; sc.arov = sc.ar0 + d / sizeof(int);
    }
    rc = pack_to_bits(src, (uint32_t*)a.p, n, H, W, st);
    if (rc) return rc;
    rc = launch_contour_filter(nullptr, (const uint32_t*)a.p, (uint32_t*)b.p, n, H, W, min_area, sc, st);
    if (rc) return rc;
    return unpack_from_bits((const uint32_t*)b.p, dst, n, H, W, st);
}

extern "C" int dvc_resize_linear_u8(const uint8_t* src, uint8_t* dst, int32_t n, int32_t src_h, int32_t src_w, int32_t dst_h,
                                    int32_t dst_w, int32_t channels, void* stream) {
    char* ERRBUF = nullptr;
    int rc = check_dims(n, src_h, src_w, "dvc_resize_linear_u8");
    if (rc || n == 0) return rc;
    if (dst_h <= 0 || dst_w <= 0) return set_err(nullptr, DVC_ERR_INVALID, "dvc_resize_linear_u8: bad destination size %dx%d", dst_w, dst_h);
    if (!src || !dst) return set_err(nullptr, DVC_ERR_INVALID, "dvc_resize_linear_u8: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    ResizeHostTables ht;
    make_resize_tables(src_h, src_w, dst_h, dst_w, ht);
    std::vector<char> blob;
    resize_tables_pack(ht, dst_h, dst_w, blob);
    ScopedAsyncBuf tb(st);
    CU(tb.alloc(blob.size()));
    CU(cudaMemcpyAsync(tb.p, blob.data(), blob.size(), cudaMemcpyHostToDevice, st));
    rc = launch_resize(nullptr, src, dst, n, src_h, src_w, dst_h, dst_w, channels, resize_tables_view(tb.p, dst_h, dst_w), st);
    CU(cudaStreamSynchronize(st));          // the pageable host blob must outlive the copy
    return rc;
}

extern "C" int dvc_mask_rectangles_u8(const uint8_t* src, uint8_t* dst, int32_t n, int32_t H, int32_t W, void* stream) {
    char* ERRBUF = nullptr;
    int rc = check_dims(n, H, W, "dvc_mask_rectangles_u8");
    if (rc || n == 0) return rc;
    if (!src || !dst) return set_err(nullptr, DVC_ERR_INVALID, "dvc_mask_rectangles_u8: null pointer");
    if (W > 32767 || H > 32767) return set_err(nullptr, DVC_ERR_UNSUPPORTED, "dvc_mask_rectangles_u8: image larger than 32767");
    cudaStream_t st = (cudaStream_t)stream;
    const int wpr = words_per_row(W);
    const size_t pw = (size_t)H * wpr;
    const int fr = std::min(n, 4);
    const size_t d = ccl_dense_ints(H, W) * sizeof(int) * fr, o = ccl_overflow_ints(H, W) * sizeof(int) * fr;
    ScopedAsyncBuf a(st), b(st), pp(st), bbuf(st);
    CU(a.alloc(pw * 4 * n));
    CU(b.alloc(pw * 4 * n));
    CU(pp.alloc(d + o)); CU(bbuf.alloc(3 * (d + o)));                     // dense + overflow pairs, one allocation each
    struct { void* p; } p0{pp.p}, pov{(char*)pp.p + d}, bd{bbuf.p}, bo{(char*)bbuf.p + 3 * d};
    rc = pack_to_bits(src, (uint32_t*)a.p, n, H, W, st);
    if (rc) return rc;
    CU(cudaMemsetAsync(b.p, 0, pw * 4 * n, st));
    BBoxArrays bb;
    for (int k = 0; k < 3; ++k) { bb.d[k] = (int*)((char*)bd.p + k * d); bb.ov[k] = (int*)((char*)bo.p + k * o); }
    for (int i0 = 0; i0 < n; i0 += fr) {
        const int m = std::min(fr, n - i0);
        dim3 grid(cdiv(pw, 256), m), grow((H + 7) / 8, m);
        const uint32_t* r = (const uint32_t*)a.p + (size_t)i0 * pw;
        CU(cudaMemsetAsync(bd.p, 0x7f, 3 * d, st));           // 0x7f7f7f7f: larger than any coordinate or negated coordinate
        CU(cudaMemsetAsync(bo.p, 0x7f, 3 * o, st));
        k_ccl_rowlink<false, false><<<grow, 256, 0, st>>>(r, (int*)p0.p, (int*)pov.p, nullptr, nullptr, H, W, wpr, nullptr);
        k_ccl_union<false, 8><<<CCL_GRID(wpr, H, m), 256, 0, st>>>(r, (int*)p0.p, (int*)pov.p, H, W, wpr, nullptr);
        k_ccl_bbox<<<grid, 256, 0, st>>>(r, (int*)p0.p, (int*)pov.p, bb, H, W, wpr);
        k_ccl_paint_rects<<<grid, 256, 0, st>>>(r, (int*)p0.p, (int*)pov.p, bb, (uint32_t*)b.p + (size_t)i0 * pw, H, W, wpr);
        CHECK_LAUNCH();
    }
    return unpack_from_bits((const uint32_t*)b.p, dst, n, H, W, st);
}

extern "C" int dvc_degrade_blend_u8(const uint8_t* bgr, const uint8_t* mask, uint8_t* compressed, uint8_t* overlay, int32_t n,
                                    int32_t H, int32_t W, int32_t block_size, float q, int32_t flavour, uint64_t* counters,
                                    void* stream) {
    char* ERRBUF = nullptr;
    int rc = check_dims(n, H, W, "dvc_degrade_blend_u8");
    if (rc || n == 0) return rc;
    if (!bgr || !mask) return set_err(nullptr, DVC_ERR_INVALID, "dvc_degrade_blend_u8: null pointer");
    if (flavour != DVC_DEGRADE_FD && flavour != DVC_DEGRADE_MCO) return set_err(nullptr, DVC_ERR_INVALID, "dvc_degrade_blend_u8: bad flavour");
    cudaStream_t st = (cudaStream_t)stream;
    const int wpr = words_per_row(W);
    const size_t pw = (size_t)H * wpr;
    ScopedAsyncBuf hi(st), nz(st);
    CU(hi.alloc(pw * 4 * n));
    CU(nz.alloc(pw * 4 * n));
    dim3 g(cdiv((size_t)((W + 15) / 16) * H, 256), n);
    CU(cudaMemsetAsync(hi.p, 0, pw * 4 * n, st));
    CU(cudaMemsetAsync(nz.p, 0, pw * 4 * n, st));
    if (W % 16 == 0) k_pack_bits<true, true><<<g, 256, 0, st>>>(mask, (uint32_t*)nz.p, (uint32_t*)hi.p, H, W, wpr);
    else k_pack_bits<false, true><<<g, 256, 0, st>>>(mask, (uint32_t*)nz.p, (uint32_t*)hi.p, H, W, wpr);
    CHECK_LAUNCH();
    rc = launch_degrade(nullptr, bgr, (const uint32_t*)hi.p, (const uint32_t*)nz.p, compressed, overlay, n, H, W, block_size, q,
                        flavour, (Counters*)counters, st);
    if (rc) return rc;
    if (counters) {
        k_counters_add<<<1, 1, 0, st>>>((Counters*)counters, (unsigned long long)n, (unsigned long long)n * H * W,
                                         (unsigned long long)n * ((H + block_size - 1) / block_size) * ((W + block_size - 1) / block_size));
        CHECK_LAUNCH();
    }
    return DVC_OK;
}

extern "C" int dvc_dct_blocks_f32(const float* src, float* dst, int64_t n, int32_t bh, int32_t bw, int32_t inverse, void* stream) {
    char* ERRBUF = nullptr;
    if (n < 0 || bh < 1 || bh > 8 || bw < 1 || bw > 8) return set_err(nullptr, DVC_ERR_INVALID, "dvc_dct_blocks_f32: n >= 0, block sides 1..8");
    if (n == 0) return DVC_OK;
    if (!src || !dst) return set_err(nullptr, DVC_ERR_INVALID, "dvc_dct_blocks_f32: null pointer");
    k_dct_blocks<<<(unsigned)cdiv((size_t)n, 128), 128, 0, (cudaStream_t)stream>>>(src, dst, (long long)n, bh, bw, inverse);
    CHECK_LAUNCH();
    return DVC_OK;
}

extern "C" int dvc_gaussian_blur_u8(const uint8_t* src, uint8_t* dst, int32_t n, int32_t H, int32_t W, int32_t ksize, double sigma,
                                    void* stream) {
    char* ERRBUF = nullptr;
    int rc = check_dims(n, H, W, "dvc_gaussian_blur_u8");
    if (rc || n == 0) return rc;
    if (!src || !dst) return set_err(nullptr, DVC_ERR_INVALID, "dvc_gaussian_blur_u8: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    ScopedAsyncBuf tmp(st);
    CU(tmp.alloc((size_t)n * H * W * 2));
    return launch_gaussian(nullptr, src, dst, (uint16_t*)tmp.p, n, H, W, ksize, sigma, st);
}

extern "C" int dvc_begin_stream_frames(dvc_handle* h, const uint8_t* first_frames_host) {
    char* ERRBUF = h ? h->err : nullptr;
    if (!h || !first_frames_host) return set_err(h ? h->err : nullptr, DVC_ERR_INVALID, "dvc_begin_stream_frames: null argument");
    CU(cudaSetDevice(h->cfg.device));
    CU(handle_join(h));
    const int S = h->S, H = h->H, W = h->W;
    cudaStream_t st = h->s_mask;
    ScopedAsyncBuf src(st), bgr(st), gray(st), tmp(st);
    CU(src.alloc((size_t)S * h->src_frame_bytes));
    CU(cudaMemcpyAsync(src.p, first_frames_host, (size_t)S * h->src_frame_bytes, cudaMemcpyHostToDevice, st));
    const uint8_t* frames = (const uint8_t*)src.p;
    if (h->resizing) {                                   // frame_differencing.py:74
        CU(bgr.alloc((size_t)S * h->frame_bytes));
        int rc = launch_resize(h->err, (const uint8_t*)src.p, (uint8_t*)bgr.p, S, h->cfg.src_height, h->cfg.src_width, H, W, 3,
                               resize_tables_view(h->resize_tables, H, W), st);
        if (rc) return rc;
        frames = (const uint8_t*)bgr.p;
    }
    dim3 g(cdiv((size_t)((W + 15) / 16) * H, 256), S);
    uint8_t* pg = h->prev_gray[h->cur];
    if (h->cfg.mode == DVC_MODE_FD) {                    // :75-77: gray, then GaussianBlur((25, 25), 30)
        CU(gray.alloc((size_t)S * h->plane_bytes));
        CU(tmp.alloc((size_t)S * h->plane_bytes * 2));
        if (h->aligned) k_bgr2gray<true><<<g, 256, 0, st>>>(frames, (uint8_t*)gray.p, H, W);
        else k_bgr2gray<false><<<g, 256, 0, st>>>(frames, (uint8_t*)gray.p, H, W);
        CHECK_LAUNCH();
        int rc = launch_gaussian(h->err, (const uint8_t*)gray.p, pg, (uint16_t*)tmp.p, S, H, W, 25, 30.0, st);
        if (rc) return rc;
    } else {                                             // motion_compression_opt.py:60: gray only
        if (h->aligned) k_bgr2gray<true><<<g, 256, 0, st>>>(frames, pg, H, W);
        else k_bgr2gray<false><<<g, 256, 0, st>>>(frames, pg, H, W);
        CHECK_LAUNCH();
    }
    if (h->acc) CU(cudaMemsetAsync(h->acc, 0, h->plane_bytes * S, st));
    if (h->ring) CU(cudaMemsetAsync(h->ring, 0, h->plane_words * 4 * h->ring_cap * S, st));
    h->n_masks = 0;
    CU(cudaStreamSynchronize(st));
    return DVC_OK;
}

// ------------------------------------------------------------------------------------------------
// Farneback flow (motion_compression_opt.py:72-83)
// ------------------------------------------------------------------------------------------------
struct FlowPlan {
    int levels = 0;                       // index of the coarsest level
    std::vector<FlowLevelGeom> geo;       // per level, 0 = full resolution
    std::vector<size_t> off;              // pixel offset of each level inside one frame's pyramid
    size_t P = 0;                         // pixels of all levels of one frame
    FlowPolyTab poly;
};

// getGaussianKernel(n, sigma, CV_32F): the small fixed kernels when sigma <= 0, float taps normalised in double
static void gauss_kernel_f32(int n, double sigma, float* half) {
    static const float fixed[4][7] = {{1.f}, {0.25f, 0.5f, 0.25f}, {0.0625f, 0.25f, 0.375f, 0.25f, 0.0625f},
                                      {0.03125f, 0.109375f, 0.21875f, 0.28125f, 0.21875f, 0.109375f, 0.03125f}};
    const bool use_fixed = n % 2 == 1 && n <= 7 && sigma <= 0;
    const double sx = sigma > 0 ? sigma : ((n - 1) * 0.5 - 1) * 0.3 + 0.8;
    const double scale2x = -0.5 / (sx * sx);
    std::vector<float> c(n);
    double sum = 0;
    for (int i = 0; i < n; ++i) {
        const double x = i - (n - 1) * 0.5;
        c[i] = (float)(use_fixed ? (double)fixed[n / 2][i] : std::exp(scale2x * x * x));
        sum += c[i];
    }
    sum = 1. / sum;
    for (int i = n / 2; i < n; ++i) half[i - n / 2] = (float)(c[i] * sum);
}

// FarnebackPrepareGaussian: float taps, the 6 x 6 Gram matrix in double and four entries of its inverse
static void flow_poly_tab(int n, double sigma, FlowPolyTab& t) {
    if (sigma < 1.1920928955078125e-07) sigma = n * 0.3;
    float g[2 * FLOW_MAX_POLY_N + 1];
    double s = 0;
    for (int x = -n; x <= n; ++x) { g[x + n] = (float)std::exp(-x * x / (2 * sigma * sigma)); s += g[x + n]; }
    s = 1. / s;
    for (int x = -n; x <= n; ++x) g[x + n] = (float)(g[x + n] * s);
    t.n = n;
    for (int k = 0; k <= n; ++k) { t.g[k] = g[k + n]; t.xg[k] = (float)k * g[k + n]; t.xxg[k] = (float)(k * k) * g[k + n]; }
    double G[6][12] = {};
    for (int y = -n; y <= n; ++y)
        for (int x = -n; x <= n; ++x) {
            const float gy = g[y + n], gx = g[x + n], fx = (float)x, fy = (float)y;
            G[0][0] += gy * gx;
            G[1][1] += gy * gx * fx * fx;
            G[3][3] += gy * gx * fx * fx * fx * fx;
            G[5][5] += gy * gx * fx * fx * fy * fy;
        }
    G[2][2] = G[0][3] = G[0][4] = G[3][0] = G[4][0] = G[1][1];
    G[4][4] = G[3][3];
    G[3][4] = G[4][3] = G[5][5];
    for (int i = 0; i < 6; ++i) G[i][6 + i] = 1.0;
    for (int c = 0; c < 6; ++c) {                         // Gauss-Jordan with partial pivoting (G is positive definite)
        int piv = c;
        for (int r = c + 1; r < 6; ++r) if (std::fabs(G[r][c]) > std::fabs(G[piv][c])) piv = r;
        for (int j = 0; j < 12; ++j) std::swap(G[c][j], G[piv][j]);
        const double d = G[c][c];
        for (int j = 0; j < 12; ++j) G[c][j] /= d;
        for (int r = 0; r < 6; ++r)
            if (r != c && G[r][c] != 0.0) {
                const double f = G[r][c];
                for (int j = 0; j < 12; ++j) G[r][j] -= f * G[c][j];
            }
    }
    t.ig11 = G[1][7]; t.ig03 = G[0][9]; t.ig33 = G[3][9]; t.ig55 = G[5][11];
}

static int cv_round(double v) { return (int)std::lrint(v); }

// Argument rules of both entry points, then the pyramid: cv2 stops adding levels once a side drops below 32 pixels.
static int flow_plan(const char* who, int n, int H, int W, double pyr_scale, int levels, int winsize, int iterations, int poly_n,
                     double poly_sigma, int flags, FlowPlan& pl) {
    if (n < 0 || H < 1 || W < 1) return set_err(nullptr, DVC_ERR_INVALID, "%s: bad dimensions n=%d H=%d W=%d", who, n, H, W);
    if (!(pyr_scale > 0 && pyr_scale < 1)) return set_err(nullptr, DVC_ERR_INVALID, "%s: pyr_scale %g outside (0, 1)", who, pyr_scale);
    if (levels < 0 || winsize < 1 || iterations < 1)
        return set_err(nullptr, DVC_ERR_INVALID, "%s: levels %d, winsize %d, iterations %d: need levels >= 0, winsize >= 1, iterations >= 1",
                       who, levels, winsize, iterations);
    if (!(poly_sigma >= 0) || !(poly_sigma < 1e6)) return set_err(nullptr, DVC_ERR_INVALID, "%s: poly_sigma %g", who, poly_sigma);
    if (poly_n != 5 && poly_n != 7) return set_err(nullptr, DVC_ERR_UNSUPPORTED, "%s: poly_n %d: the GPU path implements 5 and 7", who, poly_n);
    if (flags != 0)
        return set_err(nullptr, DVC_ERR_UNSUPPORTED, "%s: flags %d: OPTFLOW_USE_INITIAL_FLOW and OPTFLOW_FARNEBACK_GAUSSIAN are not implemented", who, flags);
    if (H > 32767 || W > 32767) return set_err(nullptr, DVC_ERR_UNSUPPORTED, "%s: image larger than 32767", who);
    if (winsize > 32767) return set_err(nullptr, DVC_ERR_UNSUPPORTED, "%s: winsize %d larger than 32767", who, winsize);
    double scale = 1;
    int k = 0;
    for (; k < levels; ++k) {
        scale *= pyr_scale;
        if (W * scale < 32 || H * scale < 32) break;
        if (k == 64) return set_err(nullptr, DVC_ERR_UNSUPPORTED, "%s: more than 64 pyramid levels", who);
    }
    pl.levels = k;
    pl.geo.assign(k + 1, FlowLevelGeom());
    pl.off.assign(k + 1, 0);
    pl.P = 0;
    for (int l = 0; l <= k; ++l) {
        double s = 1;
        for (int i = 0; i < l; ++i) s *= pyr_scale;
        const double sigma = (1. / s - 1) * 0.5;
        const int ks = std::max(cv_round(sigma * 5) | 1, 3);
        if (ks / 2 > FLOW_MAX_BLUR_HALF)
            return set_err(nullptr, DVC_ERR_UNSUPPORTED, "%s: level %d needs a %d-tap Gaussian, more than %d", who, l, ks, 2 * FLOW_MAX_BLUR_HALF + 1);
        FlowLevelGeom& g = pl.geo[l];
        gauss_kernel_f32(ks, sigma, g.k);
        g.half = ks / 2;
        g.w = cv_round(W * s);
        g.h = cv_round(H * s);
        g.scale_x = 1. / ((double)g.w / W);
        g.scale_y = 1. / ((double)g.h / H);
        pl.off[l] = pl.P;
        pl.P += (size_t)g.w * g.h;
    }
    flow_poly_tab(poly_n, poly_sigma, pl.poly);
    return DVC_OK;
}

// frames [F][H][W] -> their pyramids of polynomial coefficients, R [F][P][5]
static int flow_pyramids(const uint8_t* src, int F, int H, int W, const FlowPlan& pl, float* img, float* R, cudaStream_t st) {
    char* ERRBUF = nullptr;
    for (int l = 0; l <= pl.levels; ++l) {
        const FlowLevelGeom& g = pl.geo[l];
        k_flow_level<<<dim3(cdiv((size_t)g.w * g.h, 256), F), 256, 0, st>>>(src, H, W, img, (size_t)H * W, g);
        k_flow_poly<<<dim3(cdiv(g.w, POLY_TW), cdiv(g.h, POLY_TH), F), 256, 0, st>>>(img, (size_t)H * W, g.w, g.h, R + pl.off[l] * 5,
                                                                                    pl.P * 5, pl.poly);
        CHECK_LAUNCH();
    }
    return DVC_OK;
}

struct FlowScratch {
    float* img;       // [F][H][W] level image
    float* R;         // [F][P][5]
    float* M;         // [G][H][W][5]
    double* V;        // [G][H][W][5] column sums
    double* S;        // [G][H][W][5] box sums
    float2* fl[2];    // [G][H][W] flow of the last two levels
};

// G pairs, coarse to fine.  Pair p's polynomial pyramids are R0 + p * P * 5 and R1 + p * P * 5.  The finest level's last
// solve writes flow_out (stride H*W) or mask_out.
static int flow_pairs(const float* R0, const float* R1, int G, int H, int W, const FlowPlan& pl, double pyr_scale, int winsize,
                      int iterations, const FlowScratch& sc, float2* flow_out, uint8_t* mask_out, float thr, cudaStream_t st) {
    char* ERRBUF = nullptr;
    const size_t WH = (size_t)H * W;
    const int m = winsize / 2;
    const double box = 1. / ((double)winsize * winsize);
    const float up = (float)(1. / pyr_scale);
    const float2* coarse = nullptr;
    int cw = 0, ch = 0, cur = 0;
    for (int l = pl.levels; l >= 0; --l) {
        const FlowLevelGeom& g = pl.geo[l];
        const FlowPair pr{R0 + pl.off[l] * 5, R1 + pl.off[l] * 5, pl.P * 5, WH, g.w, g.h};
        const dim3 gp(cdiv((size_t)g.w * g.h, 256), G);
        k_flow_matrices<<<gp, 256, 0, st>>>(pr, coarse, cw, ch, coarse ? 1. / ((double)g.w / cw) : 0., coarse ? 1. / ((double)g.h / ch) : 0.,
                                            up, sc.M);
        CHECK_LAUNCH();
        for (int it = 0; it < iterations; ++it) {
            const bool last = it == iterations - 1;
            float2* fo = last ? sc.fl[cur] : nullptr;
            uint8_t* mo = nullptr;
            if (last && l == 0) { fo = flow_out; mo = mask_out; }
            k_flow_vsum<<<dim3(cdiv((size_t)g.w * 5, 128), G), 128, 0, st>>>(sc.M, sc.V, g.w, g.h, m, WH);
            k_flow_hsum<<<dim3(cdiv((size_t)g.h * 5, 128), G), 128, 0, st>>>(sc.V, sc.S, g.w, g.h, m, WH);
            k_flow_solve<<<gp, 256, 0, st>>>(pr, sc.S, box, fo, WH, mo, WH, thr, last ? nullptr : sc.M);
            CHECK_LAUNCH();
        }
        coarse = sc.fl[cur];
        cw = g.w; ch = g.h;
        cur ^= 1;
    }
    return DVC_OK;
}

// Pairs per launch group: scratch for one group stays near 1 GiB.
static int flow_group(int n, int H, int W, const FlowPlan& pl) {
    const size_t WH = (size_t)H * W;
    const size_t per_pair = 2 * (pl.P * 20 + WH * 4) + WH * (20 + 80 + 16);
    return (int)std::max<size_t>(1, std::min<size_t>({(size_t)n, ((size_t)1 << 30) / per_pair, 4096}));
}

static int flow_alloc(ScopedAsyncBuf* b, int F, int G, int H, int W, const FlowPlan& pl, FlowScratch& sc) {
    char* ERRBUF = nullptr;
    const size_t WH = (size_t)H * W;
    CU(b[0].alloc((size_t)F * WH * 4));
    CU(b[1].alloc((size_t)F * pl.P * 20));
    CU(b[2].alloc((size_t)G * WH * 20));
    CU(b[3].alloc((size_t)G * WH * 80));
    CU(b[4].alloc((size_t)G * WH * 16));
    sc.img = (float*)b[0].p; sc.R = (float*)b[1].p; sc.M = (float*)b[2].p; sc.V = (double*)b[3].p; sc.S = sc.V + (size_t)G * WH * 5;
    sc.fl[0] = (float2*)b[4].p; sc.fl[1] = sc.fl[0] + (size_t)G * WH;
    return DVC_OK;
}

extern "C" int dvc_farneback_flow_f32(const uint8_t* prev, const uint8_t* next, float* flow, int32_t n, int32_t H, int32_t W,
                                      double pyr_scale, int32_t levels, int32_t winsize, int32_t iterations, int32_t poly_n,
                                      double poly_sigma, int32_t flags, void* stream) {
    FlowPlan pl;
    int rc = flow_plan("dvc_farneback_flow_f32", n, H, W, pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags, pl);
    if (rc || n == 0) return rc;
    if (!prev || !next || !flow) return set_err(nullptr, DVC_ERR_INVALID, "dvc_farneback_flow_f32: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t WH = (size_t)H * W;
    const int G = flow_group(n, H, W, pl);
    ScopedAsyncBuf b[5] = {ScopedAsyncBuf(st), ScopedAsyncBuf(st), ScopedAsyncBuf(st), ScopedAsyncBuf(st), ScopedAsyncBuf(st)};
    FlowScratch sc;
    if ((rc = flow_alloc(b, 2 * G, G, H, W, pl, sc))) return rc;
    float* R1 = sc.R + (size_t)G * pl.P * 5;
    for (int i0 = 0; i0 < n; i0 += G) {
        const int g = std::min(G, n - i0);
        if ((rc = flow_pyramids(prev + i0 * WH, g, H, W, pl, sc.img, sc.R, st))) return rc;
        if ((rc = flow_pyramids(next + i0 * WH, g, H, W, pl, sc.img, R1, st))) return rc;
        if ((rc = flow_pairs(sc.R, R1, g, H, W, pl, pyr_scale, winsize, iterations, sc, (float2*)flow + i0 * WH, nullptr, 0.f, st))) return rc;
    }
    return DVC_OK;
}

extern "C" int dvc_flow_masks_u8(const uint8_t* gray, uint8_t* mask, int32_t n, int32_t H, int32_t W, double pyr_scale, int32_t levels,
                                 int32_t winsize, int32_t iterations, int32_t poly_n, double poly_sigma, int32_t flags,
                                 float flow_threshold, void* stream) {
    char* ERRBUF = nullptr;
    FlowPlan pl;
    int rc = flow_plan("dvc_flow_masks_u8", n, H, W, pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags, pl);
    if (rc || n == 0) return rc;
    if (!gray || !mask) return set_err(nullptr, DVC_ERR_INVALID, "dvc_flow_masks_u8: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t WH = (size_t)H * W, RF = pl.P * 5;
    const int G = flow_group(n, H, W, pl);
    ScopedAsyncBuf b[5] = {ScopedAsyncBuf(st), ScopedAsyncBuf(st), ScopedAsyncBuf(st), ScopedAsyncBuf(st), ScopedAsyncBuf(st)};
    FlowScratch sc;
    if ((rc = flow_alloc(b, G + 1, G, H, W, pl, sc))) return rc;
    // frame i + 1's pyramid serves pair i and pair i + 1: the last frame of a group moves to slot 0 for the next group
    if ((rc = flow_pyramids(gray, 1, H, W, pl, sc.img, sc.R, st))) return rc;
    for (int i0 = 0; i0 < n; i0 += G) {
        const int g = std::min(G, n - i0);
        if (i0 > 0) CU(cudaMemcpyAsync(sc.R, sc.R + (size_t)G * RF, RF * sizeof(float), cudaMemcpyDeviceToDevice, st));
        if ((rc = flow_pyramids(gray + (i0 + 1) * WH, g, H, W, pl, sc.img, sc.R + RF, st))) return rc;
        if ((rc = flow_pairs(sc.R, sc.R + RF, g, H, W, pl, pyr_scale, winsize, iterations, sc, nullptr, mask + i0 * WH, flow_threshold, st)))
            return rc;
    }
    return DVC_OK;
}
