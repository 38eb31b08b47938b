/* dvc_b200.h -- C ABI of the B200-native frame-differencing hot loop.
 *
 * This is the drop-in boundary for the per-frame loop of the reference
 * (carlozamu/dynamic-video-compression-surveillance).  The reference has no FFI
 * of its own: every arithmetic step is a cv2/numpy call made from Python.  Each
 * entry point below therefore cites the reference lines (file:line under
 * /root/reference) whose arithmetic it replaces.  The Python host shim
 * (dynamic_video_compression_surveillance_b200/dropin/frame_differencing.py)
 * binds these with ctypes; INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++/torch types.
 *   - Every function returns 0 on success or a negative DVC_ERR_* code; no C++
 *     exception crosses the boundary.  dvc_last_error() gives the message.
 *   - Images are C-contiguous uint8, [H][W] (planes) or [H][W][3] in BGR order,
 *     exactly the numpy layout cv2 hands the reference.
 *   - "dev" pointers are device pointers; a `stream` argument is a cudaStream_t
 *     passed as void* (NULL = the legacy default stream).  Device-pointer calls
 *     are asynchronous on that stream.
 *   - A handle is used by one host thread at a time; handles are independent.
 *   - There is no CPU fallback: without a CUDA device every call fails with
 *     DVC_ERR_CUDA.
 */
#ifndef DVC_B200_H
#define DVC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DVC_ABI_VERSION 3

enum {
    DVC_OK = 0,
    DVC_ERR_INVALID = -1,     /* bad argument */
    DVC_ERR_UNSUPPORTED = -2, /* valid for the reference, not implemented on the GPU path */
    DVC_ERR_CUDA = -3,        /* CUDA runtime error (message has the cudaError string) */
    DVC_ERR_NOMEM = -4
};

/* Which loop a handle runs. */
enum {
    /* frame_differencing.py:85-133 exactly: gray -> GaussianBlur 5x5 -> absdiff -> threshold ->
     * contour filter -> dilate -> addWeighted EMA -> overlay + block-DCT degrade. */
    DVC_MODE_FD = 0,
    /* The loop BASELINE.json's north_star names: gray -> absdiff -> threshold
     * (frame_differencing.py:92,96-97) -> K-frame window vote -> close/open
     * (motion_compression_opt.py:61-62,84-90) -> dilate -> overlay + block-DCT degrade
     * (frame_differencing.py:106,110-130). */
    DVC_MODE_WINDOW = 1
};

enum { DVC_MORPH_ERODE = 0, DVC_MORPH_DILATE = 1, DVC_MORPH_OPEN = 2, DVC_MORPH_CLOSE = 3 };
enum { DVC_SHAPE_RECT = 0, DVC_SHAPE_ELLIPSE = 1 };
/* Degrade flavour: FD = frame_differencing.py:115-130 (luma only, chroma -> 128);
 * MCO = motion_compression_opt.py:152-183 (8x8, three channels, re-gray, full blocks only). */
enum { DVC_DEGRADE_FD = 0, DVC_DEGRADE_MCO = 1 };

typedef struct dvc_config {
    int32_t width, height;        /* frame size after the reference's resize (frame_differencing.py:59-60); any size >= 1:
                                   * blocks clipped by the frame edge are handled as the reference slices them (:117-121) */
    int32_t mode;                 /* DVC_MODE_* */
    int32_t block_size;           /* frame_differencing.py:22 (4); 1..8 (4 and 8 have the fast kernels) */
    float   motion_threshold;     /* frame_differencing.py:24 (0.5); cv2.threshold floors it */
    double  min_area;             /* frame_differencing.py:25 (500) */
    int32_t kernel_size;          /* frame_differencing.py:26 (7): k x k ones, dilate; 0 = skip (window mode) */
    double  release_factor;       /* frame_differencing.py:27 (0.5): addWeighted alpha; beta = 1 - alpha */
    float   quantization_level;   /* frame_differencing.py:28 (100) */
    int32_t window_size;          /* motion_compression_opt.py:30 window_size (30), <= 127 */
    double  alpha_fraction;       /* motion_compression_opt.py:29 alpha_fraction (0.2) */
    int32_t morph_kernel;         /* motion_compression_opt.py:30 morph_kernel (2); 0 = skip open/close */
    int32_t morph_shape;          /* DVC_SHAPE_ELLIPSE as in motion_compression_opt.py:62 */
    int32_t max_batch;            /* frames per device batch / pipelined host chunk (>= 1) */
    int32_t device;               /* CUDA device ordinal */
    int32_t src_width, src_height; /* 0, or the size of the frames handed to dvc_process_host when it differs from
                                    * width x height: the library then does the reference's cv2.resize (default
                                    * INTER_LINEAR, frame_differencing.py:74,91) on the GPU after the upload */
    int32_t n_streams;            /* 0 or 1: one stream.  S > 1: a lock-step group of S independent camera streams (the reference
                                   * loops over files one by one, windows.py:142-160; BASELINE config 4) that share every kernel
                                   * launch.  Each call then advances every stream by n_frames: frame / output buffers are
                                   * [S][n_frames][H][W](x3), dvc_begin_stream takes [S][H][W] planes, state blobs and counters
                                   * cover all S streams. */
} dvc_config;

typedef struct dvc_handle dvc_handle;

/* Counters accumulated by the degrade kernel (the in-loop statistics north_star asks for; the
 * reference only derives a file-size percentage after the fact, performance_analysis.py:195-204). */
typedef struct dvc_counters {
    uint64_t frames;         /* frames processed (frame_differencing.py:134 frame_count) */
    uint64_t pixels;         /* frames * H * W */
    uint64_t motion_pixels;  /* pixels painted red in the overlay: acc > 127 (frame_differencing.py:111) */
    uint64_t blocks;         /* blocks visited (frame_differencing.py:117-118) */
    uint64_t static_blocks;  /* blocks whose mask block is all zero and were degraded (:120) */
} dvc_counters;

int         dvc_abi_version(void);
/* 1 for the -DDVC_MEASURE flavour (tools/: environment switches select kernel generations and copy-only probes, outputs may
 * be wrong), 0 for the product library, which reads no environment variable at all. */
int         dvc_measure_build(void);
const char* dvc_last_error(const dvc_handle* h);   /* h may be NULL: error of the last failed create / stage call */
void        dvc_default_config(dvc_config* cfg);   /* the reference's defaults, mode FD */

/* ---- per-stream state: prev_gray, accumulated_mask / mask_queue (frame_differencing.py:75-81,
 *      motion_compression_opt.py:60-61) ---------------------------------------------------------- */
int dvc_create(const dvc_config* cfg, dvc_handle** out);
int dvc_destroy(dvc_handle* h);
/* Seed prev_gray from a HOST plane [H][W] (frame_differencing.py:75-77: the first frame's gray after
 * the (25,25),sigma=30 blur, which stays on the host; motion_compression_opt.py:60 in window mode) and
 * clear accumulated_mask / the mask window.  Synchronous. */
int dvc_begin_stream(dvc_handle* h, const uint8_t* prev_gray_host);
/* The same from the first FRAME(S) of the stream(s), HOST [S][src_h][src_w][3] BGR as decoded: the library does the
 * reference's first-frame work on the GPU -- cv2.resize when cfg.src_width / src_height are set (frame_differencing.py:74),
 * BGR2GRAY (:75) and, in FD mode, GaussianBlur((25, 25), 30) (:77; OpenCV's fixed-point Gaussian, bit for bit) -- and
 * clears accumulated_mask / the mask window.  Synchronous. */
int dvc_begin_stream_frames(dvc_handle* h, const uint8_t* first_frames_host);
/* Chunk hand-off (SURVEY.md section 8e): serialise / restore prev_gray + EMA plane or mask window.
 * Query the size with dvc_state_bytes().  Synchronous, host buffers. */
size_t dvc_state_bytes(const dvc_handle* h);
int dvc_get_state(dvc_handle* h, void* host_buf, size_t bytes);
int dvc_set_state(dvc_handle* h, const void* host_buf, size_t bytes);
int dvc_get_counters(dvc_handle* h, dvc_counters* out);   /* synchronises the handle's streams */
int dvc_reset_counters(dvc_handle* h);

/* ---- the loop body: frame_differencing.py:85-133 for n_frames consecutive frames ----------------
 * frames_dev   [n][H][W][3]  input frames (after cap.read(), frame_differencing.py:87)
 * overlay_dev  [n][H][W][3]  what mask_out.write() receives (:110-112), may be NULL
 * compressed_dev [n][H][W][3] what final_out.write() receives (:115-131), may be NULL
 * mask_dev     [n][H][W]     accumulated_mask after each frame (FD) / final mask (WINDOW), may be NULL
 * n_frames <= cfg.max_batch.  When W % 16 == 0, frames_dev must be 16-byte aligned: the front kernels load it
 * 16 bytes at a time. */
int dvc_process_batch(dvc_handle* h, const uint8_t* frames_dev, int32_t n_frames, uint8_t* overlay_dev,
                      uint8_t* compressed_dev, uint8_t* mask_dev, void* stream);
/* Software pipelining across batches (off by default).  When on, dvc_process_batch runs the mask kernels and the
 * degrade kernel on two internal streams so that the mask kernels of batch c+1 overlap the degrade kernel of
 * batch c.  Each batch is still ordered after the work already queued in `stream`, but `stream` is re-joined
 * only by dvc_flush(): input and output buffers must stay untouched until then. */
int dvc_set_overlap(dvc_handle* h, int32_t on);
int dvc_flush(dvc_handle* h, void* stream);     /* make `stream` wait for every batch issued so far */
/* Same loop with HOST buffers (pinned for full speed): frames are uploaded, processed and the results
 * downloaded in chunks of min(cfg.max_batch, 8) frames, double-buffered on the handle's own copy/compute
 * streams.  With cfg.src_width / src_height set, frames_host holds frames of that size and the library does the
 * reference's cv2.resize (frame_differencing.py:91) after the upload; the outputs are width x height.
 * Returns after everything has landed in the host buffers.  Any n_frames >= 0. */
int dvc_process_host(dvc_handle* h, const uint8_t* frames_host, int64_t n_frames, uint8_t* overlay_host,
                     uint8_t* compressed_host, uint8_t* mask_host);

/* ---- measurement hooks (bench.py): per kernel group, time between CUDA events recorded on the launching
 *      stream around the group's launches inside dvc_process_batch / dvc_process_host ------------- */
enum {
    DVC_PROF_FRONT = 0,   /* K1: gray (+blur5) (+absdiff+threshold in window mode) */
    DVC_PROF_DIFF = 1,    /* K1 fd mode: absdiff + threshold on blurred planes */
    DVC_PROF_VOTE = 2,    /* K2: window vote */
    DVC_PROF_EMA = 3,     /* K2: addWeighted EMA */
    DVC_PROF_MORPH = 4,   /* K3: morphology chain */
    DVC_PROF_CCL = 5,     /* contour filter */
    DVC_PROF_DEGRADE = 6, /* K4: overlay + degrade + statistics */
    DVC_PROF_MISC = 7,    /* mask unpacking for callers that ask for uint8 masks */
    DVC_PROF_KERNELS = 8
};
int     dvc_profile_enable(dvc_handle* h, int32_t on);
/* Synchronises, sums the recorded intervals per group (milliseconds, launches) and clears the records. */
int     dvc_profile_read(dvc_handle* h, double* ms_by_kernel, int64_t* launches_by_kernel, int32_t n_kernels);
int64_t dvc_launch_count(const dvc_handle* h);   /* kernels launched by this handle's loop so far */

/* ---- stage-level entry points (one per cv2 call; device pointers; used by the parity tests and
 *      available to callers that want a single op) ------------------------------------------------ */
/* cv2.cvtColor(BGR2GRAY), frame_differencing.py:75,92.  n images. */
int dvc_bgr2gray_u8(const uint8_t* bgr_dev, uint8_t* gray_dev, int32_t n, int32_t H, int32_t W, void* stream);
/* cvtColor + [GaussianBlur 5x5] + absdiff + threshold, frame_differencing.py:92-97, for n consecutive
 * frames.  prev_gray_dev [H][W] is the (blurred) gray of the frame before bgr_dev[0]; frame i > 0
 * differences against frame i-1.  gray_out_dev [n][H][W] (the new prev_gray values) and/or
 * mask_out_dev [n][H][W] (0/255) may be NULL. */
int dvc_gray_absdiff_thresh_u8(const uint8_t* bgr_dev, const uint8_t* prev_gray_dev, uint8_t* gray_out_dev,
                               uint8_t* mask_out_dev, int32_t n, int32_t H, int32_t W, float motion_threshold,
                               int32_t blur5, void* stream);
/* deque(maxlen=K) + np.sum + compare, motion_compression_opt.py:61,84-86, for n consecutive 0/non-zero
 * masks starting from an empty window. */
int dvc_temporal_ring_u8(const uint8_t* masks_dev, uint8_t* smoothed_dev, int32_t n, int32_t H, int32_t W,
                         int32_t window_size, double alpha_fraction, void* stream);
/* cv2.addWeighted(acc, rf, dilated, 1 - rf, 0), frame_differencing.py:107, for n consecutive dilated masks
 * (0/255).  acc_inout_dev [H][W] is read and left at its final value; acc_all_dev [n][H][W] may be NULL. */
int dvc_temporal_ema_u8(uint8_t* acc_inout_dev, const uint8_t* dilated_dev, uint8_t* acc_all_dev, int32_t n,
                        int32_t H, int32_t W, double release_factor, void* stream);
/* cv2.erode / cv2.dilate / cv2.morphologyEx(OPEN|CLOSE) on binary (0 / non-zero) masks,
 * frame_differencing.py:106, motion_compression_opt.py:89-90.  k x k rect (np.ones) or
 * getStructuringElement(MORPH_ELLIPSE); k <= 33.  n images. */
int dvc_morph_u8(const uint8_t* src_dev, uint8_t* dst_dev, int32_t n, int32_t H, int32_t W, int32_t op,
                 int32_t shape, int32_t k, void* stream);
/* findContours(RETR_EXTERNAL) + contourArea > min_area + drawContours(FILLED),
 * frame_differencing.py:100-104.  n images. */
int dvc_contour_filter_u8(const uint8_t* src_dev, uint8_t* dst_dev, int32_t n, int32_t H, int32_t W,
                          double min_area, void* stream);
/* cv2.resize(src, (dst_w, dst_h)) with the default INTER_LINEAR on uint8, frame_differencing.py:74,91 (scale_factor != 1):
 * OpenCV's 11-bit fixed-point bilinear, bit for bit.  n images [src_h][src_w][channels] -> [dst_h][dst_w][channels],
 * channels 1 or 3. */
int dvc_resize_linear_u8(const uint8_t* src_dev, uint8_t* dst_dev, int32_t n, int32_t src_h, int32_t src_w, int32_t dst_h,
                         int32_t dst_w, int32_t channels, void* stream);
/* findContours(RETR_EXTERNAL) + boundingRect + rectangle((x, y), (x + w, y + h), 255, FILLED),
 * motion_compression_opt.py:93-97: every 8-connected component is replaced by its bounding rectangle
 * grown by one column and one row (cv2.rectangle includes both corners), clipped to the image.  n images. */
int dvc_mask_rectangles_u8(const uint8_t* src_dev, uint8_t* dst_dev, int32_t n, int32_t H, int32_t W, void* stream);
/* overlay paint + colour round trip + block-DCT degrade, frame_differencing.py:110-111,115-130
 * (flavour FD) or motion_compression_opt.py:152-183 (flavour MCO).  mask_dev [n][H][W] is
 * accumulated_mask (any uint8 values).  Either output may be NULL.  counters_dev (5 x uint64 in
 * dvc_counters order, accumulated atomically) may be NULL.  bgr_dev, compressed_dev and overlay_dev may have
 * any alignment; 16-byte aligned pointers take the fastest kernels. */
int dvc_degrade_blend_u8(const uint8_t* bgr_dev, const uint8_t* mask_dev, uint8_t* compressed_dev,
                         uint8_t* overlay_dev, int32_t n, int32_t H, int32_t W, int32_t block_size,
                         float quantization_level, int32_t flavour, uint64_t* counters_dev, void* stream);

/* cv2.GaussianBlur(src, (ksize, ksize), sigma) on n uint8 planes [H][W], default border (REFLECT_101), ksize odd <= 33:
 * frame_differencing.py:77 ((25, 25), 30) and :93 ((5, 5), 0); OpenCV's 8.8 fixed-point kernel and rounding, bit for bit. */
int dvc_gaussian_blur_u8(const uint8_t* src_dev, uint8_t* dst_dev, int32_t n, int32_t H, int32_t W, int32_t ksize, double sigma,
                         void* stream);
/* cv2.dct / cv2.idct on n float32 blocks [n][bh][bw] (bh, bw in 1..8), frame_differencing.py:122,124 and
 * motion_compression_opt.py:165,167: the transform pair the degrade kernels apply, bit for bit (8 x 8 is cv2's
 * dedicated 2-D routine, every other shape rows-then-columns through the 1-D routine of each length). */
int dvc_dct_blocks_f32(const float* src_dev, float* dst_dev, int64_t n, int32_t bh, int32_t bw, int32_t inverse,
                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DVC_B200_H */
