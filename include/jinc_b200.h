/*
 * jinc_b200.h -- C ABI of the B200-native EWA-Jinc resampling path (libjinc_b200.so).
 *
 * This is the drop-in boundary between a host-side plugin (AviSynth+ C plugin in
 * avisynth-jincresize_b200/plugin/, or any FFI binding) and the sm_100a kernels.  Plain C:
 * opaque handles, plain pointers, sizes and pitches in bytes; no C++ types, no exceptions, no torch
 * types.  Every call returns 0 on success or a negative JINC_E_* code, with a human-readable
 * message available from jinc_last_error() (thread-local).
 *
 * Each entry point names the reference interface it replaces (paths relative to the reference
 * repository, Asd-g/AviSynth-JincResize v2.1.4).  There is NO CPU fallback: every compute entry
 * point fails with JINC_E_CUDA when no CUDA device is usable.
 */
#ifndef JINC_B200_H
#define JINC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define JINC_API __attribute__((visibility("default")))

#define JINC_ABI_VERSION 2
#define JINC_LUT_SAMPLES 1024 /* src/JincResize.cpp:795 `samples` */
#define JINC_MAX_PLANES 4
#define JINC_MAX_DEVICES 16

enum {
    JINC_OK = 0,
    JINC_E_INVALID = -1, /* bad argument */
    JINC_E_CUDA = -2,    /* CUDA runtime/driver error, or no device */
    JINC_E_NOMEM = -3,
    JINC_E_UNSUPPORTED = -4,
    JINC_E_BUSY = -5     /* jinc_filter_try_submit: every in-flight slot is taken */
};

/* Sample format of an IEEE binary16 (half-precision float) plane, accepted wherever the ABI takes `sample_bytes`
 * (jinc_filter_params.sample_bytes with bits = 16, jinc_resize_plane_device with peak ignored).  The low byte is the
 * sample size.  Half planes are resampled like float planes: every sample is widened to float exactly, the sum is
 * accumulated in float in the same order as for a float plane, and the result is rounded to the nearest half (ties to
 * even) with no clamp: sums of magnitude 65520 or more become +-Inf, NaN and Inf inputs propagate.  So a half frame
 * equals the float frame of the widened input, rounded to half. */
#define JINC_SAMPLE_F16 0x102

/* chroma sample location (src/JincResize.cpp:715-745; README "cplace") */
enum { JINC_CPLACE_MPEG2 = 0, JINC_CPLACE_MPEG1 = 1, JINC_CPLACE_TOPLEFT = 2 };

typedef struct jinc_ctx jinc_ctx;       /* one GPU: device id, streams, scratch */
typedef struct jinc_table jinc_table;   /* device-resident coefficient table of one plane geometry */
typedef struct jinc_filter jinc_filter; /* one filter instance: tables + frame pipeline over >=1 GPUs */

JINC_API int jinc_abi_version(void);
JINC_API const char* jinc_last_error(void);
/* number of usable CUDA devices (0 when none; never negative) */
JINC_API int jinc_device_count(void);

/* ---------------------------------------------------------------- Jinc math / LUT (host, FP64)
 * Replaces: jinc_zeros[] (src/JincResize.cpp:84-102), jinc_sqr (:200-245),
 *           Lut::InitLut (:265-275).                                                         */
JINC_API double jinc_radius_for_tap(int tap); /* 0.0 when tap is outside 1..16 */
JINC_API double jinc_eval_sqr(double x2);     /* jinc(sqrt(x2)) */
/* lut[JINC_LUT_SAMPLES] doubles; blur == 0 means 1.0 (src/JincResize.cpp:772-774) */
JINC_API int jinc_lut_build(double radius, double blur, double* lut);

/* ---------------------------------------------------------------- device context */
JINC_API int jinc_ctx_create(int device, jinc_ctx** out);
JINC_API void jinc_ctx_destroy(jinc_ctx* ctx);
JINC_API int jinc_ctx_device(const jinc_ctx* ctx);

/* ---------------------------------------------------------------- coefficient tables (device kernels)
 * Replaces: generate_coeff_params (src/JincResize.cpp:315-333), init_coeff_table (:286-306),
 *           generate_coeff_table_c (:336-533), delete_coeff_table (:308-313).
 * initial_capacity / initial_factor have no counterpart: they only steer the reference's host
 * arena growth (:369-376,458-475) and never change results.                                  */
typedef struct jinc_table_params {
    int32_t quant_x, quant_y; /* 1..256 */
    int32_t src_w, src_h, dst_w, dst_h;
    double radius; /* jinc_radius_for_tap(tap) */
    double blur;   /* as given by the script (0 => 1.0) */
    double crop_left, crop_top, crop_w, crop_h;
} jinc_table_params;

/* how the resample kernels will walk this table */
enum {
    JINC_PATH_GENERAL = 0,   /* one thread per output sample, weights gathered per sample */
    JINC_PATH_UP2X = 1,      /* exact 2x upscale: 2x2 phase classes, register-tiled FFMA2 kernel */
    JINC_PATH_DOWN_INT = 2,  /* integer-ratio downscale: one phase, polyphase register-tiled kernel */
    JINC_PATH_PERIODIC = 3,  /* exactly periodic rational ratio (2:3, e.g. 1080p -> 720p): P x P passes of the polyphase kernel */
    JINC_PATH_CELLS = 4      /* rational ratio P:Q with piecewise-periodic phases (3:2 = 720p -> 1080p, 4:3, 3x, 4x): one
                                thread per chunk of cells, one weight block per residue pair held in registers */
};

typedef struct jinc_table_info {
    int32_t filter_size;   /* EWAPixelCoeff::filter_size (src/JincResize.h:23) */
    int32_t n_phase_x;     /* distinct quantised x phases among non-border columns */
    int32_t n_phase_y;
    int32_t n_border_cols; /* columns whose window was clamped (src/JincResize.cpp:395-418) */
    int32_t n_border_rows;
    int32_t fast_path;     /* JINC_PATH_* chosen for the interior */
    int32_t interior_x0, interior_x1, interior_y0, interior_y1; /* output rectangle run by the fast path */
    float filter_support;  /* src/JincResize.cpp:355 */
    float build_ms;        /* host wall time of jinc_table_create: LUT + device kernels + plans (the reference's
                              generate_coeff_table_c call, src/JincResize.cpp:829,864) */
    int32_t up2x_taps;     /* JINC_PATH_UP2X: taps per 2x2 output cell the kernel multiplies on 8/16-bit planes (4 * fs^2
                              unless exactly-zero taps are skipped); 0 on the other paths */
} jinc_table_info;

JINC_API int jinc_table_create(jinc_ctx* ctx, const jinc_table_params* p, jinc_table** out);
JINC_API void jinc_table_destroy(jinc_table* t);
JINC_API int jinc_table_get_info(const jinc_table* t, jinc_table_info* info);

/* Parity/introspection views (device -> host copies).  The reference stores, per output pixel,
 * {start_x, start_y, coeff_meta} (EWAPixelCoeffMeta, src/JincResize.h:11-16); positions are separable
 * (:363-364,524-528), so the device table keeps them per axis.
 * axis 0 = x (n = dst_w), axis 1 = y (n = dst_h).  Any output pointer may be NULL.
 *   start[i]  : window origin written to meta (:420-421)
 *   phase[i]  : quantised phase value q_int % quant (:426-427)
 *   border[i] : 1 when the window was clamped on this axis (:395-418)
 *   pos[i]    : accumulated float position xpos / ypos (:363-364,524,527)                       */
JINC_API int jinc_table_axis(const jinc_table* t, int axis, int32_t* start, int32_t* phase, uint8_t* border, float* pos);
/* filter_size*filter_size normalised weights the kernels apply at output pixel (x, y): the shared phase
 * block for interior pixels, per-pixel weights for border pixels (:443-514).  Row-major, no padding. */
JINC_API int jinc_table_pixel_weights(const jinc_table* t, int x, int y, float* weights);
/* block id of pixel (x,y): equal ids <=> the reference gives both pixels the same coeff_meta offset.
 * Border pixels get a unique negative id. */
JINC_API int jinc_table_pixel_block(const jinc_table* t, int x, int y, int64_t* block_id);

/* ---------------------------------------------------------------- resampling, device-resident planes
 * Replaces: JincResize::resize_plane_c<T,thr,subsampled> inner loops (src/JincResize.cpp:560-587) and its
 * SIMD siblings (src/resize_plane_{sse41,avx2,avx512}.cpp) for ONE plane.
 * sample_bytes: 1 (uint8), 2 (uint16, 10..16 bit), 4 (float) or JINC_SAMPLE_F16 (half).  peak: (1<<bits)-1 for
 * integer samples (clamp + round-half-even, :581-582); ignored for float and half (:583-584).
 * d_src/d_dst are device pointers, pitches in bytes; `stream` is a cudaStream_t (NULL = the context's
 * own stream).  Asynchronous with respect to the host.                                            */
JINC_API int jinc_resize_plane_device(jinc_ctx* ctx, const jinc_table* t, int sample_bytes, float peak,
                                      const void* d_src, ptrdiff_t src_pitch, void* d_dst, ptrdiff_t dst_pitch,
                                      void* stream);
/* number of kernel launches the call above issues for this table (fast-path interior + border strips) */
JINC_API int jinc_table_launches_per_plane(const jinc_table* t);
/* n_planes planes of one geometry; plane i at d_src + i*src_plane_stride / d_dst + i*dst_plane_stride (bytes).
 * Byte-identical to n_planes calls of jinc_resize_plane_device; one launch per kernel for the whole batch (planes are grouped
 * by up to four per record, in chunks of at most 65535 records).  Same sample_bytes, peak, pitch and alignment rules as
 * jinc_resize_plane_device; the destination plane stride must also be a multiple of 16 when n_planes > 1.  The device
 * array of plane records a launch reads comes from a small ring owned by ctx, whose entries are not reused before that
 * launch has finished, so calls may use different streams.  Asynchronous on `stream` (NULL = the context's stream). */
JINC_API int jinc_resize_planes_device(jinc_ctx* ctx, const jinc_table* t, int sample_bytes, float peak, int n_planes,
                                       const void* d_src, ptrdiff_t src_pitch, ptrdiff_t src_plane_stride,
                                       void* d_dst, ptrdiff_t dst_pitch, ptrdiff_t dst_plane_stride, void* stream);
/* Adjoint of n_planes float32 gradient planes of the table's output size into float32 planes of its source size (no
 * reference counterpart).  The resampler is a fixed linear map out = A * src; this computes A^T g:
 *   grad_src[sy][sx] = sum over outputs (x, y) with start_x[x] <= sx < start_x[x]+fs and start_y[y] <= sy < start_y[y]+fs
 *                      of w_{x,y}[sy - start_y[y]][sx - start_x[x]] * g[y][x]
 * with start_x / start_y the window origins (jinc_table_axis) and w_{x,y} the weights of output (x, y)
 * (jinc_table_pixel_weights), fs the filter size.
 *  - Canonical order: output rows y ascending, within a row x ascending, acc = fmaf(w, g, acc) from 0.  Every kernel uses
 *    it, so a source sample's bits do not depend on which kernel, tile, batch position or launch computed it.
 *  - Every covering tap is multiplied, zero weights included: an Inf or NaN in g reaches every source sample of that
 *    output's fs x fs window.
 *  - Samples no output covers (outside a crop) are written as 0: every sample of grad_src is written, nothing accumulates.
 *  - Gradients are float32 whatever the forward sample type; for integer planes this is the transpose of the linear map,
 *    without the forward's rounding and clamping.
 * 4-byte alignment and pitches only; pitches must hold a row and, when n_planes > 1, plane strides a plane.  d_grad_src
 * must not overlap d_grad_dst.  Asynchronous on `stream` (NULL = the context's stream). */
JINC_API int jinc_resize_adjoint_planes_device(jinc_ctx* ctx, const jinc_table* t, int n_planes,
                                               const float* d_grad_dst, ptrdiff_t grad_dst_pitch, ptrdiff_t grad_dst_plane_stride,
                                               float* d_grad_src, ptrdiff_t grad_src_pitch, ptrdiff_t grad_src_plane_stride,
                                               void* stream);
/* Anti-ringing clamp, in place, on a plane that jinc_resize_plane_device produced from d_src with the same table (no
 * reference counterpart: the reference has no anti-ringing).  Every output sample y is pulled toward the range [lo, hi]
 * of the 2x2 source samples around its position: with pos_x / pos_y the table's accumulated positions (jinc_table_axis),
 * ax0 = clamp(floor(pos_x), 0, src_w-1), ax1 = clamp(floor(pos_x)+1, 0, src_w-1), ay0 / ay1 likewise; lo / hi are fminf /
 * fmaxf over src[ay0|ay1][ax0|ax1] (NaN samples ignored); c = fminf(fmaxf(y, lo), hi); the result is c when
 * strength == 1, else fmaf(strength, c, (1 - strength) * y) in float, and y itself when y is NaN.  Integer samples are
 * rounded half to even, half samples to the nearest half.  At strength 1 every output lies in [lo, hi] (a +-Inf output
 * becomes the bound); below 1 a +-Inf output stays +-Inf.  strength: 0..1, 0 = off (a valid call that launches nothing).
 * Same sample_bytes, pitch and alignment rules (destination 16-byte aligned, pitch multiple of 16) and stream semantics as
 * jinc_resize_plane_device.                                                                      */
JINC_API int jinc_antiring_plane_device(jinc_ctx* ctx, const jinc_table* t, int sample_bytes, float strength,
                                        const void* d_src, ptrdiff_t src_pitch, void* d_dst, ptrdiff_t dst_pitch,
                                        void* stream);
/* Introspection of the table's strip plan (no reference counterpart: the reference keeps one weight block per border
 * pixel, src/JincResize.cpp:443-518, and has no notion of patches).  Whole-frame launches of the exact-2x, chunked-cells
 * and integer-ratio kernels run their border strips from descriptors worked out once per table; returns the number of
 * strip patches per plane (0: no plan, the strips derive everything per block) and, through `staged` when it is not
 * NULL, how many of them keep their weight blocks in shared memory.                                  */
JINC_API int jinc_table_strip_plan(const jinc_table* t, int* staged);

/* ---------------------------------------------------------------- filter instance + frame pipeline
 * Replaces: the geometry part of Create_JincResize (src/JincResize.cpp:762-866), JincResize_GetFrame's
 * process_frame call (:615), free_JincResize (:632-647).                                          */
typedef struct jinc_filter_params {
    int32_t src_w, src_h;       /* luma size of the input clip */
    int32_t target_w, target_h; /* luma size of the output clip */
    double src_left, src_top;   /* crop origin */
    double src_width, src_height; /* > 0: crop size; <= 0: offset from the right/bottom edge (:762-770);
                                     pass src_w / src_h for "not given" */
    int32_t quant_x, quant_y;
    int32_t tap;
    double blur;                /* 0 => 1.0 */
    int32_t cplace;             /* JINC_CPLACE_* (used only when chroma is subsampled) */
    int32_t n_planes;           /* 1..4, processing order Y,U,V,A or G,B,R,A (:539-540) */
    int32_t sub_w, sub_h;       /* log2 chroma subsampling of planes 1,2 (0,0 for Y/444/RGB) */
    int32_t sample_bytes;       /* 1, 2, 4 or JINC_SAMPLE_F16 */
    int32_t bits;               /* bits per component (8..16, 32; 16 for JINC_SAMPLE_F16) -> peak (:793) */
    int32_t n_devices;          /* 0 => all visible devices */
    int32_t devices[JINC_MAX_DEVICES];
    int32_t slots_per_device;   /* frames in flight per GPU (0 => 3..8, by frame size) */
    int32_t flags;              /* JINC_FILTER_* */
} jinc_filter_params;

/* jinc_filter_params.flags */
enum {
    /* Page-lock the caller's frame buffers.  A pageable buffer is staged through the pipeline's pinned mirror when it
     * is first seen; with this flag a buffer that comes back (hosts recycle their frame buffers) is registered with
     * cudaHostRegister and from then on moved by DMA directly.  The caller promises that such buffers are recycled, not
     * freed, while filters with this flag exist: a stale registration sends DMA to the buffer's former pages and makes
     * unrelated CUDA calls on the re-used address range fail.  The pipeline checks every transfer through its own
     * registrations (arrival sentinels in destination planes, probe words read back from source planes), drops a
     * registration that fails and redoes that frame through the staged path; registrations idle for five seconds are
     * dropped, and all of them when the last such filter is destroyed.  Memory the caller allocated page-locked is
     * always used directly, flag or not.  The plugin sets the flag unless JINCRESIZE_B200_HOSTREG=0. */
    JINC_FILTER_HOST_REGISTER = 1,
    /* The padding bytes inside the destination planes' pitch belong to the frame (true for AviSynth+ frame buffers):
     * a destination frame whose planes are packed like the pipeline's own may then move with ONE device-to-host
     * transfer that also covers the padding. */
    JINC_FILTER_DST_PADDING_WRITABLE = 2
};

typedef struct jinc_frame {
    const void* src[JINC_MAX_PLANES]; /* host pointers (pageable or pinned) */
    ptrdiff_t src_pitch[JINC_MAX_PLANES];
    void* dst[JINC_MAX_PLANES];
    ptrdiff_t dst_pitch[JINC_MAX_PLANES];
} jinc_frame;

JINC_API int jinc_filter_create(const jinc_filter_params* p, jinc_filter** out);
JINC_API void jinc_filter_destroy(jinc_filter* f);
/* filter objects alive in this process (leak checks; the plugin shares one filter between identical instances) */
JINC_API int jinc_filter_live_count(void);
/* table k (0 = luma/all planes, 1 = subsampled chroma) on the filter's first device; NULL if absent */
JINC_API const jinc_table* jinc_filter_table(const jinc_filter* f, int k);
JINC_API int jinc_filter_num_tables(const jinc_filter* f);
JINC_API int jinc_filter_num_devices(const jinc_filter* f);
/* in-flight slots over all GPUs: how many jinc_filter_submit calls can be outstanding before one blocks */
JINC_API int jinc_filter_num_slots(const jinc_filter* f);
/* Synchronous: stage -> H2D -> kernels -> D2H -> dst.  Thread-safe: concurrent callers take different
 * in-flight slots (round-robin over the filter's GPUs), which is how frames overlap. */
JINC_API int jinc_filter_process(jinc_filter* f, const jinc_frame* frame);
/* Asynchronous pair: submit returns a ticket at once (blocking only when every slot is busy); wait blocks
 * until that frame's dst planes are complete.  src/dst memory must stay valid until wait returns. */
JINC_API int jinc_filter_submit(jinc_filter* f, const jinc_frame* frame, int64_t* ticket);
/* as jinc_filter_submit, but returns JINC_E_BUSY instead of blocking when every slot is taken (a single-threaded
 * producer that submits more than jinc_filter_num_slots() frames before waiting would otherwise block itself) */
JINC_API int jinc_filter_try_submit(jinc_filter* f, const jinc_frame* frame, int64_t* ticket);
/* each ticket is waited on exactly once; a second wait on it fails with JINC_E_INVALID */
JINC_API int jinc_filter_wait(jinc_filter* f, int64_t ticket);
/* The partition rules, host-only (usable without a GPU; multi-process drivers use the same rules across ranks):
 *   frames  -- frame n of a clip belongs to part n % n_parts (what jinc_filter_submit's round-robin does);
 *   bands   -- one frame is cut into n_parts bands of output rows, each a multiple of 16 luma rows (whole cell pairs
 *              for luma and for 4:2:0 chroma) except the last; parts beyond the frame get empty bands.
 * Replaces the reference's row-parallel loop (src/JincResize.cpp:594-599) and AviSynth's per-thread frame hand-out for
 * this MT_MULTI_INSTANCE filter (:649-652) as the unit of parallelism. */
JINC_API int jinc_plan_frame_owner(int64_t frame, int n_parts);
JINC_API int jinc_plan_row_bands(int target_h, int n_parts, int32_t* y_begin, int32_t* y_end);

/* Row-band split of ONE frame across all of the filter's GPUs (each GPU gets a band of output rows plus
 * the source rows its windows reach; no GPU<->GPU traffic).  = jinc_filter_process_bands(f, frame, number of GPUs);
 * with one GPU it is jinc_filter_process. */
JINC_API int jinc_filter_process_split(jinc_filter* f, const jinc_frame* frame);
/* The same with an explicit band count: band i of jinc_plan_row_bands(target_h, n_bands) runs on GPU i % G through
 * its own in-flight slot (own streams and buffers), so with n_bands > G -- or on ONE GPU -- the bands of a frame also
 * overlap their transfers with each other's kernels.  The result is byte-identical to jinc_filter_process. */
JINC_API int jinc_filter_process_bands(jinc_filter* f, const jinc_frame* frame, int n_bands);
/* Device-resident frame: the kernels of jinc_filter_process without staging or PCIe copies.  `frame` holds DEVICE
 * pointers on the filter's GPU `device_index` (destination planes 16-byte aligned, pitch multiple of 16).
 * table_mask selects which tables run (bit 0: luma/shared table, bit 1: subsampled-chroma table); parts selects the
 * kernels (JINC_PART_*), which lets a profiler or bench bracket the interior kernel alone.  Asynchronous on
 * `stream` (a cudaStream_t; NULL = the context's stream). */
enum { JINC_PART_INTERIOR = 1, JINC_PART_BORDER = 2, JINC_PART_ALL = 3 };
JINC_API int jinc_filter_process_device(jinc_filter* f, int device_index, const jinc_frame* frame, int table_mask,
                                        int parts, void* stream);
/* Same for a BATCH of device-resident frames: one launch per table covers every frame of the batch (grid.y = frame).
 * This is the throughput path for callers that keep many frames on the GPU (bench.py's kernel-only leg).  Calls may
 * use different streams: the small device array of plane pointers a launch reads is not reused before that launch
 * has finished. */
JINC_API int jinc_filter_process_device_batch(jinc_filter* f, int device_index, const jinc_frame* frames, int n_frames,
                                              int table_mask, int parts, void* stream);
/* Anti-ringing strength of the filter (no reference counterpart): 0 (the default) = off, 1 = every output sample clamped
 * to the range of the 2x2 source samples around it, in between a blend (see jinc_antiring_plane_device for the exact
 * definition).  When it is > 0, each resample launch of a frame is followed by one anti-ringing launch on the same stream,
 * before the copy back; jinc_filter_process_device(_batch) run it only with parts = JINC_PART_ALL.  Thread-safe; a frame
 * uses the strength current when it is submitted (jinc_filter_process, _submit, _try_submit, _process_bands / _split, the
 * device calls), so it applies to frames submitted after this call returns.  JINC_E_INVALID for a NULL filter or a
 * strength that is NaN or outside [0, 1]. */
JINC_API int jinc_filter_set_antiring(jinc_filter* f, float strength);
/* kernels launched so far by this filter (all devices) */
JINC_API int64_t jinc_filter_kernel_launches(const jinc_filter* f);
/* host-buffer bookkeeping of the frame pipeline (process-wide): bytes of caller memory currently page-locked by
 * cudaHostRegister, number of registrations made, frames that moved without a staging copy on the source / on the
 * destination side, frames staged.  Any pointer may be NULL. */
JINC_API void jinc_host_buffer_stats(int64_t* registered_bytes, int64_t* registrations, int64_t* direct_src_frames,
                                     int64_t* direct_dst_frames, int64_t* staged_frames);

#ifdef __cplusplus
}
#endif
#endif /* JINC_B200_H */
