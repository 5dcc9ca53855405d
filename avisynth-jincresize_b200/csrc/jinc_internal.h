// jinc_internal.h -- shared declarations of libjinc_b200.so (not part of the public ABI).
#ifndef JINC_INTERNAL_H
#define JINC_INTERNAL_H

#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <functional>
#include <mutex>
#include <string>
#include <vector>

#include "jinc_b200.h"
#include "jinc_border.h"

// ---------------------------------------------------------------- errors
void jinc_set_error(const char* fmt, ...) __attribute__((format(printf, 1, 2)));
int jinc_fail(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));

#define JINC_CUDA(call)                                                                                     \
    do {                                                                                                    \
        cudaError_t err_ = (call);                                                                          \
        if (err_ != cudaSuccess) {                                                                          \
            cudaGetLastError(); /* reported here: must not resurface at the next launch check */            \
            return jinc_fail(JINC_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(err_), __FILE__, \
                             __LINE__);                                                                     \
        }                                                                                                   \
    } while (0)

// ---------------------------------------------------------------- context
// Ring of small device buffers holding the plane-pointer records of batched launches.  An entry is reused only after the
// launch that read it has finished (event), whatever streams the calls use.
struct RecordRing {
    static constexpr int kRing = 8;
    std::mutex mu;
    unsigned char* ptrs[kRing] = {};
    size_t cap[kRing] = {};
    cudaEvent_t done[kRing] = {};
    int next = 0;
};

struct jinc_ctx {
    int device = -1;
    int sm_count = 0;
    size_t smem_optin = 0;
    cudaStream_t stream = nullptr; // default stream for table builds and callers that pass none
    RecordRing ring;
};

// Uploads `bytes` of host records into the next entry of the context's ring on `st`, calls launch(device copy) and records
// the entry's event after it.  The whole sequence runs under the ring's lock, so two callers on different streams cannot
// interleave on one entry.  Returns launch's result, or the error of the upload.  Call with ctx->device current.
int jinc_ring_launch(jinc_ctx* ctx, const void* host, size_t bytes, cudaStream_t st, const std::function<int(const void*)>& launch);
void jinc_ring_free(jinc_ctx* ctx); // waits for the ring's last readers

// ---------------------------------------------------------------- table
// Geometry scalars of one table, derived on the host in the reference's own precision
// (src/JincResize.cpp:349-364) and handed to the device kernels.
struct TableScalars {
    int quant_x, quant_y;
    int src_w, src_h, dst_w, dst_h;
    int fs;              // filter_size
    float support;       // filter_support (max of x/y)
    float pos0[2];       // start_x, initial ypos
    float pos_step[2];   // x_step, y_step
    double filt_step[2]; // filter_step_x, filter_step_y
    double radius2;
    double idx_scale;    // (samples-1)/radius2, only used to pre-screen the exact index computation
};

// Per-axis device arrays (axis 0 = x over dst_w, axis 1 = y over dst_h).
struct AxisArrays {
    float* pos = nullptr;       // accumulated position
    int32_t* start = nullptr;   // window origin (meta)
    int32_t* qint = nullptr;    // (int)(pos*quant)
    int32_t* phase = nullptr;   // qint % quant
    int32_t* rank = nullptr;    // compact index of the phase among used ones; -1 on border
    uint8_t* border = nullptr;
    int32_t* rep = nullptr;     // [quant] first non-border index with that phase value (INT_MAX if unused)
    int32_t* rank_of = nullptr; // [quant] phase value -> rank (-1 unused)
    double* rep_d2 = nullptr;   // [n_rank][fs] squared scaled distances of the phase representative
    int n = 0;
    int n_rank = 0;
};

// Description of the exact-2x interior handled by the register-tiled kernel.
struct Up2xPlan {
    bool ok = false;
    int x0 = 0, y0 = 0;       // first output pixel of the periodic interior (multiple of 8 / 2)
    int ncx = 0, ncy = 0;     // cells (2x2 output quads) per axis
    int sx0 = 0, sy0 = 0;     // window origin of cell (0,0), phase 0
    int ox1 = 0, oy1 = 0;     // extra origin offset of phase 1 on each axis (0 or 1)
    int wblock[2][2] = {{0, 0}, {0, 0}}; // [py][px] -> phase-block index
    int taps = 0;      // tap-mask variant of integer planes (UpTaps<fs, taps>, jinc_up2x_taps.h); 0: every tap
    int live_taps = 0; // taps per cell that variant multiplies
};

// Integer-ratio downscale interior (one phase).
struct DownPlan {
    bool ok = false;
    int x0 = 0, y0 = 0, nx = 0, ny = 0; // output rectangle
    int sx0 = 0, sy0 = 0;               // window origin of output (x0,y0)
    int qx = 0, qy = 0;                 // source step per output pixel
    int wblock = 0;
};

// Exactly periodic rational ratio: output P*c + p reads the window at Q*c + off[p] with phase block p, on both axes
// (the reference accumulates positions in float, so this needs crop/dst = m/2^k: 2:3 and 3:4 ratios).  Every (py, px)
// sub-lattice is an integer-ratio-Q problem of its own, run as one pass of the polyphase kernel with output stride P.
struct PeriodicPlan {
    bool ok = false;
    int P = 0, Q = 0;
    int x0 = 0, y0 = 0, ncx = 0, ncy = 0; // first output of the periodic interior, cells per axis
    int sx0 = 0, sy0 = 0;                 // window origin of cell (0,0), phase (0,0)
    int ox[4] = {0, 0, 0, 0}, oy[4] = {0, 0, 0, 0}; // origin offset of phase p
    int wblock[4][4] = {};                // [py][px] -> phase-block index
};

// Piecewise-periodic rational ratio (jinc_cells.cuh): crop/dst = Q/P on both axes.  Each axis is a regular grid of groups
// of JINC_CELLS_N* cells (a cell = P consecutive outputs), cut into CHUNKS inside which every residue p keeps its phase
// rank and its window origins advance by exactly Q per cell: one chunk per group, more where a residue changes rank.
constexpr int JINC_CELLS_NX = 4, JINC_CELLS_NY = 4;
// y-chunks per tile (one per warp): four.  128-thread blocks, four of them per SM for the small windows and steps, overlap
// their staging and store phases better than two 256-thread blocks did (config 6: 21.1 -> 23.3 % of the FMA peak)
constexpr int jinc_cells_warps(int, int) { return 4; }
// samples staged along one axis for a tile of `chunks` chunks of n cells: the chunks' cells, the window, and slack for the
// residues' origin offsets and one irregular origin step
constexpr int jinc_cells_footprint(int q, int fs, int n, int chunks) { return q * n * chunks + fs + q + 2; }
constexpr bool jinc_cells_instantiated(int q, int fs)
{
    return (q >= 1 && q <= 4 && (fs == 7 || fs == 9)) || ((q == 1 || q == 2) && (fs == 5 || fs == 11)) ||
           (q == 3 && fs == 10); // tap 3 at 2:3 (1080p -> 720p): one staging per tile instead of one per pass of the periodic path
}

struct CellsAxis {
    int P = 0, Q = 0;
    int first = 0, ncells = 0; // first output of cell 0, number of cells
    int n_chunks = 0;
    // per chunk: first cell of its group, first cell of the chunk inside the group, cells of the chunk; per (chunk, residue):
    // window origin of the GROUP's first cell (extrapolated from the chunk's), phase rank
    std::vector<int32_t> cell, i0, n, org, rank;
    int32_t* d_cell = nullptr;
    int32_t* d_i0 = nullptr;
    int32_t* d_n = nullptr;
    int32_t* d_org = nullptr;
    int32_t* d_rank = nullptr;
};

struct CellsPlan {
    bool ok = false;
    int Q = 0;
    CellsAxis ax[2];
};

// Strip plan (whole-frame launches of a fast path; jinc_resize.cu builds it once per table, jinc_resample.cuh runs it).
// Everything a strip block otherwise derives in its prologue -- the patches of the border strips, a patch's source
// footprint, every thread's samples, their window offsets, weight blocks and the way they are accumulated -- is worked
// out once on the host, and the few distinct weight blocks of a patch are packed next to each other so the block
// copies them into shared memory with its footprint.
struct StripPlanPatch {
    int32_t sx_lo, sy_lo, fw, fh; // source footprint of the patch
    uint32_t magic;               // floor(e / fw) = umulhi(e, magic)
    int32_t n_wb;                 // weight blocks staged in shared memory; < 0: too many, read from the packed copy
    uint32_t wdata_off;           // first float of the patch's packed weight blocks in StripPlan::d_wdata
    uint32_t tile_floats;         // shared-memory offset of the staged blocks (footprint rounded up to 16 bytes)
    int32_t row_stride;           // floats per staged footprint row (fw, or step * sub when de-interleaved)
    int32_t sub;                  // de-interleaved rows: column c sits at (c % step) * sub + c / step
    int32_t deint;                // 1: the footprint is staged de-interleaved by the window step (patches of row runs only)
    int32_t ring;                 // > 0: float offset of the weight-row rings in the block's shared memory (plan_run_rows_ring), else 0
};
constexpr int JINC_PLAN_RING_DEPTH = 8; // weight rows in flight per half-warp (wide windows read from the table's blocks)
enum { JINC_SK_NONE = 0, JINC_SK_RUN_ROWS, JINC_SK_RUN_COLS, JINC_SK_FUSED_SHARED, JINC_SK_FUSED_SEP, JINC_SK_PER_SAMPLE, JINC_SK_PER_PIXEL };
struct StripPlan {
    bool ok = false;
    int threads = 0, spt = 0, px = 0, py = 0;
    unsigned n_patches = 0;  // strip blocks per plane
    unsigned n_staged = 0;   // patches whose weight blocks are staged in shared memory
    StripPlanPatch* d_patches = nullptr;
    // [patch][sample k][thread]: .x = x | y << 16, .y = offset of the window origin in the staged footprint,
    // .z = float offset of the weight block among the staged ones (JINC_SK_PER_PIXEL: the pixel's border slot),
    // .w (sample 0) = kind | live mask << 8
    uint4* d_threads = nullptr;
    float* d_wdata = nullptr;
};

struct jinc_table {
    jinc_ctx* ctx = nullptr;
    jinc_table_params params{};
    TableScalars sc{};
    AxisArrays ax[2];
    float* d_lut = nullptr;      // JINC_LUT_SAMPLES floats (Lut::GetFactor values)
    float* d_weights = nullptr;  // [n_rank_y][n_rank_x][fs*fs] normalised phase blocks
    std::vector<float> h_weights; // host copy (kernel parameters for the fast paths)
    float* d_weights_p = nullptr; // the blocks again as [block][fs][fsp], fsp = fs rounded up to 4 (null: fs % 4 == 0 or over budget)
    BorderGeom bgeom{};          // strips of border pixels
    float* d_border_sum = nullptr; // [bgeom.total] per-border-pixel normaliser
    float* d_border_w = nullptr;   // [bgeom.total/32][fs*fs][32] resident per-pixel border weights (null: rebuilt on the fly)
    // Border pixels whose clamped position sits at the same offset from its window origin on both axes have identical
    // weight blocks; when that folds the border into few classes the blocks are kept once, [block][fs*fs], plus a map
    int32_t* d_border_block = nullptr; // [bgeom.total] slot -> class block (null: per-slot weights above)
    float* d_border_wb = nullptr;      // [n_border_blocks][fs][fsp], fsp = fs rounded up to 4 (16-byte rows, pad = 0)
    int n_border_blocks = 0;
    std::vector<int32_t> h_border_block; // host copy of the slot -> class map (strip plan)
    StripPlan strip_plan;
    // host mirrors of the small per-axis arrays (for planning and introspection)
    std::vector<int32_t> h_start[2], h_phase[2], h_rank[2], h_qint[2];
    std::vector<uint8_t> h_border[2];
    std::vector<float> h_pos[2];
    Up2xPlan up2x;
    DownPlan down;
    PeriodicPlan periodic;
    CellsPlan cells;
    int fast_path = JINC_PATH_GENERAL;
    int ix0 = 0, ix1 = 0, iy0 = 0, iy1 = 0; // interior rectangle run by the fast path (empty if none)
    float build_ms = 0.f;                   // host wall time of jinc_table_create
};

// jinc_lut.cpp
void jinc_lut_build_host(double radius, double blur, double* lut);

// jinc_table.cu
int jinc_table_build_device(jinc_table* t, const double* lut);
cudaError_t jinc_gather_blocks(float* out, const uint32_t* list, unsigned n, const float* phase_blocks, const float* border_blocks,
                               int block_floats, cudaStream_t st);

// Sample format of the C ABI (the `sample_bytes` arguments): 1 (uint8), 2 (uint16), 4 (float) or JINC_SAMPLE_F16 (IEEE
// binary16).  The launchers below take this code; byte counts (pitches, plane sizes, transfers) take jinc_sample_size.
inline bool jinc_sample_valid(int sample) { return sample == 1 || sample == 2 || sample == 4 || sample == JINC_SAMPLE_F16; }
inline int jinc_sample_size(int sample) { return sample & 0xff; }
inline bool jinc_sample_is_float(int sample) { return sample == 4 || sample == JINC_SAMPLE_F16; }

// jinc_resize.cu
int jinc_build_strip_plan(jinc_table* t); // after plan_fast_paths and the weight blocks; no plan is not an error
void jinc_free_strip_plan(jinc_table* t);
int jinc_launch_resize(jinc_ctx* ctx, const jinc_table* t, int sample, float peak, const void* d_src,
                       ptrdiff_t src_pitch, void* d_dst, ptrdiff_t dst_pitch, int y_begin, int y_end,
                       cudaStream_t stream, int* launches);
// several planes that share one table in a single launch (blockIdx.z / .y = plane); rows [y_begin,y_end)
int jinc_launch_resize_planes(jinc_ctx* ctx, const jinc_table* t, int sample, float peak, int n_planes,
                              const void* const* d_src, const ptrdiff_t* src_pitch, void* const* d_dst,
                              const ptrdiff_t* dst_pitch, int y_begin, int y_end, cudaStream_t stream, int* launches,
                              int parts = JINC_PART_ALL);
// batched: d_frame_ptrs is a DEVICE array of n_frames packed plane-pointer records (jinc_pack_plane_ptrs)
size_t jinc_plane_ptrs_size();
int jinc_pack_plane_ptrs(void* out, int sample, int n_planes, const void* const* d_src, const ptrdiff_t* src_pitch,
                         void* const* d_dst, const ptrdiff_t* dst_pitch);
int jinc_launch_resize_batch(jinc_ctx* ctx, const jinc_table* t, int sample, float peak, int n_planes,
                             const void* d_frame_ptrs, int n_frames, cudaStream_t stream, int* launches, int parts);
// jinc_antiring.cu: the anti-ringing clamp in place on planes the two launchers above produced, with the same plane
// arguments (rows [y_begin,y_end) read the same source rows as the resample launch of that band).  strength in [0, 1];
// 0 launches nothing.  Needs complete output samples: run it after a JINC_PART_ALL resample launch.
int jinc_launch_antiring_planes(const jinc_table* t, int sample, float strength, int n_planes, const void* const* d_src,
                                const ptrdiff_t* src_pitch, void* const* d_dst, const ptrdiff_t* dst_pitch, int y_begin,
                                int y_end, cudaStream_t stream, int* launches);
int jinc_launch_antiring_batch(const jinc_table* t, int sample, float strength, int n_planes, const void* d_frame_ptrs,
                               int n_frames, cudaStream_t stream, int* launches);
// jinc_adjoint.cu: the adjoint (jinc_b200.h, jinc_resize_adjoint_planes_device) of n_planes float planes; pitches and plane
// strides in floats.  Adds the number of kernels launched to *launches.
int jinc_launch_adjoint(const jinc_table* t, int n_planes, const float* g, long long g_pitch, long long g_stride, float* out,
                        long long out_pitch, long long out_stride, cudaStream_t stream, int* launches);
// jinc_antiring_adjoint.cu: the derivative of the anti-ringing clamp (jinc_b200.h, jinc_antiring_adjoint_planes_device).
// Plane i of each array at base + i * stride; pitches and strides in elements (src / y: the forward's float or half samples).
struct ArAdjPlanes {
    const void* src;
    long long src_pitch, src_stride;
    const void* y; // the resized planes before the clamp
    long long y_pitch, y_stride;
    const float* g; // output gradient
    long long g_pitch, g_stride;
    float* gy; // written: gradient of the resized planes
    long long gy_pitch, gy_stride;
    float* gs; // written: source gradient
    long long gs_pitch, gs_stride;
    int n_planes;
};
// Three launches on `stream`: antiring_grad_out (g -> gy), jinc_launch_adjoint (gy -> gs), antiring_route_gather (gs += r);
// at strength 0 a copy of g into gy and the plain adjoint.  sample 4 or JINC_SAMPLE_F16, strength in [0, 1].  Adds the
// number of kernels launched to *launches.
int jinc_launch_antiring_adjoint(const jinc_table* t, int sample, float strength, const ArAdjPlanes& p, cudaStream_t stream,
                                 int* launches);
int jinc_debug_pixel_weights(const jinc_table* t, int x, int y, float* out);
// probe words of a device buffer: d_out[k] = 32-bit word jinc_probe_index(seed, k, n_words) of d_buf, k < JINC_PROBE_WORDS
constexpr int JINC_PROBE_WORDS = 256;
#ifdef __CUDACC__
#define JINC_HOST_DEVICE __host__ __device__
#else
#define JINC_HOST_DEVICE
#endif
JINC_HOST_DEVICE inline uint32_t jinc_probe_index(uint32_t seed, uint32_t k, uint32_t n_words)
{
    uint32_t x = seed + k * 0x9E3779B9u;
    x ^= x >> 16;
    x *= 0x7feb352du;
    x ^= x >> 15;
    x *= 0x846ca68bu;
    x ^= x >> 16;
    return static_cast<uint32_t>((static_cast<uint64_t>(x) * n_words) >> 32);
}
int jinc_launch_probe(const void* d_buf, uint32_t n_words, uint32_t seed, uint32_t* d_out, cudaStream_t stream);

#endif
