// jinc_antiring.cu -- the anti-ringing clamp: an in-place pass over a resized plane (no reference counterpart).
//
// Every output sample y is pulled toward the range [lo, hi] of the 2x2 source samples around its position:
//   ax0 = clamp(floor(pos_x), 0, W-1), ax1 = clamp(floor(pos_x) + 1, 0, W-1), ay0 / ay1 likewise from pos_y
//   lo / hi = fminf / fmaxf over src[ay0|ay1][ax0|ax1]        (NaN neighbours are ignored)
//   c = fminf(fmaxf(y, lo), hi);  out = s == 1 ? c : fmaf(s, c, (1 - s) * y);  NaN y stays NaN
// stored with round-half-even for integer planes (out lies between y and c, so no clamp), __float2half_rn for half.
// pos_x / pos_y are the table's accumulated positions (AxisArrays::pos).  The pass is a pure function of the stored
// resized plane, the source plane and the table, so it can follow any resample launch; DESIGN.md §4.7.
//
// Work split: a block covers ArVec<T>::COLS = 32 * V output columns (V samples per 16-byte vector) and AR_ROWS rows; its
// columns' anchors are worked out once into shared memory, a warp takes whole rows, a lane one 16-byte vector of a row.
// Source samples are read through the read-only path; output rows with 16-byte loads and stores (a row's partial last
// vector sample by sample, so bytes past the plane's width are never written).
#include <cuda_fp16.h>

#include "jinc_resample.cuh"

namespace jinc_rs {

constexpr int AR_THREADS = 256;
constexpr int AR_WARP_ROWS = 4; // rows per warp
constexpr int AR_ROWS = AR_THREADS / 32 * AR_WARP_ROWS;

template <typename T>
struct ArVec {
    static constexpr int V = 16 / (int)sizeof(T);
    static constexpr int COLS = 32 * V;
};

struct AntiringArgs {
    FrameSet fr;
    const float* pos_x;
    const float* pos_y;
    int src_w, src_h, dst_w;
    int y_begin, y_end;
    int col_tiles; // blockIdx.x = row tile * col_tiles + column tile
    float s;
};

template <typename T>
__device__ __forceinline__ float ar_widen(T v)
{
    if constexpr (std::is_same<T, __half>::value)
        return __half2float(v);
    else
        return (float)v;
}

template <typename T>
__device__ __forceinline__ T ar_store(float v)
{
    if constexpr (std::is_same<T, float>::value)
        return v;
    else if constexpr (std::is_same<T, __half>::value)
        return __float2half_rn(v);
    else
        return (T)__float2int_rn(v);
}

template <typename T>
__device__ __forceinline__ float ar_sample(float y, const T* __restrict__ r0, const T* __restrict__ r1, int xp, float s)
{
    const int x0 = xp >> 1, x1 = x0 + (xp & 1);
    const float a = ar_widen<T>(__ldg(r0 + x0)), b = ar_widen<T>(__ldg(r0 + x1));
    const float c = ar_widen<T>(__ldg(r1 + x0)), d = ar_widen<T>(__ldg(r1 + x1));
    const float lo = fminf(fminf(a, b), fminf(c, d)), hi = fmaxf(fmaxf(a, b), fmaxf(c, d));
    const float cl = fminf(fmaxf(y, lo), hi);
    if (isnan(y))
        return y;
    return s == 1.f ? cl : fmaf(s, cl, __fmul_rn(1.f - s, y));
}

template <typename T>
__global__ void __launch_bounds__(AR_THREADS) antiring_pass(AntiringArgs a)
{
    using A = ArVec<T>;
    // anchors of column lane * V + k at [k][lane] (conflict-free reads), packed as 2 * ax0 + (ax1 - ax0)
    __shared__ int sx[A::COLS];
    const int tile_x = blockIdx.x % a.col_tiles, tile_y = blockIdx.x / a.col_tiles;
    const int cx0 = tile_x * A::COLS;
    for (int i = threadIdx.x; i < A::COLS; i += AR_THREADS) {
        const int f = __float2int_rd(a.pos_x[min(cx0 + i, a.dst_w - 1)]);
        const int x0 = min(max(f, 0), a.src_w - 1), x1 = min(max(f + 1, 0), a.src_w - 1);
        sx[(i % A::V) * 32 + i / A::V] = 2 * x0 + (x1 - x0);
    }
    __syncthreads();

    const PlanePtrs& pp = frame_ptrs(a.fr);
    const int plane = blockIdx.z;
    const T* __restrict__ src = static_cast<const T*>(pp.src[plane]);
    T* dst = static_cast<T*>(pp.dst[plane]);
    const long long sp = pp.src_pitch[plane], dp = pp.dst_pitch[plane];
    const float s = a.s;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c0 = lane * A::V;       // first column of this lane inside the block's columns
    const int x = cx0 + c0;
    const int ry0 = a.y_begin + tile_y * AR_ROWS + warp * AR_WARP_ROWS;
    if (x >= a.dst_w)
        return;
    int ax[A::V];
#pragma unroll
    for (int k = 0; k < A::V; ++k)
        ax[k] = sx[k * 32 + lane];
#pragma unroll 1
    for (int r = 0; r < AR_WARP_ROWS; ++r) {
        const int y = ry0 + r;
        if (y >= a.y_end)
            break;
        const int fy = __float2int_rd(a.pos_y[y]);
        const T* __restrict__ r0 = src + sp * min(max(fy, 0), a.src_h - 1);
        const T* __restrict__ r1 = src + sp * min(max(fy + 1, 0), a.src_h - 1);
        T* row = dst + dp * y + x;
        if (x + A::V <= a.dst_w) {
            union {
                uint4 u;
                T v[A::V];
            } buf;
            buf.u = *reinterpret_cast<const uint4*>(row);
#pragma unroll
            for (int k = 0; k < A::V; ++k)
                buf.v[k] = ar_store<T>(ar_sample<T>(ar_widen<T>(buf.v[k]), r0, r1, ax[k], s));
            *reinterpret_cast<uint4*>(row) = buf.u;
        } else {
            for (int k = 0; k < a.dst_w - x; ++k)
                row[k] = ar_store<T>(ar_sample<T>(ar_widen<T>(row[k]), r0, r1, sx[k * 32 + lane], s));
        }
    }
}

} // namespace jinc_rs

namespace {

using namespace jinc_rs;

template <typename T>
cudaError_t launch_antiring_typed(const AntiringArgs& a0, int n_planes, int n_frames, cudaStream_t st)
{
    AntiringArgs a = a0;
    a.col_tiles = (a.dst_w + ArVec<T>::COLS - 1) / ArVec<T>::COLS;
    const int row_tiles = (a.y_end - a.y_begin + AR_ROWS - 1) / AR_ROWS;
    antiring_pass<T><<<dim3((unsigned)(a.col_tiles * row_tiles), (unsigned)n_frames, (unsigned)n_planes), AR_THREADS, 0, st>>>(a);
    return cudaGetLastError();
}

int launch_antiring(const jinc_table* t, int sample, float strength, const FrameSet& fr, int n_frames, int y_begin, int y_end,
                    cudaStream_t st, int* launches)
{
    if (!jinc_sample_valid(sample))
        return jinc_fail(JINC_E_INVALID, "antiring: sample_bytes must be 1, 2, 4 or JINC_SAMPLE_F16");
    if (!(strength >= 0.f && strength <= 1.f))
        return jinc_fail(JINC_E_INVALID, "antiring: strength must be between 0.0 and 1.0");
    y_begin = std::max(y_begin, 0);
    y_end = std::min(y_end, t->sc.dst_h);
    if (strength == 0.f || y_end <= y_begin || n_frames <= 0)
        return JINC_OK;
    AntiringArgs a;
    memset(&a, 0, sizeof(a));
    a.fr = fr;
    a.pos_x = t->ax[0].pos;
    a.pos_y = t->ax[1].pos;
    a.src_w = t->sc.src_w;
    a.src_h = t->sc.src_h;
    a.dst_w = t->sc.dst_w;
    a.y_begin = y_begin;
    a.y_end = y_end;
    a.s = strength;
    cudaError_t e = cudaSuccess;
    switch (sample) {
    case 1: e = launch_antiring_typed<uint8_t>(a, fr.n_planes, n_frames, st); break;
    case 2: e = launch_antiring_typed<uint16_t>(a, fr.n_planes, n_frames, st); break;
    case 4: e = launch_antiring_typed<float>(a, fr.n_planes, n_frames, st); break;
    default: e = launch_antiring_typed<__half>(a, fr.n_planes, n_frames, st); break;
    }
    if (e != cudaSuccess)
        return jinc_fail(JINC_E_CUDA, "antiring_pass launch failed: %s", cudaGetErrorString(e));
    if (launches)
        ++*launches;
    return JINC_OK;
}

} // namespace

int jinc_launch_antiring_planes(const jinc_table* t, int sample, float strength, int n_planes, const void* const* d_src,
                                const ptrdiff_t* src_pitch, void* const* d_dst, const ptrdiff_t* dst_pitch, int y_begin,
                                int y_end, cudaStream_t stream, int* launches)
{
    FrameSet fr;
    memset(&fr, 0, sizeof(fr));
    if (int rc = jinc_pack_plane_ptrs(&fr.one, sample, n_planes, d_src, src_pitch, d_dst, dst_pitch))
        return rc;
    fr.frames = nullptr;
    fr.n_planes = n_planes;
    return launch_antiring(t, sample, strength, fr, 1, y_begin, y_end, stream, launches);
}

int jinc_launch_antiring_batch(const jinc_table* t, int sample, float strength, int n_planes, const void* d_frame_ptrs,
                               int n_frames, cudaStream_t stream, int* launches)
{
    FrameSet fr;
    memset(&fr, 0, sizeof(fr));
    fr.frames = static_cast<const PlanePtrs*>(d_frame_ptrs);
    fr.n_planes = n_planes;
    return launch_antiring(t, sample, strength, fr, n_frames, 0, t->sc.dst_h, stream, launches);
}

extern "C" int jinc_antiring_plane_device(jinc_ctx* ctx, const jinc_table* t, int sample_bytes, float strength,
                                          const void* d_src, ptrdiff_t src_pitch, void* d_dst, ptrdiff_t dst_pitch, void* stream)
{
    if (!ctx || !t)
        return jinc_fail(JINC_E_INVALID, "jinc_antiring_plane_device: null argument");
    JINC_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    return jinc_launch_antiring_planes(t, sample_bytes, strength, 1, &d_src, &src_pitch, &d_dst, &dst_pitch, 0, t->sc.dst_h,
                                       st, nullptr);
}
