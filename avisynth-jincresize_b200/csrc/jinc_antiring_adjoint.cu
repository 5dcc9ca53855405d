// jinc_antiring_adjoint.cu -- the derivative of the anti-ringing clamp (jinc_antiring.cu) for float and half planes.
//
// Per output sample, with y the stored resized sample (before the clamp), anchors a0..a3 = src[ay0][ax0], src[ay0][ax1],
// src[ay1][ax0], src[ay1][ax1] and lo / hi = fminf / fmaxf over them, exactly as the forward pass computes them:
//   inside  (y NaN, or lo <= y <= hi, all-NaN anchors included):  g_y = g, nothing routed
//   below   (y < lo):  g_y = s == 1 ? +0 : (1 - s) * g;  s == 1 ? g : s * g  routed to the FIRST anchor in a0..a3 order == lo
//   above   (y > hi):  the same with hi
// and grad_src = A^T g_y + r, A^T the resize adjoint (jinc_adjoint.cu), r[sy][sx] the values routed to that sample summed
// in canonical order (output rows ascending, then columns, __fadd_rn from the first routed value); a sample that receives
// nothing keeps A^T g_y bit for bit, one that does gets __fadd_rn(A^T g_y, r).  DESIGN.md 4.9.
//
//   antiring_grad_out      per output sample: g_y.  The shape of antiring_pass: a block covers 32 * V columns x 32 rows,
//                          the columns' anchors are worked out once into shared memory, blockIdx.z = plane of a record of
//                          up to four planes, grid.y = record.  Column k * 32 + lane of the block goes to lane `lane`, so
//                          every load and store of a warp is one contiguous run.
//   antiring_route_gather  per source sample, after the adjoint on the same stream: adds r into grad_src in place.  Source
//                          column sx is an anchor exactly of the outputs with ax0(x) <= sx <= ax1(x); pos never decreases,
//                          so they are one range [first x with ax1(x) >= sx, first x with ax0(x) > sx), found by binary
//                          search on the table's positions (the same for rows).  A block takes 32 x 8 source samples,
//                          stages them with a one-sample halo (every anchor of a candidate output lies there), works out
//                          each candidate output's case and routed anchor once from shared memory, and each thread then
//                          sums what was routed to its sample in canonical order: no atomics, no scratch planes.
#include <cuda_fp16.h>

#include "jinc_resample.cuh"

using namespace jinc_rs;

namespace {

constexpr int GO_THREADS = 256;
constexpr int GO_WARP_ROWS = 4;
constexpr int GO_ROWS = GO_THREADS / 32 * GO_WARP_ROWS;

constexpr int RG_TW = 32, RG_TH = 8, RG_THREADS = RG_TW * RG_TH;
constexpr int RG_HW = RG_TW + 2;   // staged source row: the tile's columns and one on each side
constexpr int RG_CAND = 4096;      // candidate outputs staged per pass (code + value: 32 KB; six blocks per SM)

struct ArAdjArgs {
    ArAdjPlanes p;
    const float* pos_x;
    const float* pos_y;
    int src_w, src_h, dst_w, dst_h;
    int per, n_rec;   // antiring_grad_out: planes per record (grid.z), records
    int col_tiles;    // antiring_grad_out: blockIdx.x = row tile * col_tiles + column tile
    int tiles_x;      // antiring_route_gather: blockIdx.x = tile row * tiles_x + tile column
    float s;
};

template <typename T>
__device__ __forceinline__ float widen(T v)
{
    if constexpr (std::is_same<T, __half>::value)
        return __half2float(v);
    else
        return v;
}

__device__ __forceinline__ int anchor0(const float* __restrict__ pos, int i, int n_src)
{
    return min(max(__float2int_rd(__ldg(pos + i)), 0), n_src - 1);
}

__device__ __forceinline__ int anchor1(const float* __restrict__ pos, int i, int n_src)
{
    return min(max(__float2int_rd(__ldg(pos + i)) + 1, 0), n_src - 1);
}

// ABOVE ? first output i in [0, n) with anchor0(i) > s : first with anchor1(i) >= s  (n when none; both non-decreasing)
template <bool ABOVE>
__device__ __forceinline__ int anchor_bound(const float* __restrict__ pos, int n, int n_src, int s)
{
    int lo = 0, hi = n;
    while (lo < hi) {
        const int m = (lo + hi) >> 1;
        if (ABOVE ? anchor0(pos, m, n_src) <= s : anchor1(pos, m, n_src) < s)
            lo = m + 1;
        else
            hi = m;
    }
    return lo;
}

template <typename T>
__global__ void __launch_bounds__(GO_THREADS) antiring_grad_out(const __grid_constant__ ArAdjArgs a)
{
    constexpr int V = 16 / (int)sizeof(T);
    constexpr int COLS = 32 * V;
    __shared__ int sx[COLS]; // column cx0 + i: 2 * ax0 + (ax1 - ax0)
    const int tile_x = blockIdx.x % a.col_tiles, tile_y = blockIdx.x / a.col_tiles;
    const int cx0 = tile_x * COLS;
    for (int i = threadIdx.x; i < COLS; i += GO_THREADS) {
        const int x = min(cx0 + i, a.dst_w - 1);
        const int x0 = anchor0(a.pos_x, x, a.src_w);
        sx[i] = 2 * x0 + (anchor1(a.pos_x, x, a.src_w) - x0);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ry0 = tile_y * GO_ROWS + warp * GO_WARP_ROWS;
    int ax[V];
#pragma unroll
    for (int k = 0; k < V; ++k)
        ax[k] = sx[k * 32 + lane];
    const float s = a.s;
    const float g_scale = 1.f - s;
    for (int rec = blockIdx.y; rec < a.n_rec; rec += gridDim.y) {
        const long long plane = (long long)rec * a.per + blockIdx.z;
        const T* __restrict__ src = static_cast<const T*>(a.p.src) + plane * a.p.src_stride;
        const T* __restrict__ yp = static_cast<const T*>(a.p.y) + plane * a.p.y_stride;
        const float* __restrict__ gp = a.p.g + plane * a.p.g_stride;
        float* __restrict__ gyp = a.p.gy + plane * a.p.gy_stride;
#pragma unroll 1
        for (int r = 0; r < GO_WARP_ROWS; ++r) {
            const int row = ry0 + r;
            if (row >= a.dst_h)
                break;
            const int ay0 = anchor0(a.pos_y, row, a.src_h), ay1 = anchor1(a.pos_y, row, a.src_h);
            const T* __restrict__ r0 = src + a.p.src_pitch * ay0;
            const T* __restrict__ r1 = src + a.p.src_pitch * ay1;
            const T* __restrict__ yr = yp + a.p.y_pitch * row;
            const float* __restrict__ gr = gp + a.p.g_pitch * row;
            float* __restrict__ gyr = gyp + a.p.gy_pitch * row;
#pragma unroll
            for (int k = 0; k < V; ++k) {
                const int x = cx0 + k * 32 + lane;
                if (x >= a.dst_w)
                    break;
                const int x0 = ax[k] >> 1, x1 = x0 + (ax[k] & 1);
                const float a0 = widen<T>(__ldg(r0 + x0)), a1 = widen<T>(__ldg(r0 + x1));
                const float a2 = widen<T>(__ldg(r1 + x0)), a3 = widen<T>(__ldg(r1 + x1));
                const float lo = fminf(fminf(a0, a1), fminf(a2, a3)), hi = fmaxf(fmaxf(a0, a1), fmaxf(a2, a3));
                const float y = widen<T>(__ldg(yr + x));
                const float g = __ldg(gr + x);
                gyr[x] = (y < lo || y > hi) ? (s == 1.f ? 0.f : __fmul_rn(g_scale, g)) : g;
            }
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(RG_THREADS, 6) antiring_route_gather(const __grid_constant__ ArAdjArgs a)
{
    __shared__ int s_xlo[RG_TW], s_xhi[RG_TW], s_ylo[RG_TH], s_yhi[RG_TH];
    __shared__ float s_src[(RG_TH + 2) * RG_HW];
    __shared__ int s_code[RG_CAND];   // candidate's routed sample inside the tile (ly * RG_TW + lx), or -1
    __shared__ float s_val[RG_CAND];  // the value routed to it

    const int tyi = blockIdx.x / a.tiles_x, txi = blockIdx.x - tyi * a.tiles_x;
    const int x0 = txi * RG_TW, y0 = tyi * RG_TH;
    const int tw = min(RG_TW, a.src_w - x0), th = min(RG_TH, a.src_h - y0);
    const int tid = threadIdx.x;
    if (tid < tw) {
        s_xlo[tid] = anchor_bound<false>(a.pos_x, a.dst_w, a.src_w, x0 + tid);
        s_xhi[tid] = anchor_bound<true>(a.pos_x, a.dst_w, a.src_w, x0 + tid);
    } else if (tid >= 32 && tid - 32 < th) {
        s_ylo[tid - 32] = anchor_bound<false>(a.pos_y, a.dst_h, a.src_h, y0 + tid - 32);
        s_yhi[tid - 32] = anchor_bound<true>(a.pos_y, a.dst_h, a.src_h, y0 + tid - 32);
    }
    __syncthreads();
    // candidate outputs of the tile: [X0, X1) x [Y0, Y1), staged in passes of whole rows (a single row cut into column runs
    // when one row does not fit), so a thread visits its candidates in canonical order
    const int X0 = s_xlo[0], X1 = max(s_xhi[tw - 1], X0), Y0 = s_ylo[0], Y1 = max(s_yhi[th - 1], Y0);
    const int nx = X1 - X0;
    const int cols_per = min(nx, RG_CAND), rows_per = nx <= RG_CAND ? RG_CAND / max(nx, 1) : 1;
    const int txl = tid % RG_TW, tyl = tid / RG_TW;
    const bool live = txl < tw && tyl < th;
    const int xl = live ? s_xlo[txl] : 0, xh = live ? s_xhi[txl] : 0;
    const int yl = live ? s_ylo[tyl] : 0, yh = live ? s_yhi[tyl] : 0;
    const int me = tyl * RG_TW + txl;
    const float s = a.s;

    for (int plane = blockIdx.y; plane < a.p.n_planes; plane += gridDim.y) {
        const T* __restrict__ src = static_cast<const T*>(a.p.src) + (long long)plane * a.p.src_stride;
        const T* __restrict__ yp = static_cast<const T*>(a.p.y) + (long long)plane * a.p.y_stride;
        const float* __restrict__ gp = a.p.g + (long long)plane * a.p.g_stride;
        __syncthreads(); // the previous plane's tile is no longer read
        for (int e = tid; e < (th + 2) * RG_HW; e += RG_THREADS) {
            const int r = e / RG_HW, c = e - r * RG_HW;
            const int sy = min(max(y0 - 1 + r, 0), a.src_h - 1), sxx = min(max(x0 - 1 + c, 0), a.src_w - 1);
            s_src[e] = widen<T>(__ldg(src + (long long)sy * a.p.src_pitch + sxx));
        }
        float acc = 0.f;
        bool any = false;
        for (int cy0 = Y0; cy0 < Y1; cy0 += rows_per) {
            const int cy1 = min(cy0 + rows_per, Y1);
            for (int cx0 = X0; cx0 < X1; cx0 += cols_per) {
                const int cw = min(cols_per, X1 - cx0);
                __syncthreads(); // the source tile is staged; the previous pass's candidates are no longer read
                for (int e = tid; e < (cy1 - cy0) * cw; e += RG_THREADS) {
                    const int row = cy0 + e / cw, x = cx0 + e % cw;
                    const int ax0 = anchor0(a.pos_x, x, a.src_w), ax1 = anchor1(a.pos_x, x, a.src_w);
                    const int ay0 = anchor0(a.pos_y, row, a.src_h), ay1 = anchor1(a.pos_y, row, a.src_h);
                    const float* r0 = s_src + (ay0 - y0 + 1) * RG_HW - x0 + 1;
                    const float* r1 = s_src + (ay1 - y0 + 1) * RG_HW - x0 + 1;
                    const float a0 = r0[ax0], a1 = r0[ax1], a2 = r1[ax0], a3 = r1[ax1];
                    const float lo = fminf(fminf(a0, a1), fminf(a2, a3)), hi = fmaxf(fmaxf(a0, a1), fmaxf(a2, a3));
                    const float y = widen<T>(__ldg(yp + (long long)row * a.p.y_pitch + x));
                    int code = -1;
                    float v = 0.f;
                    if (y < lo || y > hi) {
                        const float b = y < lo ? lo : hi;
                        const int k = a0 == b ? 0 : a1 == b ? 1 : a2 == b ? 2 : 3;
                        const int lx = ((k & 1) ? ax1 : ax0) - x0, ly = ((k & 2) ? ay1 : ay0) - y0;
                        if (lx >= 0 && lx < tw && ly >= 0 && ly < th) {
                            const float g = __ldg(gp + (long long)row * a.p.g_pitch + x);
                            code = ly * RG_TW + lx;
                            v = s == 1.f ? g : __fmul_rn(s, g);
                        }
                    }
                    s_code[e] = code;
                    s_val[e] = v;
                }
                __syncthreads();
                if (live) {
                    for (int row = max(yl, cy0); row < min(yh, cy1); ++row)
                        for (int x = max(xl, cx0); x < min(xh, cx0 + cw); ++x) {
                            const int e = (row - cy0) * cw + x - cx0;
                            if (s_code[e] == me) {
                                acc = any ? __fadd_rn(acc, s_val[e]) : s_val[e];
                                any = true;
                            }
                        }
                }
            }
        }
        if (any) {
            float* o = a.p.gs + (long long)plane * a.p.gs_stride + (long long)(y0 + tyl) * a.p.gs_pitch + x0 + txl;
            *o = __fadd_rn(*o, acc);
        }
    }
}

template <typename T>
int launch_typed(ArAdjArgs a, const jinc_table* t, cudaStream_t st, int* launches)
{
    constexpr int COLS = 32 * (16 / (int)sizeof(T));
    a.col_tiles = (a.dst_w + COLS - 1) / COLS;
    const int row_tiles = (a.dst_h + GO_ROWS - 1) / GO_ROWS;
    antiring_grad_out<T><<<dim3((unsigned)(a.col_tiles * row_tiles), (unsigned)std::min(a.n_rec, 65535), (unsigned)a.per),
                           GO_THREADS, 0, st>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess)
        return jinc_fail(JINC_E_CUDA, "antiring_grad_out launch failed: %s", cudaGetErrorString(e));
    ++*launches;
    const ArAdjPlanes& p = a.p;
    if (int rc = jinc_launch_adjoint(t, p.n_planes, p.gy, p.gy_pitch, p.gy_stride, p.gs, p.gs_pitch, p.gs_stride, st, launches))
        return rc;
    a.tiles_x = (a.src_w + RG_TW - 1) / RG_TW;
    const unsigned tiles = (unsigned)(a.tiles_x * ((a.src_h + RG_TH - 1) / RG_TH));
    antiring_route_gather<T><<<dim3(tiles, (unsigned)std::min(p.n_planes, 65535)), RG_THREADS, 0, st>>>(a);
    e = cudaGetLastError();
    if (e != cudaSuccess)
        return jinc_fail(JINC_E_CUDA, "antiring_route_gather launch failed: %s", cudaGetErrorString(e));
    ++*launches;
    return JINC_OK;
}

// [lo, hi) bytes of n planes of `rows` rows of `row_bytes` each
void plane_span(const void* base, int n, ptrdiff_t stride, long long rows, ptrdiff_t pitch, long long row_bytes, uintptr_t& lo,
                uintptr_t& hi)
{
    lo = reinterpret_cast<uintptr_t>(base);
    hi = lo + (uintptr_t)((n - 1) * (long long)stride + (rows - 1) * pitch + row_bytes);
}

} // namespace

int jinc_launch_antiring_adjoint(const jinc_table* t, int sample, float strength, const ArAdjPlanes& p, cudaStream_t st,
                                 int* launches)
{
    const int h = t->sc.dst_h, w = t->sc.dst_w;
    if (strength == 0.f) { // g_y = g bit for bit, nothing routed: the plain adjoint
        if (p.n_planes == 1 || (p.g_stride == h * p.g_pitch && p.gy_stride == h * p.gy_pitch)) {
            JINC_CUDA(cudaMemcpy2DAsync(p.gy, p.gy_pitch * 4, p.g, p.g_pitch * 4, (size_t)w * 4, (size_t)h * p.n_planes,
                                        cudaMemcpyDeviceToDevice, st));
        } else {
            for (int i = 0; i < p.n_planes; ++i)
                JINC_CUDA(cudaMemcpy2DAsync(p.gy + i * p.gy_stride, p.gy_pitch * 4, p.g + i * p.g_stride, p.g_pitch * 4,
                                            (size_t)w * 4, (size_t)h, cudaMemcpyDeviceToDevice, st));
        }
        return jinc_launch_adjoint(t, p.n_planes, p.gy, p.gy_pitch, p.gy_stride, p.gs, p.gs_pitch, p.gs_stride, st, launches);
    }
    ArAdjArgs a;
    memset(&a, 0, sizeof(a));
    a.p = p;
    a.pos_x = t->ax[0].pos;
    a.pos_y = t->ax[1].pos;
    a.src_w = t->sc.src_w;
    a.src_h = t->sc.src_h;
    a.dst_w = w;
    a.dst_h = h;
    a.per = JINC_MAX_PLANES; // records of up to four planes, as the forward's
    while (p.n_planes % a.per)
        --a.per;
    a.n_rec = p.n_planes / a.per;
    a.s = strength;
    return sample == 4 ? launch_typed<float>(a, t, st, launches) : launch_typed<__half>(a, t, st, launches);
}

extern "C" int jinc_antiring_adjoint_planes_device(jinc_ctx* ctx, const jinc_table* t, int sample_bytes, float strength,
                                                   int n_planes, const void* d_src, ptrdiff_t src_pitch,
                                                   ptrdiff_t src_plane_stride, const void* d_y, ptrdiff_t y_pitch,
                                                   ptrdiff_t y_plane_stride, const float* d_grad_dst, ptrdiff_t g_pitch,
                                                   ptrdiff_t g_plane_stride, float* d_grad_y, ptrdiff_t gy_pitch,
                                                   ptrdiff_t gy_plane_stride, float* d_grad_src, ptrdiff_t gs_pitch,
                                                   ptrdiff_t gs_plane_stride, void* stream)
{
    static const char* fn = "jinc_antiring_adjoint_planes_device";
    if (!ctx || !t || !d_src || !d_y || !d_grad_dst || !d_grad_y || !d_grad_src)
        return jinc_fail(JINC_E_INVALID, "%s: null argument", fn);
    if (n_planes < 1)
        return jinc_fail(JINC_E_INVALID, "%s: n_planes must be at least 1", fn);
    if (sample_bytes != 4 && sample_bytes != JINC_SAMPLE_F16)
        return jinc_fail(JINC_E_INVALID, "%s: sample_bytes must be 4 or JINC_SAMPLE_F16 (only float planes have a gradient)", fn);
    if (!(strength >= 0.f && strength <= 1.f))
        return jinc_fail(JINC_E_INVALID, "%s: strength must be between 0.0 and 1.0", fn);
    const long long dw = t->sc.dst_w, dh = t->sc.dst_h, sw = t->sc.src_w, sh = t->sc.src_h;
    const int sz = jinc_sample_size(sample_bytes);
    struct Planes {
        const void* p;
        ptrdiff_t pitch, stride;
        long long w, h;
        int sz;
        const char* name;
    } pl[5] = {{d_src, src_pitch, src_plane_stride, sw, sh, sz, "d_src"},
               {d_y, y_pitch, y_plane_stride, dw, dh, sz, "d_y"},
               {d_grad_dst, g_pitch, g_plane_stride, dw, dh, 4, "d_grad_dst"},
               {d_grad_y, gy_pitch, gy_plane_stride, dw, dh, 4, "d_grad_y"},
               {d_grad_src, gs_pitch, gs_plane_stride, sw, sh, 4, "d_grad_src"}};
    uintptr_t lo[5], hi[5];
    for (int i = 0; i < 5; ++i) {
        const Planes& q = pl[i];
        if (reinterpret_cast<uintptr_t>(q.p) % q.sz || q.pitch % q.sz || q.pitch < q.w * q.sz)
            return jinc_fail(JINC_E_INVALID, "%s: %s must be aligned to its sample size, with a pitch that is a multiple of it "
                                             "and holds a row", fn, q.name);
        if (n_planes > 1 && (q.stride % q.sz || q.stride < q.h * q.pitch))
            return jinc_fail(JINC_E_INVALID, "%s: the plane stride of %s must be a multiple of its sample size and hold a plane",
                             fn, q.name);
        plane_span(q.p, n_planes, q.stride, q.h, q.pitch, q.w * q.sz, lo[i], hi[i]);
    }
    if ((lo[4] < hi[2] && lo[2] < hi[4]) || (lo[4] < hi[3] && lo[3] < hi[4]))
        return jinc_fail(JINC_E_INVALID, "%s: d_grad_src must not overlap d_grad_dst or d_grad_y", fn);
    if (lo[3] < hi[2] && lo[2] < hi[3])
        return jinc_fail(JINC_E_INVALID, "%s: d_grad_y must not overlap d_grad_dst", fn);
    JINC_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    const long long ssz = sz;
    ArAdjPlanes p{d_src, src_pitch / ssz, src_plane_stride / ssz, d_y, y_pitch / ssz, y_plane_stride / ssz,
                  d_grad_dst, g_pitch / 4, g_plane_stride / 4, d_grad_y, gy_pitch / 4, gy_plane_stride / 4,
                  d_grad_src, gs_pitch / 4, gs_plane_stride / 4, n_planes};
    int launches = 0;
    return jinc_launch_antiring_adjoint(t, sample_bytes, strength, p, st, &launches);
}
