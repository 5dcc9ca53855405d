// jinc_up2x.cuh -- exact-2x interior kernel (see jinc_resample.cuh for the layout); included by jinc_up2x_<type>.cu,
// which instantiates launch_up2x for one sample type.
#ifndef JINC_UP2X_CUH
#define JINC_UP2X_CUH

#include <cstdlib>
#include <utility>

#include "jinc_resample.cuh"
#include "jinc_up2x_taps.h"

namespace jinc_rs {

constexpr int UP_UNROLL_MAX_FS = 9; // windows up to this size get a fully unrolled row loop

// ---- bulk-copy (TMA engine) staging of float tiles: raw rows land in shared memory asynchronously, one cp.async.bulk per
//      tile row, all completing on one mbarrier; the pair layout is then made from shared memory instead of from
//      registers filled by LDG.  Opt-in (JINCRESIZE_B200_TMA=1): measured against the register path in DESIGN.md 4.1.
template <int FS>
struct UpTma {
    using G = UpGeom<FS>;
    static constexpr int RAWC = (G::NC + 4 + 3) & ~3;  // floats per landed row: the tile's columns from an aligned start
    static constexpr int ROWS = G::NR + 1;             // raw rows (pair row r needs rows r and r + 1)
    static constexpr size_t LANDING = (size_t)ROWS * RAWC * sizeof(float);
    static constexpr size_t SMEM = G::SMEM + LANDING + 16; // + the mbarrier
};

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes),
                 "r"(bar)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok)
                 : "r"(bar), "r"(parity)
                 : "memory");
    return ok != 0;
}

// One pair row of the tile applied to the thread's 16 accumulators: phase row 0 uses weight row rr, phase row 1 uses
// weight row rr - OY1.  Bit lx of C<py><px> clear: column lx of that phase's weight row is exactly zero and emits no FFMA2
// (nor the LDS of a pair column no live tap reads); the remaining taps keep their order.
template <int FS, int OX1, int OY1, uint32_t C00 = ~0u, uint32_t C01 = ~0u, uint32_t C10 = ~0u, uint32_t C11 = ~0u>
__device__ __forceinline__ void up_row(const float2* __restrict__ trow, int rr, const UpWeights<FS>& W, float2 (&acc)[2][2][UP_TX])
{
    using G = UpGeom<FS>;
    float2 seg[G::NSEG];
#pragma unroll
    for (int m = 0; m < G::NSEG; ++m)
        seg[m] = trow[(m & 3) * G::SUB + (m >> 2)]; // column 4*lane + m

    if (OY1 == 0 || rr < FS) { // phase row 0: ly = rr
#pragma unroll
        for (int lx = 0; lx < FS; ++lx) {
            const float w0 = W.w[0][0][rr][lx], w1 = W.w[0][1][rr][lx];
#pragma unroll
            for (int i = 0; i < UP_TX; ++i) {
                if ((C00 >> lx) & 1)
                    acc[0][0][i] = __ffma2_rn(seg[i + lx], make_float2(w0, w0), acc[0][0][i]);
                if ((C01 >> lx) & 1)
                    acc[0][1][i] = __ffma2_rn(seg[i + OX1 + lx], make_float2(w1, w1), acc[0][1][i]);
            }
        }
    }
    const int ly1 = rr - OY1; // phase row 1
    if (OY1 == 0 || rr >= OY1) {
#pragma unroll
        for (int lx = 0; lx < FS; ++lx) {
            const float w0 = W.w[1][0][ly1][lx], w1 = W.w[1][1][ly1][lx];
#pragma unroll
            for (int i = 0; i < UP_TX; ++i) {
                if ((C10 >> lx) & 1)
                    acc[1][0][i] = __ffma2_rn(seg[i + lx], make_float2(w0, w0), acc[1][0][i]);
                if ((C11 >> lx) & 1)
                    acc[1][1][i] = __ffma2_rn(seg[i + OX1 + lx], make_float2(w1, w1), acc[1][1][i]);
            }
        }
    }
}

// Every pair row of a small window, each with the live columns of tap-mask variant M as compile-time constants (a mask
// read inside a run-time row loop would keep that loop rolled)
template <int FS, int OX1, int OY1, int M, int... RR>
__device__ __forceinline__ void up_rows(const float2* __restrict__ trow, const UpWeights<FS>& W, float2 (&acc)[2][2][UP_TX],
                                        std::integer_sequence<int, RR...>)
{
    using K = UpTaps<FS, M>;
    (up_row<FS, OX1, OY1, K::cols(0, 0, RR), K::cols(0, 1, RR), K::cols(1, 0, RR - OY1), K::cols(1, 1, RR - OY1)>(
         trow + RR * UpGeom<FS>::NCP, RR, W, acc),
     ...);
}

template <typename T, int FS, int OX1, int OY1, bool TMA = false, int M = 0>
__global__ void __launch_bounds__(UP_THREADS, (FS >= 13 ? 4 : FS <= 7 ? 5 : 6))
    resample_up2x(const __grid_constant__ UpArgs a, const __grid_constant__ UpWeights<FS> W)
{
    using G = UpGeom<FS>;
    extern __shared__ __align__(16) unsigned char smem_raw[];

    unsigned role_id;
    if (block_role(blockIdx.x, (unsigned)a.strip_blocks, a.strip_shift, role_id)) {
        // ---------------- strip role
        // samples two outputs apart, origins one apart; whole-frame launches run from the table's strip plan
        if (a.st.plan_patches)
            strip_block_planned<T, FS, UP_THREADS, UP_STRIP_SPT, 1>(a.st, a.fr, role_id, reinterpret_cast<float*>(smem_raw));
        else
            strip_block_unplanned<T, FS, UP_THREADS, UP_STRIP_SPT, 2, 1>(a.st, a.fr, role_id, reinterpret_cast<float*>(smem_raw));
        return;
    }

    // -------------------- interior tile role
    float2* tile = reinterpret_cast<float2*>(smem_raw); // [NR][4][SUB] pairs {S[r][c], S[r+1][c]}
    const int plane = (int)div_by(role_id, a.tiles_per_plane_magic);
    const int tidx = role_id - plane * a.tiles_per_plane;
    const int tile_y = (int)div_by((unsigned)tidx, a.tiles_x_magic), tile_x = tidx - tile_y * a.tiles_x;
    const PlanePtrs& pp = frame_ptrs(a.fr);
    const T* __restrict__ src = static_cast<const T*>(pp.src[plane]);
    T* __restrict__ dst = static_cast<T*>(pp.dst[plane]);
    const long long sp = pp.src_pitch[plane], dp = pp.dst_pitch[plane];

    const int cell_x0 = tile_x * UP_CW; // first cell of this tile
    const int cell_y0 = a.cy_begin + tile_y * G::CH;
    const int tsx = a.sx0 + cell_x0, tsy = a.sy0 + cell_y0; // source coordinates of tile(0,0)

    // ---- stage the source tile: every row is paired with the one below it and converted to float once.  A thread owns
    //      one 4-sample group per row over a segment of rows and issues ALL its loads before the first conversion (one
    //      memory round trip per tile).  When the plane base and pitch allow it the groups are aligned vector loads
    //      (4 samples per LDG); the tile columns then start d = tsx & 3 samples into the first group.
    const bool vec_ok = ((reinterpret_cast<uintptr_t>(src) | (uintptr_t)(sp * (long long)sizeof(T))) & (4 * sizeof(T) - 1)) == 0;
    if constexpr (TMA) {
        static_assert(std::is_same<T, float>::value, "bulk-copy staging lands float rows");
        // One cp.async.bulk per raw tile row (a contiguous, 16-byte aligned segment of the plane row: vec_ok is required by the
        // launcher), issued by the lanes of warp 0, all completing on one mbarrier.  The segment is cut at the end of the
        // plane row; what lies beyond only feeds discarded cells.
        using TM = UpTma<FS>;
        const uint32_t bar = smem_addr(smem_raw + G::SMEM + TM::LANDING);
        const int x_al = tsx & ~3;
        const int len = min(TM::RAWC, (int)sp - x_al) & ~3; // floats per row copy
        if (threadIdx.x == 0)
            mbar_init(bar, 1);
        __syncthreads();
        if (threadIdx.x < 32) {
            if (threadIdx.x == 0)
                mbar_expect_tx(bar, (uint32_t)(TM::ROWS * len * (int)sizeof(float)));
            for (int r = threadIdx.x; r < TM::ROWS; r += 32) {
                const T* row = src + (long long)min(max(tsy + r, 0), a.src_h - 1) * sp + x_al;
                bulk_g2s(smem_addr(smem_raw + G::SMEM + (size_t)r * TM::RAWC * sizeof(float)), row, (uint32_t)(len * (int)sizeof(float)), bar);
            }
        }
        unsigned spins = 0;
        while (!mbar_try_wait(bar, 0))
            if (++spins > (1u << 24))
                __trap(); // a transfer that never completes must not hang the device
    }
    if (vec_ok) {
        using V = typename Vec4Of<T>::type;
        constexpr int GRP = G::SUB + 1;                 // groups per row (one more: the row starts inside a group)
        constexpr int SEGS = UP_THREADS / GRP;          // row segments
        constexpr int ROWS = (G::NR + SEGS - 1) / SEGS; // pair rows per segment
        const int q = threadIdx.x % GRP, seg = threadIdx.x / GRP;
        if (seg < SEGS) {
            const int d = tsx & 3;
            const int g = min(max((tsx >> 2) + q, 0), (a.src_w - 1) >> 2); // groups outside the plane only feed discarded cells
            const int r0 = seg * ROWS;
            V raw[ROWS + 1];
            if constexpr (TMA) {
                // the rows were landed by the bulk-copy engine (below): group q of landed row r0 + j
                const V* __restrict__ landed = reinterpret_cast<const V*>(smem_raw + G::SMEM);
#pragma unroll
                for (int j = 0; j <= ROWS; ++j)
                    raw[j] = landed[min(r0 + j, UpTma<FS>::ROWS - 1) * (UpTma<FS>::RAWC / 4) + q];
            } else {
#pragma unroll
                for (int j = 0; j <= ROWS; ++j) {
                    const T* row = src + (long long)min(max(tsy + r0 + j, 0), a.src_h - 1) * sp;
                    raw[j] = __ldg(reinterpret_cast<const V*>(row) + g);
                }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int cc = k - d;                      // tile column of sample k is 4 q + cc
                const int idx = q + (cc >> 2);
                if (idx >= 0 && idx < G::SUB) {
                    float2* out = tile + (r0 * 4 + (cc & 3)) * G::SUB + idx;
                    float prev = vec4_sample<T>(raw[0], k);
#pragma unroll
                    for (int j = 0; j < ROWS; ++j) {
                        const float cur = vec4_sample<T>(raw[j + 1], k);
                        if (r0 + j < G::NR)
                            out[j * 4 * G::SUB] = make_float2(prev, cur);
                        prev = cur;
                    }
                }
            }
        }
    } else {
        constexpr int SEGS = UP_THREADS / G::SUB;       // row segments
        constexpr int ROWS = (G::NR + SEGS - 1) / SEGS; // pair rows per segment
        const int q = threadIdx.x % G::SUB, seg = threadIdx.x / G::SUB;
        if (seg < SEGS) {
            int xo[4];
#pragma unroll
            for (int k = 0; k < 4; ++k)
                xo[k] = min(max(tsx + 4 * q + k, 0), a.src_w - 1); // out-of-plane taps only feed discarded cells
            const int r0 = seg * ROWS;
            T raw[ROWS + 1][4];
#pragma unroll
            for (int j = 0; j <= ROWS; ++j) {
                const T* row = src + (long long)min(max(tsy + r0 + j, 0), a.src_h - 1) * sp;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    raw[j][k] = __ldg(row + xo[k]);
            }
#pragma unroll
            for (int j = 0; j < ROWS; ++j) {
                if (r0 + j < G::NR) {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        tile[((r0 + j) * 4 + k) * G::SUB + q] = make_float2(sample_to_float(raw[j][k]), sample_to_float(raw[j + 1][k]));
                }
            }
        }
    }
    __syncthreads();

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

#pragma unroll 1
    for (int rp = warp; rp < UP_WARPS * G::RPW; rp += UP_WARPS) {
        const int cy = cell_y0 + 2 * rp; // first cell row of the pair
        if (cy >= a.cy_end)
            break;
        float2 acc[2][2][UP_TX];
#pragma unroll
        for (int py = 0; py < 2; ++py)
#pragma unroll
            for (int px = 0; px < 2; ++px)
#pragma unroll
                for (int i = 0; i < UP_TX; ++i)
                    acc[py][px][i] = make_float2(0.f, 0.f);

        const float2* trow = tile + (size_t)(2 * rp) * G::NCP + lane;
        if constexpr (FS <= UP_UNROLL_MAX_FS) {
            // small windows: the row loop is unrolled completely, so every weight has a fixed constant-bank address
            // and there is no loop control between the FFMA2 runs
            up_rows<FS, OX1, OY1, M>(trow, W, acc, std::make_integer_sequence<int, FS + OY1>{});
        } else {
            static_assert(M == 0, "tap masks need the unrolled row loop");
#pragma unroll 1
            for (int rr = 0; rr < FS + OY1; ++rr, trow += G::NCP)
                up_row<FS, OX1, OY1>(trow, rr, W, acc);
        }

        // ---- epilogue: 4 output rows x 8 consecutive samples per thread
        const int cx = cell_x0 + UP_TX * lane;
        if (cx >= a.ncx)
            continue;
        const int ox = a.x0 + 2 * cx;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (cy + h < a.cy_end) {
#pragma unroll
                for (int py = 0; py < 2; ++py) {
                    float v[8];
#pragma unroll
                    for (int i = 0; i < UP_TX; ++i) {
                        v[2 * i] = h ? acc[py][0][i].y : acc[py][0][i].x;
                        v[2 * i + 1] = h ? acc[py][1][i].y : acc[py][1][i].x;
                    }
                    T* o = dst + (long long)(a.y0 + 2 * (cy + h) + py) * dp + ox;
                    if (cx + UP_TX <= a.ncx) {
                        store8<T>(o, v, a.fr.peak);
                    } else {
                        const int nk = 2 * (a.ncx - cx);
#pragma unroll
                        for (int k = 0; k < 8; ++k)
                            if (k < nk)
                                o[k] = finish<T>(v[k], a.fr.peak);
                    }
                }
            }
        }
    }
}

// float planes staged by the bulk-copy engine: instantiated in its own translation unit (jinc_up2x_f32_bulk.cu)
int launch_up2x_bulkcopy(const jinc_table* t, UpArgs& a, long long strip_blocks, int n_frames, cudaStream_t st);

// M = 0: every tap, for the table's (ox1, oy1); M > 0: the tap-mask variant UpTaps<FS, M>, whose (ox1, oy1) the table has
template <typename T, int FS, bool TMA, int M = 0>
int launch_up2x_fs(const jinc_table* t, UpArgs& a, long long strip_blocks, int n_frames, cudaStream_t st)
{
    using G = UpGeom<FS>;
    const Up2xPlan& u = t->up2x;
    UpWeights<FS> w;
    memset(&w, 0, sizeof(w));
    for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px) {
            const float* blk = t->h_weights.data() + (size_t)u.wblock[py][px] * FS * FS;
            for (int ly = 0; ly < FS; ++ly)
                for (int lx = 0; lx < FS; ++lx)
                    w.w[py][px][ly][lx] = blk[ly * FS + lx];
        }
    void (*kern)(UpArgs, UpWeights<FS>);
    if constexpr (M == 0)
        kern = u.ox1 ? (u.oy1 ? resample_up2x<T, FS, 1, 1, TMA> : resample_up2x<T, FS, 1, 0, TMA>)
                     : (u.oy1 ? resample_up2x<T, FS, 0, 1, TMA> : resample_up2x<T, FS, 0, 0, TMA>);
    else
        kern = resample_up2x<T, FS, UpTaps<FS, M>::OX1, UpTaps<FS, M>::OY1, TMA, M>;
    size_t smem = G::SMEM;
    if constexpr (TMA)
        smem = UpTma<FS>::SMEM;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess)
        return jinc_fail(JINC_E_CUDA, "cudaFuncSetAttribute(up2x smem %zu): %s", smem, cudaGetErrorString(e));
    a.strip_blocks = (int)strip_blocks;
    a.strip_shift = strip_role_shift(a.interior_blocks, strip_blocks);
    dim3 grid((unsigned)(a.interior_blocks + strip_blocks), n_frames, 1);
    kern<<<grid, UP_THREADS, smem, st>>>(a, w);
    e = cudaGetLastError();
    if (e != cudaSuccess)
        return jinc_fail(JINC_E_CUDA, "resample_up2x launch failed: %s", cudaGetErrorString(e));
    return JINC_OK;
}

template <typename T, bool TMA>
int launch_up2x_any(const jinc_table* t, UpArgs& a, long long strip_blocks, int n_frames, cudaStream_t st)
{
    switch (t->sc.fs) {
    case 7: return launch_up2x_fs<T, 7, TMA>(t, a, strip_blocks, n_frames, st);   // tap 3  (Jinc36Resize)
    case 9: return launch_up2x_fs<T, 9, TMA>(t, a, strip_blocks, n_frames, st);   // tap 4  (Jinc64Resize)
    case 11: return launch_up2x_fs<T, 11, TMA>(t, a, strip_blocks, n_frames, st); // tap 5
    case 13: return launch_up2x_fs<T, 13, TMA>(t, a, strip_blocks, n_frames, st); // tap 6  (Jinc144Resize)
    case 15: return launch_up2x_fs<T, 15, TMA>(t, a, strip_blocks, n_frames, st); // tap 7
    case 17: return launch_up2x_fs<T, 17, TMA>(t, a, strip_blocks, n_frames, st); // tap 8  (Jinc256Resize)
    default: return 1;
    }
}

// integer planes of a table with a tap-mask variant (Up2xPlan::taps): one translation unit per (type, fs),
// jinc_up2x_taps_<type>_fs<fs>.cu
template <typename T, int FS>
int launch_up2x_taps(const jinc_table* t, UpArgs& a, long long strip_blocks, int n_frames, cudaStream_t st)
{
    switch (t->up2x.taps) {
    case 1: return launch_up2x_fs<T, FS, false, 1>(t, a, strip_blocks, n_frames, st);
    case 2: return launch_up2x_fs<T, FS, false, 2>(t, a, strip_blocks, n_frames, st);
    case 3: return launch_up2x_fs<T, FS, false, 3>(t, a, strip_blocks, n_frames, st);
    case 4: return launch_up2x_fs<T, FS, false, 4>(t, a, strip_blocks, n_frames, st);
    case 5: return launch_up2x_fs<T, FS, false, 5>(t, a, strip_blocks, n_frames, st);
    case 6: return launch_up2x_fs<T, FS, false, 6>(t, a, strip_blocks, n_frames, st);
    case 7: return launch_up2x_fs<T, FS, false, 7>(t, a, strip_blocks, n_frames, st);
    default: return jinc_fail(JINC_E_INVALID, "resample_up2x: no tap-mask variant %d for fs %d", t->up2x.taps, FS);
    }
}
static_assert(UP_TAP_VARIANTS == 8, "launch_up2x_taps dispatches variants 1..7");
extern template int launch_up2x_taps<uint8_t, 7>(const jinc_table*, UpArgs&, long long, int, cudaStream_t);
extern template int launch_up2x_taps<uint8_t, 9>(const jinc_table*, UpArgs&, long long, int, cudaStream_t);
extern template int launch_up2x_taps<uint16_t, 7>(const jinc_table*, UpArgs&, long long, int, cudaStream_t);
extern template int launch_up2x_taps<uint16_t, 9>(const jinc_table*, UpArgs&, long long, int, cudaStream_t);

template <typename T>
int launch_up2x(const jinc_table* t, UpArgs& a, long long strip_blocks, int n_frames, cudaStream_t st)
{
    if constexpr (!is_float_sample<T>::value) {
        // float and half planes always take every tap: 0 * Inf and 0 * NaN must reach the output as they do in the reference
        if (t->up2x.taps > 0) {
            if (t->sc.fs == 7)
                return launch_up2x_taps<T, 7>(t, a, strip_blocks, n_frames, st);
            if (t->sc.fs == 9)
                return launch_up2x_taps<T, 9>(t, a, strip_blocks, n_frames, st);
        }
    }
    if constexpr (std::is_same<T, float>::value) { // half planes ignore the switch: the landed rows are float rows
        const char* tma_env = getenv("JINCRESIZE_B200_TMA");
        if (tma_env && tma_env[0] == '1' && up2x_supported(t->sc.fs)) {
            // bulk-copy staging needs 16-byte aligned plane rows in every frame; batched launches (device-side plane
            // records) are the caller's promise, single frames are checked here
            bool aligned = true;
            if (!a.fr.frames)
                for (int i = 0; i < a.fr.n_planes; ++i)
                    aligned = aligned && ((reinterpret_cast<uintptr_t>(a.fr.one.src[i]) | (uintptr_t)(a.fr.one.src_pitch[i] * 4)) & 15) == 0;
            if (aligned)
                return launch_up2x_bulkcopy(t, a, strip_blocks, n_frames, st);
        }
    }
    return launch_up2x_any<T, false>(t, a, strip_blocks, n_frames, st);
}

} // namespace jinc_rs

#endif
