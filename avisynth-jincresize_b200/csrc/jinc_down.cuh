// jinc_down.cuh -- integer-ratio downscale interior kernel; included by jinc_down_<type>.cu, which instantiates
// launch_down for one sample type.
#ifndef JINC_DOWN_CUH
#define JINC_DOWN_CUH

#include "jinc_resample.cuh"

namespace jinc_rs {

template <int CVT>
__device__ __forceinline__ float2 down_cvt(uint32_t w)
{
    if (CVT == DN_CVT_PRMT)
        return make_float2(__uint_as_float(__byte_perm(w, 0x3F000000u, 0x7104)), __uint_as_float(__byte_perm(w, 0x3F000000u, 0x7324)));
    return make_float2((float)(w & 0xffffu), (float)(w >> 16));
}
template <int CVT>
__device__ __forceinline__ float2 down_cvt(float2 w)
{
    return w;
}

template <typename T>
__device__ __forceinline__ void down_pack(uint32_t& out, const T* r0, const T* r1, int sh)
{
    out = ((uint32_t)__ldg(r0) << sh) | ((uint32_t)__ldg(r1) << (16 + sh));
}
__device__ __forceinline__ void down_pack(float2& out, const float* r0, const float* r1, int)
{
    out = make_float2(__ldg(r0), __ldg(r1));
}
__device__ __forceinline__ void down_pack(float2& out, const __half* r0, const __half* r1, int)
{
    out = make_float2(__half2float(__ldg(r0)), __half2float(__ldg(r1)));
}

template <typename T, int N>
__device__ __forceinline__ void store_run(T* p, const float (&v)[N], float peak)
{
    static_assert(N % 4 == 0, "runs are multiples of four samples");
#pragma unroll
    for (int q = 0; q < N; q += 4) {
        if constexpr (std::is_same<T, float>::value) {
            *reinterpret_cast<float4*>(p + q) = make_float4(v[q], v[q + 1], v[q + 2], v[q + 3]);
        } else if constexpr (std::is_same<T, __half>::value) {
            *reinterpret_cast<uint2*>(p + q) = make_uint2(pack_half2(v[q], v[q + 1]), pack_half2(v[q + 2], v[q + 3]));
        } else if constexpr (sizeof(T) == 2) {
            *reinterpret_cast<uint2*>(p + q) = make_uint2(finish_u16(v[q], peak) | (finish_u16(v[q + 1], peak) << 16),
                                                          finish_u16(v[q + 2], peak) | (finish_u16(v[q + 3], peak) << 16));
        } else {
            *reinterpret_cast<uint32_t*>(p + q) = finish_u8(v[q], peak) | (finish_u8(v[q + 1], peak) << 8) |
                                                  (finish_u8(v[q + 2], peak) << 16) | (finish_u8(v[q + 3], peak) << 24);
        }
    }
}

// one row pair of the thread's walk.  ALL: every output row of the thread is inside its window (no tests)
template <typename G, int FS, int Q, int NX, int NY, int CVT, bool ALL>
__device__ __forceinline__ void down_row_pair(const typename G::Word* __restrict__ trow, int k, const DownWeights<FS, Q>& W,
                                              float2 (&acc)[NY][NX])
{
#pragma unroll
    for (int p = 0; p < Q; ++p) {
        float2 s[G::SPAN];
#pragma unroll
        for (int m = 0; m < G::SPAN; ++m) {
            const int cc = Q * m + p;
            s[m] = down_cvt<CVT>(trow[(cc % G::D) * G::SUB + cc / G::D]);
        }
#pragma unroll
        for (int j = 0; j < NY; ++j) {
            const int kk = k - j * G::OFF1; // weight row pair of output row j
            if (ALL || (kk >= 0 && kk < (j == 0 ? G::NKW : G::NKW1))) {
#pragma unroll
                for (int m = 0; m < G::MT; ++m) {
                    if (Q * m + p < FS) {
                        const float2 w = W.w[G::ODD ? j : 0][kk][p][m];
#pragma unroll
                        for (int i = 0; i < NX; ++i)
                            acc[j][i] = __ffma2_rn(s[i + m], w, acc[j][i]);
                    }
                }
            }
        }
    }
}

template <typename T, int FS, int Q, int NX, int NY, int CVT, int NPASS>
__global__ void __launch_bounds__((DownGeom<T, FS, Q, NX, NY>::THREADS), 2)
    resample_down(const __grid_constant__ DownArgs a, const __grid_constant__ DownWeightsN<FS, Q, NPASS> WN)
{
    using G = DownGeom<T, FS, Q, NX, NY>;
    using Word = typename G::Word;
    extern __shared__ __align__(16) unsigned char smem_raw[];

    // blockIdx.z = pass (periodic paths); the border strips ride on pass 0
    const int pz = NPASS > 1 ? (int)blockIdx.z : 0;
    const DownPass& ps = a.pass[pz];
    const DownWeights<FS, Q>& W = WN.pass[pz];
    unsigned role_id;
    if (block_role(blockIdx.x, pz == 0 ? (unsigned)a.strip_blocks : 0u, a.strip_shift, role_id)) {
        if (NPASS == 1 && a.st.plan_patches) // whole-frame launch of an integer-ratio table: the strips run from its plan
            strip_block_planned<T, FS, G::THREADS, DN_STRIP_SPT, Q>(a.st, a.fr, role_id, reinterpret_cast<float*>(smem_raw));
        else
            strip_block<T, FS, G::THREADS, DN_STRIP_SPT>(a.st, a.fr, role_id, reinterpret_cast<float*>(smem_raw));
        return;
    }
    if (role_id >= (unsigned)a.interior_blocks)
        return; // grid positions of pass 0's strip blocks in the other passes
    Word* tile = reinterpret_cast<Word*>(smem_raw); // [NROWP][D][SUB] (+pad): word (k, c) at k*RS + (c%D)*SUB + c/D
    const int plane = (int)div_by(role_id, a.tiles_per_plane_magic);
    const int tidx = role_id - plane * a.tiles_per_plane;
    const int tile_y = (int)div_by((unsigned)tidx, a.tiles_x_magic), tile_x = tidx - tile_y * a.tiles_x;
    const PlanePtrs& pp = frame_ptrs(a.fr);
    const T* __restrict__ src = static_cast<const T*>(pp.src[plane]);
    T* __restrict__ dst = static_cast<T*>(pp.dst[plane]);
    const int sp = (int)pp.src_pitch[plane];
    const long long dp = pp.dst_pitch[plane];

    const int ox0 = a.x0 + tile_x * DN_TW, oy0 = a.y0 + tile_y * G::TH; // first output of the tile
    const int tsx = ps.tsx0 + Q * (tile_x * DN_TW), tsy = ps.tsy0 + Q * (tile_y * G::TH);

    // ---- stage the tile: a warp takes whole row pairs, a lane the columns lane + 32 q.  All loads of KU row pairs are
    //      issued before the first store so ~40 global loads per thread are in flight.
    {
        constexpr int NCOLS = G::D * G::SUB;
        constexpr int CQ = (NCOLS + 31) / 32;
        constexpr int KU = 2;
        const int sh = CVT == DN_CVT_PRMT ? a.pre_shift : 0;
        const int lane_ = threadIdx.x & 31, warp_ = threadIdx.x >> 5;
        int gx[CQ];
#pragma unroll
        for (int q = 0; q < CQ; ++q)
            gx[q] = min(max(tsx + lane_ + 32 * q, 0), a.src_w - 1); // clamped taps only feed masked outputs or zero weights
        for (int k0 = warp_; k0 < G::NROWP; k0 += KU * G::WARPS) {
            Word wv[KU][CQ];
#pragma unroll
            for (int u = 0; u < KU; ++u) {
                const int k = min(k0 + u * G::WARPS, G::NROWP - 1);
                const T* r0 = src + (long long)min(max(tsy + 2 * k, 0), a.src_h - 1) * sp;
                const T* r1 = src + (long long)min(max(tsy + 2 * k + 1, 0), a.src_h - 1) * sp;
#pragma unroll
                for (int q = 0; q < CQ; ++q)
                    down_pack(wv[u][q], r0 + gx[q], r1 + gx[q], sh);
            }
#pragma unroll
            for (int u = 0; u < KU; ++u) {
                const int k = k0 + u * G::WARPS;
                if (k < G::NROWP) {
#pragma unroll
                    for (int q = 0; q < CQ; ++q) {
                        const int c = lane_ + 32 * q;
                        if (NCOLS % 32 == 0 || c < NCOLS)
                            tile[k * G::RS + (c % G::D) * G::SUB + c / G::D] = wv[u][q];
                    }
                }
            }
        }
    }
    __syncthreads();

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int lx_ = lane % G::LX, ly_ = lane / G::LX;
    const int row0 = (warp * G::LY + ly_) * NY; // first output row of this thread inside the tile
    const Word* __restrict__ trow = tile + (size_t)((warp * G::LY + ly_) * G::HALF) * G::RS + lx_;

    float2 acc[NY][NX];
#pragma unroll
    for (int j = 0; j < NY; ++j)
#pragma unroll
        for (int i = 0; i < NX; ++i)
            acc[j][i] = make_float2(0.f, 0.f);

    constexpr int K_ALL0 = G::OFF1 * (NY - 1); // first row pair at which every output row is inside its window
    int k = 0;
#pragma unroll 1
    for (; k < K_ALL0; ++k, trow += G::RS)
        down_row_pair<G, FS, Q, NX, NY, CVT, false>(trow, k, W, acc);
#pragma unroll 1
    for (; k < G::NKW; ++k, trow += G::RS)
        down_row_pair<G, FS, Q, NX, NY, CVT, true>(trow, k, W, acc);
#pragma unroll 1
    for (; k < G::NK; ++k, trow += G::RS)
        down_row_pair<G, FS, Q, NX, NY, CVT, false>(trow, k, W, acc);

    // ---- epilogue: NY rows x NX consecutive samples
    const int ox = ox0 + NX * lx_;
    if (ox >= a.x1)
        return;
#pragma unroll
    for (int j = 0; j < NY; ++j) {
        const int oy = oy0 + row0 + j;
        if (oy >= a.y1)
            break;
        float v[NX];
#pragma unroll
        for (int i = 0; i < NX; ++i) {
            if (CVT == DN_CVT_PRMT)
                v[i] = ((acc[j][i].x - ps.bias_x[j]) + (acc[j][i].y - ps.bias_y[j])) * a.out_scale;
            else
                v[i] = acc[j][i].x + acc[j][i].y;
        }
        if (a.out_stride == 1) {
            T* o = dst + (long long)oy * dp + ox;
            if (ox + NX <= a.x1) {
                store_run<T, NX>(o, v, a.fr.peak);
            } else {
#pragma unroll
                for (int i = 0; i < NX; ++i)
                    if (ox + i < a.x1)
                        o[i] = finish<T>(v[i], a.fr.peak);
            }
        } else {
            // periodic pass: this sub-lattice owns every out_stride-th sample of every out_stride-th row
            T* o = dst + (long long)(ps.out_y0 + a.out_stride * (oy - a.y0)) * dp + (ps.out_x0 + a.out_stride * (ox - a.x0));
#pragma unroll
            for (int i = 0; i < NX; ++i)
                if (ox + i < a.x1)
                    o[i * a.out_stride] = finish<T>(v[i], a.fr.peak);
        }
    }
}

template <typename T, int FS, int Q, int NX, int NY, int CVT, int NPASS>
int launch_down_cfg(const jinc_table* t, DownArgs& a, const DownWeightsN<FS, Q, NPASS>& w, long long strip_blocks_of, int n_frames, cudaStream_t st,
                    const Rect* rects, int n_rects)
{
    using G = DownGeom<T, FS, Q, NX, NY>;
    long long strip_blocks =
        strip_blocks_of ? set_strip_rects(a.st, rects, n_rects, G::THREADS * DN_STRIP_SPT, DN_STRIP_MAX_PW, G::SMEM) * a.fr.n_planes : 0;
    if (strip_blocks_of && NPASS == 1 && a.want_strip_plan && attach_strip_plan(t, a.st, G::THREADS, DN_STRIP_SPT))
        strip_blocks = (long long)a.st.blocks_per_plane * a.fr.n_planes;
    a.tiles_x = (a.x1 - a.x0 + DN_TW - 1) / DN_TW;
    a.tiles_per_plane = a.tiles_x * ((a.y1 - a.y0 + G::TH - 1) / G::TH);
    a.tiles_x_magic = div_magic((unsigned)a.tiles_x);
    a.tiles_per_plane_magic = div_magic((unsigned)a.tiles_per_plane);
    if (a.interior_blocks)
        a.interior_blocks = a.tiles_per_plane * a.fr.n_planes;
    auto kern = resample_down<T, FS, Q, NX, NY, CVT, NPASS>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G::SMEM);
    if (e != cudaSuccess)
        return jinc_fail(JINC_E_CUDA, "cudaFuncSetAttribute(down smem %zu): %s", G::SMEM, cudaGetErrorString(e));
    if (a.interior_blocks + strip_blocks == 0)
        return 2;
    a.strip_blocks = (int)strip_blocks;
    a.strip_shift = strip_role_shift(a.interior_blocks, strip_blocks);
    a.n_passes = NPASS;
    dim3 grid((unsigned)(a.interior_blocks + strip_blocks), n_frames, NPASS);
    kern<<<grid, G::THREADS, G::SMEM, st>>>(a, w);
    e = cudaGetLastError();
    if (e != cudaSuccess)
        return jinc_fail(JINC_E_CUDA, "resample_down launch failed: %s", cudaGetErrorString(e));
    return JINC_OK;
}

constexpr int DN_NX = 8, DN_NY = 2; // outputs per thread

template <typename T, int FS, int Q, int NPASS>
int launch_down_fs(const jinc_table* t, DownArgs& a, const int* wblocks, bool want_strips, int n_frames, cudaStream_t st, const Rect* rects,
                   int n_rects)
{
    static_assert(sizeof(DownWeightsN<FS, Q, NPASS>) + sizeof(DownArgs) < 32000, "kernel parameters exceed the 32 KB limit");
    static_assert(NPASS <= DN_MAX_PASSES, "too many passes");
    DownWeightsN<FS, Q, NPASS> w;
    memset(&w, 0, sizeof(w));
    const int bits = is_float_sample<T>::value ? 32 : t_bits_from_peak(a.fr.peak);
    for (int ps = 0; ps < NPASS; ++ps) {
        const float* blk = t->h_weights.data() + (size_t)wblocks[ps] * FS * FS;
        // set 0 pairs rows (2k, 2k+1); set 1 (odd ratios) pairs rows (2k-1, 2k); sums per half for the PRMT bias
        double sum_x[2] = {0.0, 0.0}, sum_y[2] = {0.0, 0.0};
        for (int set = 0; set < DownWeights<FS, Q>::NSET; ++set)
            for (int ly = 0; ly < FS; ++ly)
                for (int lx = 0; lx < FS; ++lx) {
                    const float v = blk[ly * FS + lx];
                    const int r = ly + set; // row index inside the (shifted) pair grid
                    float2& e = w.pass[ps].w[set][r >> 1][lx % Q][lx / Q];
                    if (r & 1) {
                        e.y = v;
                        sum_y[set] += v;
                    } else {
                        e.x = v;
                        sum_x[set] += v;
                    }
                }
        if (DownWeights<FS, Q>::NSET == 1) {
            sum_x[1] = sum_x[0];
            sum_y[1] = sum_y[0];
        }
        for (int j = 0; j < 2; ++j) {
            a.pass[ps].bias_x[j] = (float)(0.5 * sum_x[j]);
            a.pass[ps].bias_y[j] = (float)(0.5 * sum_y[j]);
        }
    }
    if constexpr (is_float_sample<T>::value) { // half planes are staged as float pairs too
        return launch_down_cfg<T, FS, Q, DN_NX, DN_NY, DN_CVT_FLOAT, NPASS>(t, a, w, want_strips, n_frames, st, rects, n_rects);
    } else {
        if (bits <= 15) {
            // f = 0.5 + (x << pre_shift) / 65536  =>  sum(w f) = 0.5 sum(w) + sum(w x) * 2^(pre_shift - 16)
            a.pre_shift = 15 - bits;
            a.out_scale = (float)(1 << (16 - a.pre_shift));
            return launch_down_cfg<T, FS, Q, DN_NX, DN_NY, DN_CVT_PRMT, NPASS>(t, a, w, want_strips, n_frames, st, rects, n_rects);
        }
        if constexpr (sizeof(T) == 2)
            return launch_down_cfg<T, FS, Q, DN_NX, DN_NY, DN_CVT_I2F, NPASS>(t, a, w, want_strips, n_frames, st, rects, n_rects);
        return 1;
    }
}

// 0 launched, 2 nothing to do, 1 unsupported geometry, <0 error
template <typename T>
int launch_down(const jinc_table* t, DownArgs& a, int q, const int* wblocks, bool want_strips, int n_frames, cudaStream_t st,
                const Rect* rects, int n_rects)
{
    if (a.out_stride < 1)
        a.out_stride = 1;
    const int np = a.n_passes < 1 ? 1 : a.n_passes;
    const int key = np * 100000 + q * 1000 + t->sc.fs;
    switch (key) {
#define JINC_DOWN_CASE(NP_, Q_, FS_) \
    case NP_ * 100000 + Q_ * 1000 + FS_: return launch_down_fs<T, FS_, Q_, NP_>(t, a, wblocks, want_strips, n_frames, st, rects, n_rects);
        JINC_DOWN_CASE(16, 1, 7)  // tap 3, 4x upscale: sixteen unit-step passes in one launch
        JINC_DOWN_CASE(16, 1, 9)  // tap 4, 4x upscale
        JINC_DOWN_CASE(1, 2, 13)  // tap 3, 1/2
        JINC_DOWN_CASE(1, 2, 17)  // tap 4, 1/2
        JINC_DOWN_CASE(1, 2, 25)  // tap 6, 1/2
        JINC_DOWN_CASE(1, 2, 33)  // tap 8, 1/2
        JINC_DOWN_CASE(16, 3, 7)  // tap 3, 4:3 periodic: sixteen passes in one launch
        JINC_DOWN_CASE(16, 3, 9)  // tap 4, 4:3 periodic
        JINC_DOWN_CASE(4, 3, 10)  // tap 3, 2:3 periodic: four passes in one launch
        JINC_DOWN_CASE(4, 3, 13)  // tap 4, 2:3 periodic
        JINC_DOWN_CASE(1, 3, 20)  // tap 3, 1/3
        JINC_DOWN_CASE(1, 4, 26)  // tap 3, 1/4
        JINC_DOWN_CASE(1, 4, 34)  // tap 4, 1/4
        JINC_DOWN_CASE(1, 4, 50)  // tap 6, 1/4
#undef JINC_DOWN_CASE
    default: return 1;
    }
}

} // namespace jinc_rs

#endif
