// jinc_resample.cuh -- device code and argument blocks shared by the resample translation units.
//
// Replaces JincResize::resize_plane_c<T,thr,subsampled> (src/JincResize.cpp:536-601) and the three SIMD copies of
// its inner loop.  Every output sample is  sum_{ly,lx} src[start_y+ly][start_x+lx] * w[ly][lx]  over an fs x fs
// window, followed for integer formats by clamp to [0,peak] and round-half-even (:581-582); float is raw (:583-584).
//
// One launch covers ALL planes that share a coefficient table, for a whole BATCH of frames, interior and border
// together; blocks take one of two roles:
//
//   interior tile
//       exact 2x upscale (jinc_up2x.cuh, every "JincNNResize(2w,2h)" use): the table has 2x2 phase classes.  A thread
//       owns TX=4 source-aligned cells x 2 cell rows = 8x4 output samples in 16 float2 accumulators.  The source tile
//       lives in shared memory as VERTICAL PAIRS {S[r][c], S[r+1][c]} so one packed FFMA2 (fma.rn.f32x2, new on sm_100)
//       updates the same phase of two cell rows with a single scalar weight.  Weights arrive as kernel parameters
//       (constant bank) and reach the FMA pipe through uniform registers (LDCU -> FFMA2 R, R, UR, R): they cost no
//       shared-memory or register-file bandwidth.  Pair columns are de-interleaved by (c & 3) so a warp's LDS.64 is
//       bank-conflict free.
//       integer-ratio downscale and the passes of the periodic 2:3 / 4:3 paths (jinc_down.cuh): polyphase columns,
//       vertical tap pairing, raw sample pairs in shared memory.
//   strip patch (about 512 output samples of the border strips)
//       One thread = 4 output samples that share a border row or column (hence, normally, one weight block): the
//       patch's source footprint is staged in shared memory as floats, weights are read as float4 rows from the
//       per-class border blocks or the padded phase blocks.  Border pixels that fold into no class fall back to
//       resident per-pixel weights or to the reference's formula evaluated per tap (exact LUT index, divided by the
//       stored per-pixel normaliser, :443-514).  Whole-frame launches run the patches from the table's strip plan
//       (strip_block_planned: descriptors, thread records and packed weight blocks worked out once per table, the
//       weight blocks staged next to the footprint); row-band launches and tables without a plan derive the same
//       work per block (strip_block).  Both accumulate every sample in the same tap order.
//
// General ratios (no fast path) run resample_strips in jinc_resize.cu: the same patch scheme over the whole plane, one
// block covering the patch in every plane of the table.
//
// The kernels are split over several translation units (one per sample type and kernel family) so that the build
// runs in parallel; everything here is a template, inline, or a plain struct.
#ifndef JINC_RESAMPLE_CUH
#define JINC_RESAMPLE_CUH

#include <algorithm>
#include <cstring>
#include <type_traits>
#include <vector>

#include <cuda_fp16.h>

#include "jinc_internal.h"
#include "jinc_weights.cuh"

namespace jinc_rs {

// ------------------------------------------------------------------------------------------ sample conversion
//
// Four sample types: uint8_t, uint16_t (9..16 bits), float and __half (IEEE binary16).  Float planes -- float and half --
// keep the raw sum (no clamp, NaN and Inf propagated) and multiply every tap; half is converted to float when it is
// staged and rounded to nearest-even when it is stored, so a half plane runs the float inner loops unchanged.  Kernels
// tell the two kinds apart with is_float_sample, never with sizeof: a half is as wide as a uint16_t.
template <typename T>
struct is_float_sample : std::integral_constant<bool, std::is_same<T, float>::value || std::is_same<T, __half>::value> {
};

// clamp to [0, peak] and round half to even (lrintf) in one saturating convert; NaN -> 0
// (8-bit planes always have peak = 255, which the saturating convert already enforces)
__device__ __forceinline__ uint32_t finish_u8(float v, float)
{
    uint32_t r;
    asm("cvt.rni.sat.u8.f32 %0, %1;" : "=r"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ uint32_t finish_u16(float v, float peak)
{
    uint32_t r;
    asm("cvt.rni.sat.u16.f32 %0, %1;" : "=r"(r) : "f"(fminf(v, peak)));
    return r;
}
// full-range 16-bit: saturation is the clamp
__device__ __forceinline__ uint32_t finish_u16_full(float v)
{
    uint32_t r;
    asm("cvt.rni.sat.u16.f32 %0, %1;" : "=r"(r) : "f"(v));
    return r;
}

template <typename T>
__device__ __forceinline__ T finish(float v, float peak);
template <>
__device__ __forceinline__ float finish<float>(float v, float)
{
    return v;
}
template <>
__device__ __forceinline__ uint8_t finish<uint8_t>(float v, float peak)
{
    return (uint8_t)finish_u8(v, peak);
}
template <>
__device__ __forceinline__ uint16_t finish<uint16_t>(float v, float peak)
{
    return (uint16_t)finish_u16(v, peak);
}
// round to nearest even, no clamp: sums of magnitude >= 65520 become +-Inf
template <>
__device__ __forceinline__ __half finish<__half>(float v, float)
{
    return __float2half_rn(v);
}
// two halves in one word, the first in the low 16 bits (the lower address)
__device__ __forceinline__ uint32_t pack_half2(float lo, float hi)
{
    return (uint32_t)__half_as_ushort(__float2half_rn(lo)) | ((uint32_t)__half_as_ushort(__float2half_rn(hi)) << 16);
}
// one half of a word as float (exact, subnormals included)
__device__ __forceinline__ float half_bits_to_float(uint32_t w, int hi)
{
    return __half2float(__ushort_as_half((unsigned short)(hi ? w >> 16 : w & 0xffffu)));
}

// Integer samples become floats without the (quarter-rate) I2F: drop the bits into the mantissa of 2^23 and subtract
// 2^23 again -- exact for any value below 2^23.
template <typename T>
__device__ __forceinline__ float load_sample(const T* p)
{
    return __uint_as_float(0x4B000000u | (uint32_t)__ldg(p)) - 8388608.f;
}
template <>
__device__ __forceinline__ float load_sample<float>(const float* p)
{
    return __ldg(p);
}
template <>
__device__ __forceinline__ float load_sample<__half>(const __half* p)
{
    return __half2float(__ldg(p));
}
template <typename T>
__device__ __forceinline__ float sample_to_float(T v)
{
    return __uint_as_float(0x4B000000u | (uint32_t)v) - 8388608.f;
}
template <>
__device__ __forceinline__ float sample_to_float<float>(float v)
{
    return v;
}
template <>
__device__ __forceinline__ float sample_to_float<__half>(__half v)
{
    return __half2float(v);
}

// four consecutive samples as one aligned vector load
template <typename T>
struct Vec4Of;
template <>
struct Vec4Of<uint8_t> {
    using type = uint32_t;
};
template <>
struct Vec4Of<uint16_t> {
    using type = uint2;
};
template <>
struct Vec4Of<float> {
    using type = float4;
};
template <>
struct Vec4Of<__half> {
    using type = uint2;
};
// sample k (0..3, a constant after unrolling) of such a group as float: integer samples are dropped into the mantissa
// of 2^23 by one byte permute, then 2^23 is subtracted
template <typename T>
__device__ __forceinline__ float vec4_sample(const typename Vec4Of<T>::type& v, int k);
template <>
__device__ __forceinline__ float vec4_sample<uint8_t>(const uint32_t& v, int k)
{
    return __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7440u | (unsigned)k)) - 8388608.f;
}
template <>
__device__ __forceinline__ float vec4_sample<uint16_t>(const uint2& v, int k)
{
    return __uint_as_float(__byte_perm((k & 2) ? v.y : v.x, 0x4B000000u, (k & 1) ? 0x7432u : 0x7410u)) - 8388608.f;
}
template <>
__device__ __forceinline__ float vec4_sample<float>(const float4& v, int k)
{
    return k == 0 ? v.x : k == 1 ? v.y : k == 2 ? v.z : v.w;
}
template <>
__device__ __forceinline__ float vec4_sample<__half>(const uint2& v, int k)
{
    return half_bits_to_float((k & 2) ? v.y : v.x, k & 1);
}

template <typename T>
__device__ __forceinline__ void store8(T* p, const float (&v)[8], float peak);
template <>
__device__ __forceinline__ void store8<float>(float* p, const float (&v)[8], float)
{
    reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
}
template <>
__device__ __forceinline__ void store8<__half>(__half* p, const float (&v)[8], float)
{
    *reinterpret_cast<uint4*>(p) = make_uint4(pack_half2(v[0], v[1]), pack_half2(v[2], v[3]), pack_half2(v[4], v[5]), pack_half2(v[6], v[7]));
}
template <>
__device__ __forceinline__ void store8<uint16_t>(uint16_t* p, const float (&v)[8], float peak)
{
    uint32_t q[4];
    if (peak >= 65535.f) { // uniform: 16-bit clips need no separate upper clamp
#pragma unroll
        for (int k = 0; k < 4; ++k)
            q[k] = finish_u16_full(v[2 * k]) | (finish_u16_full(v[2 * k + 1]) << 16);
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            q[k] = finish_u16(v[2 * k], peak) | (finish_u16(v[2 * k + 1], peak) << 16);
    }
    *reinterpret_cast<uint4*>(p) = make_uint4(q[0], q[1], q[2], q[3]);
}
template <>
__device__ __forceinline__ void store8<uint8_t>(uint8_t* p, const float (&v)[8], float peak)
{
    uint32_t q[2];
#pragma unroll
    for (int k = 0; k < 2; ++k)
        q[k] = finish_u8(v[4 * k], peak) | (finish_u8(v[4 * k + 1], peak) << 8) | (finish_u8(v[4 * k + 2], peak) << 16) |
               (finish_u8(v[4 * k + 3], peak) << 24);
    *reinterpret_cast<uint2*>(p) = make_uint2(q[0], q[1]);
}

// Division of a small block index by a launch constant without the ~20-instruction integer-division sequence:
// floor(n / d) = umulhi(n, ceil(2^32 / d)) as long as n * d < 2^32 (grids here stay far below that).
inline unsigned div_magic(unsigned d) { return d <= 1 ? 0u : (unsigned)((0x100000000ull + d - 1) / d); }
__device__ __forceinline__ unsigned div_by(unsigned n, unsigned magic) { return magic ? __umulhi(n, magic) : n; }

// ------------------------------------------------------------------------------------------ shared argument blocks

struct Rect {
    int x0, y0, x1, y1;
};

// bits per component back from peak = (1 << bits) - 1
inline int t_bits_from_peak(float peak)
{
    int bits = 0;
    while (bits < 32 && (float)((1ll << bits) - 1) < peak)
        ++bits;
    return bits;
}

// planes of ONE frame that share the table being run (device pointers, pitches in elements)
struct PlanePtrs {
    const void* src[JINC_MAX_PLANES];
    void* dst[JINC_MAX_PLANES];
    long long src_pitch[JINC_MAX_PLANES];
    long long dst_pitch[JINC_MAX_PLANES];
};

// strips: up to four rectangles of output samples, each cut into patches of PW x PH outputs; one block per patch
struct StripArgs {
    const int32_t* start_x;
    const int32_t* start_y;
    const int32_t* rank_x;
    const int32_t* rank_y;
    const float* pos_x;
    const float* pos_y;
    const float* weights;
    const float* weights_p; // the phase blocks again with rows padded to 16 bytes [block][fs][fsp], or null (many phases)
    const float* lut;
    const float* border_sum;
    const float* border_w; // resident per-pixel border weights [slot/32][tap][slot%32], or null
    const int32_t* border_block; // slot -> class block, or null
    const float* border_wb;      // [block][fs][fsp] class blocks, fsp = fs rounded up to 4
    BorderGeom bg;
    int fs, n_rank_x, src_w, src_h;
    double step_x, step_y, radius2, idx_scale;
    Rect rect[4];
    unsigned patch_begin[5];   // prefix sums of patches per rect
    unsigned patches_x[4];     // patches per row of patches
    int pw_log2[4];            // log2 of the patch width (patch height = outputs per block / width)
    int row_mode[4];           // 1: a thread's samples lie in one output row (top/bottom strips), 0: in one column
    unsigned blocks_per_plane; // = patch_begin[4]; the grid holds this many strip blocks per plane
    unsigned blocks_per_plane_magic, patches_x_magic[4]; // div_magic of the two divisors above
    unsigned smem_floats;      // shared memory a strip block may use to stage its source footprint (0: none)
    // whole-frame launches of a table with a strip plan (jinc_internal.h: StripPlan), else null: the patches above are
    // then the plan's, and a strip block reads its descriptors instead of deriving them
    const StripPlanPatch* plan_patches;
    const uint4* plan_threads;
    const float* plan_wdata;
    int plan_px, plan_py; // phase period of the outputs: distance of a planned thread's samples
};

// whole-frame launches: the strip blocks of a table with a plan run from it (jinc_resize.cu)
bool attach_strip_plan(const jinc_table* t, StripArgs& st, int threads, int spt);
// the table's arrays and geometry scalars (no strips, no plan); jinc_resize.cu
void fill_strip_args(const jinc_table* t, StripArgs& a);

struct FrameSet {
    PlanePtrs one;           // used when frames == nullptr
    const PlanePtrs* frames; // device array [grid.y] for batched launches
    int n_planes;
    float peak;
};

__device__ __forceinline__ const PlanePtrs& frame_ptrs(const FrameSet& fs)
{
    return fs.frames ? fs.frames[blockIdx.y] : fs.one;
}

// Window rows as aligned 32-bit words (the plane base and pitch are 4-byte aligned), converted later: the words are
// funnel-shifted into place and every integer sample is dropped into the mantissa of 2^23 by one byte permute (a half
// sample is converted as it is).
template <typename T, int FS>
struct RowWords {
    static constexpr int SB = (int)sizeof(T);
    static constexpr int NA = (FS * SB + 3) / 4;      // aligned words that hold the row
    static constexpr int NW = SB == 4 ? FS : NA + 1;  // words loaded (one more when the row starts inside a word)
    // rows whose loads are issued together (the strips are latency-bound: most sample rows miss L2), about 24 registers
    static constexpr int GROUP = (24 / NW) < 1 ? 1 : ((24 / NW) > FS ? FS : (24 / NW));
};

template <typename T, int FS>
__device__ __forceinline__ void load_row_words(const T* __restrict__ s, uint32_t (&w)[RowWords<T, FS>::NW])
{
    using R = RowWords<T, FS>;
    if constexpr (R::SB == 4) {
#pragma unroll
        for (int i = 0; i < FS; ++i)
            w[i] = __ldg(reinterpret_cast<const uint32_t*>(s) + i);
    } else {
        const uintptr_t addr = reinterpret_cast<uintptr_t>(s);
        const uint32_t* __restrict__ p4 = reinterpret_cast<const uint32_t*>(addr & ~(uintptr_t)3);
#pragma unroll
        for (int j = 0; j < R::NA; ++j)
            w[j] = __ldg(p4 + j);
        w[R::NA] = ((unsigned)(addr & 3) + FS * R::SB > 4 * R::NA) ? __ldg(p4 + R::NA) : 0u; // never touch a word the row does not reach
    }
}

template <typename T, int FS>
__device__ __forceinline__ void row_words_to_float(const uint32_t (&w)[RowWords<T, FS>::NW], unsigned off, float (&v)[FS])
{
    using R = RowWords<T, FS>;
    if constexpr (R::SB == 4) {
#pragma unroll
        for (int i = 0; i < FS; ++i)
            v[i] = __uint_as_float(w[i]);
    } else {
        uint32_t al[R::NA];
#pragma unroll
        for (int j = 0; j < R::NA; ++j)
            al[j] = __funnelshift_r(w[j], w[j + 1], off * 8);
#pragma unroll
        for (int i = 0; i < FS; ++i) {
            if constexpr (is_float_sample<T>::value) {
                v[i] = half_bits_to_float(al[i >> 1], i & 1);
            } else {
                uint32_t bits;
                if (R::SB == 1)
                    bits = __byte_perm(al[i >> 2], 0x4B000000u, 0x7440 | (i & 3));
                else
                    bits = __byte_perm(al[i >> 1], 0x4B000000u, (i & 1) ? 0x7432 : 0x7410);
                v[i] = __uint_as_float(bits) - 8388608.f;
            }
        }
    }
}

// sum over an FS x FS window with a weight block whose rows are padded to 16 bytes
template <typename T, int FS>
__device__ __forceinline__ float dot_rows_vec(const T* __restrict__ s, int pitch, const float* __restrict__ w)
{
    using R = RowWords<T, FS>;
    constexpr int FSP = (FS + 3) & ~3;
    const unsigned off = (unsigned)(reinterpret_cast<uintptr_t>(s) & 3); // the pitch keeps it the same on every row
    float acc = 0.f;
#pragma unroll 1
    for (int ly0 = 0; ly0 < FS; ly0 += R::GROUP) {
        uint32_t words[R::GROUP][R::NW];
#pragma unroll
        for (int g = 0; g < R::GROUP; ++g) {
            const int ly = min(ly0 + g, FS - 1); // the last group may be short: re-read the last row, skipped below
            load_row_words<T, FS>(s + (long long)ly * pitch, words[g]);
        }
#pragma unroll
        for (int g = 0; g < R::GROUP; ++g) {
            if (FS % R::GROUP != 0 && ly0 + g >= FS)
                break;
            float wr[FSP], v[FS];
            const float4* __restrict__ w4 = reinterpret_cast<const float4*>(w + (ly0 + g) * FSP);
#pragma unroll
            for (int q = 0; q < FSP / 4; ++q) {
                const float4 t = __ldg(w4 + q);
                wr[4 * q] = t.x;
                wr[4 * q + 1] = t.y;
                wr[4 * q + 2] = t.z;
                wr[4 * q + 3] = t.w;
            }
            row_words_to_float<T, FS>(words[g], off, v);
#pragma unroll
            for (int lx = 0; lx < FS; ++lx)
                acc = fmaf(v[lx], wr[lx], acc);
        }
    }
    return acc;
}

constexpr int STRIP_THREADS = 256;

// One output sample of a strip for ONE plane, read straight from global memory.  Lean on purpose: 32-bit indexing,
// constant weight strides.  FSC > 0 fixes the window size at compile time (inner loops unroll).
template <typename T, int FSC>
__device__ __forceinline__ void strip_sample(const StripArgs& a, const FrameSet& fsx, int x, int y, int plane)
{
    const PlanePtrs& pp = frame_ptrs(fsx);
    const int fs = FSC > 0 ? FSC : a.fs;
    const int sx = a.start_x[x], sy = a.start_y[y];
    const int rx = a.rank_x[x], ry = a.rank_y[y];
    const int pitch = (int)pp.src_pitch[plane];
    const T* __restrict__ s = static_cast<const T*>(pp.src[plane]) + (long long)sy * pitch + sx;
    float acc = 0.f;

    const bool shared_block = rx >= 0 && ry >= 0;
    if (!shared_block && a.border_block) {
        // the block of this border pixel's class, rows padded to 16 bytes
        const int fsp = (fs + 3) & ~3;
        const float* __restrict__ w = a.border_wb + (size_t)a.border_block[jinc_border_slot(a.bg, x, y)] * (unsigned)(fs * fsp);
        if (FSC > 0 && ((reinterpret_cast<uintptr_t>(pp.src[plane]) | (uintptr_t)(pitch * (int)sizeof(T))) & 3) == 0) {
            acc = dot_rows_vec<T, (FSC > 0 ? FSC : 4)>(s, pitch, w);
        } else {
            for (int ly = 0; ly < fs; ++ly) {
#pragma unroll
                for (int lx = 0; lx < (FSC > 0 ? FSC : fs); ++lx)
                    acc = fmaf(load_sample(s + lx), __ldg(w + lx), acc);
                w += fsp;
                s += pitch;
            }
        }
    } else if (shared_block) {
        // shared phase block (:431-435), row-major fs x fs
        const float* __restrict__ w = a.weights + (unsigned)(ry * a.n_rank_x + rx) * (unsigned)(fs * fs);
        for (int ly = 0; ly < fs; ++ly) {
#pragma unroll
            for (int lx = 0; lx < (FSC > 0 ? FSC : fs); ++lx)
                acc = fmaf(load_sample(s + lx), __ldg(w + lx), acc);
            w += fs;
            s += pitch;
        }
    } else if (a.border_w) {
        // this border pixel's own resident block (:443-514), stored [slot / 32][tap][slot % 32]: neighbouring pixels
        // coalesce and the tap stride is the constant 32
        const long long slot = jinc_border_slot(a.bg, x, y);
        const float* __restrict__ w = a.border_w + (size_t)(slot >> 5) * (size_t)(fs * fs * 32) + (unsigned)(slot & 31);
        for (int ly = 0; ly < fs; ++ly) {
#pragma unroll
            for (int lx = 0; lx < (FSC > 0 ? FSC : fs); ++lx)
                acc = fmaf(load_sample(s + lx), __ldg(w + lx * 32), acc);
            w += fs * 32;
            s += pitch;
        }
    } else {
        // border weights did not fit the residency budget: rebuild them per sample from the UNquantised position
        // (:443-514), exact LUT index per tap, factor / divider
        const float px = a.pos_x[x], py = a.pos_y[y];
        const float sum = a.border_sum[jinc_border_slot(a.bg, x, y)];
        for (int ly = 0; ly < fs; ++ly) {
            const double dy2 = jinc_tap_dist2(py, a.src_h, sy + ly, a.step_y);
            for (int lx = 0; lx < fs; ++lx) {
                const double dx2 = jinc_tap_dist2(px, a.src_w, sx + lx, a.step_x);
                const float f = jinc_lut_weight(a.lut, __dadd_rn(dx2, dy2), a.radius2, a.idx_scale);
                acc = fmaf(load_sample(s + lx), __fdiv_rn(f, sum), acc);
            }
            s += pitch;
        }
    }
    static_cast<T*>(pp.dst[plane])[(long long)y * pp.dst_pitch[plane] + x] = finish<T>(acc, fsx.peak);
}

// What a strip sample needs besides its source window: gathered for all of a thread's samples before any is used, so
// the table loads of the SPT samples are in flight together.
struct StripMeta {
    int x, y;       // output sample (x < 0: none)
    int sx, sy;     // window origin
    const float* w; // weight block: [fs][wstride]
    int wstride;    // fs for a shared phase block, fs rounded up to 4 for a border class block; 0 = neither (slow kinds)
};

// 32-bit form of jinc_border_slot for the kernels (the table build rejects geometries with 2^31 or more border pixels)
__device__ __forceinline__ int border_slot32(const BorderGeom& g, int x, int y)
{
    if (y < g.by0)
        return y * g.W + x;
    if (y >= g.by1)
        return (int)g.off_bottom + (y - g.by1) * g.W + x;
    if (x < g.bx0)
        return (int)g.off_left + (y - g.by0) * g.bx0 + x;
    return (int)g.off_right + (y - g.by0) * (g.W - g.bx1) + (x - g.bx1);
}

template <int FSC>
__device__ __forceinline__ StripMeta strip_meta(const StripArgs& a, int x, int y)
{
    const int fs = FSC > 0 ? FSC : a.fs;
    const int fsp = (fs + 3) & ~3;
    StripMeta m;
    m.x = x;
    m.y = y;
    m.sx = a.start_x[x];
    m.sy = a.start_y[y];
    const bool border = x < a.bg.bx0 || x >= a.bg.bx1 || y < a.bg.by0 || y >= a.bg.by1; // no table load needed to know
    if (!border) {
        const unsigned blk = (unsigned)(a.rank_y[y] * a.n_rank_x + a.rank_x[x]);
        if (a.weights_p) {
            m.w = a.weights_p + blk * (unsigned)(fs * fsp);
            m.wstride = fsp;
        } else {
            m.w = a.weights + blk * (unsigned)(fs * fs);
            m.wstride = fs;
        }
    } else if (a.border_block) {
        m.w = a.border_wb + (unsigned)a.border_block[border_slot32(a.bg, x, y)] * (unsigned)(fs * fsp);
        m.wstride = fsp;
    } else {
        m.w = nullptr;
        m.wstride = 0;
    }
    return m;
}

// One sample from a staged footprint: `tile` holds the source rectangle [sy_lo, ..) x [sx_lo, sx_lo + fw) as floats.
template <typename T, int FSC>
__device__ __forceinline__ void strip_sample_staged(const StripArgs& a, const FrameSet& fsx, const StripMeta& m, int plane,
                                                    const float* __restrict__ tile, int fw, int sx_lo, int sy_lo)
{
    const int fs = FSC > 0 ? FSC : a.fs;
    const float* __restrict__ s = tile + (m.sy - sy_lo) * fw + (m.sx - sx_lo);
    float acc = 0.f;
    if ((m.wstride & 3) != 0) { // unpadded rows (the general path's phase blocks)
        const float* __restrict__ w = m.w;
        for (int ly = 0; ly < fs; ++ly) {
#pragma unroll
            for (int lx = 0; lx < (FSC > 0 ? FSC : fs); ++lx)
                acc = fmaf(s[lx], __ldg(w + lx), acc);
            w += fs;
            s += fw;
        }
    } else {
        const float4* __restrict__ w4 = reinterpret_cast<const float4*>(m.w); // rows padded to 16 bytes
        for (int ly = 0; ly < fs; ++ly) {
#pragma unroll
            for (int q = 0; q < (FSC > 0 ? (FSC + 3) / 4 : m.wstride / 4); ++q) {
                const float4 t = __ldg(w4 + q);
                const int lx = 4 * q;
                acc = fmaf(s[lx], t.x, acc);
                if (lx + 1 < fs)
                    acc = fmaf(s[lx + 1], t.y, acc);
                if (lx + 2 < fs)
                    acc = fmaf(s[lx + 2], t.z, acc);
                if (lx + 3 < fs)
                    acc = fmaf(s[lx + 3], t.w, acc);
            }
            w4 += m.wstride / 4;
            s += fw;
        }
    }
    const PlanePtrs& pp = frame_ptrs(fsx);
    static_cast<T*>(pp.dst[plane])[(long long)m.y * pp.dst_pitch[plane] + m.x] = finish<T>(acc, fsx.peak);
}

// The SPT samples of one thread, interleaved (SPT independent accumulator chains).  SHARED: they share ONE weight block
// (the usual case in the strips of the periodic geometries: a thread's samples lie in the same border row or column, a
// multiple of the phase period apart), so every weight vector is loaded once; otherwise each sample reads its own
// block (general ratios).  All blocks have rows padded to 16 bytes and the same row stride.
template <typename T, int FSC, int SPT, bool SHARED>
__device__ __forceinline__ void strip_samples_fused(const StripArgs& a, const FrameSet& fsx, const StripMeta (&m)[SPT], unsigned live,
                                                    int plane, const float* __restrict__ tile, int fw, int sx_lo, int sy_lo)
{
    const int fs = FSC > 0 ? FSC : a.fs;
    constexpr int NW = SHARED ? 1 : SPT;
    const float* __restrict__ s[SPT];
    const float4* __restrict__ w4[NW];
    float acc[SPT];
#pragma unroll
    for (int k = 0; k < SPT; ++k) {
        s[k] = tile + (m[k].sy - sy_lo) * fw + (m[k].sx - sx_lo);
        acc[k] = 0.f;
    }
#pragma unroll
    for (int k = 0; k < NW; ++k)
        w4[k] = reinterpret_cast<const float4*>(m[k].w); // rows padded to 16 bytes
    const int wq = m[0].wstride / 4;
    for (int ly = 0; ly < fs; ++ly) {
#pragma unroll
        for (int q = 0; q < (FSC > 0 ? (FSC + 3) / 4 : wq); ++q) {
            float4 t[NW];
#pragma unroll
            for (int k = 0; k < NW; ++k)
                t[k] = __ldg(w4[k] + q);
            const int lx = 4 * q;
#pragma unroll
            for (int k = 0; k < SPT; ++k) {
                const float4& tk = t[SHARED ? 0 : k];
                acc[k] = fmaf(s[k][lx], tk.x, acc[k]);
                if (lx + 1 < fs)
                    acc[k] = fmaf(s[k][lx + 1], tk.y, acc[k]);
                if (lx + 2 < fs)
                    acc[k] = fmaf(s[k][lx + 2], tk.z, acc[k]);
                if (lx + 3 < fs)
                    acc[k] = fmaf(s[k][lx + 3], tk.w, acc[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < NW; ++k)
            w4[k] += wq;
#pragma unroll
        for (int k = 0; k < SPT; ++k)
            s[k] += fw;
    }
    const PlanePtrs& pp = frame_ptrs(fsx);
    T* __restrict__ dst = static_cast<T*>(pp.dst[plane]);
    const long long dp = pp.dst_pitch[plane];
#pragma unroll
    for (int k = 0; k < SPT; ++k)
        if (live & (1u << k))
            dst[(long long)m[k].y * dp + m[k].x] = finish<T>(acc[k], fsx.peak);
}

// SPT same-block samples whose windows OVERLAP: adjacent same-phase outputs of one row, window origins STEP apart
// (the strips of the exact-2x geometry: outputs x, x+2, x+4, x+6 read columns sx, sx+1, sx+2, sx+3).  A window row of
// FSC + (SPT-1)*STEP staged values is read once and feeds SPT x FSC FMAs; the weight row is read once as vectors.
template <typename T, int FSC, int SPT, int STEP>
__device__ __forceinline__ void strip_run_rows(const FrameSet& fsx, const StripMeta (&m)[SPT], int plane, const float* __restrict__ tile,
                                               int fw, int sx_lo, int sy_lo)
{
    constexpr int FSP = (FSC + 3) & ~3, SEG = FSC + (SPT - 1) * STEP;
    const float* __restrict__ s = tile + (m[0].sy - sy_lo) * fw + (m[0].sx - sx_lo);
    const float4* __restrict__ w4 = reinterpret_cast<const float4*>(m[0].w);
    float acc[SPT];
#pragma unroll
    for (int k = 0; k < SPT; ++k)
        acc[k] = 0.f;
#pragma unroll 1
    for (int ly = 0; ly < FSC; ++ly, s += fw, w4 += FSP / 4) {
        float seg[SEG], wr[FSP];
#pragma unroll
        for (int q = 0; q < FSP / 4; ++q) {
            const float4 t = __ldg(w4 + q);
            wr[4 * q] = t.x;
            wr[4 * q + 1] = t.y;
            wr[4 * q + 2] = t.z;
            wr[4 * q + 3] = t.w;
        }
#pragma unroll
        for (int i = 0; i < SEG; ++i)
            seg[i] = s[i];
#pragma unroll
        for (int lx = 0; lx < FSC; ++lx)
#pragma unroll
            for (int k = 0; k < SPT; ++k)
                acc[k] = fmaf(seg[lx + k * STEP], wr[lx], acc[k]);
    }
    const PlanePtrs& pp = frame_ptrs(fsx);
    T* __restrict__ dst = static_cast<T*>(pp.dst[plane]) + (long long)m[0].y * pp.dst_pitch[plane];
#pragma unroll
    for (int k = 0; k < SPT; ++k)
        dst[m[k].x] = finish<T>(acc[k], fsx.peak);
}

// The same for adjacent same-phase outputs of one COLUMN (window origins one row apart): a staged window row of FSC
// values feeds up to SPT outputs, each with its own weight row; a sliding window of SPT weight rows lives in registers.
template <typename T, int FSC, int SPT>
__device__ __forceinline__ void strip_run_cols(const FrameSet& fsx, const StripMeta (&m)[SPT], int plane, const float* __restrict__ tile,
                                               int fw, int sx_lo, int sy_lo)
{
    static_assert(SPT == 4, "the weight-row window is indexed modulo 4");
    constexpr int FSP = (FSC + 3) & ~3;
    const float* __restrict__ s = tile + (m[0].sy - sy_lo) * fw + (m[0].sx - sx_lo);
    const float4* __restrict__ w4 = reinterpret_cast<const float4*>(m[0].w);
    float acc[SPT], wwin[4][FSP];
#pragma unroll
    for (int k = 0; k < SPT; ++k)
        acc[k] = 0.f;
#pragma unroll
    for (int r = 0; r < FSC + SPT - 1; ++r, s += fw) { // r: source row below the first output's window origin
        float seg[FSC];
#pragma unroll
        for (int i = 0; i < FSC; ++i)
            seg[i] = s[i];
        if (r < FSC) {
#pragma unroll
            for (int q = 0; q < FSP / 4; ++q) {
                const float4 t = __ldg(w4 + r * (FSP / 4) + q);
                wwin[r & 3][4 * q] = t.x;
                wwin[r & 3][4 * q + 1] = t.y;
                wwin[r & 3][4 * q + 2] = t.z;
                wwin[r & 3][4 * q + 3] = t.w;
            }
        }
#pragma unroll
        for (int k = 0; k < SPT; ++k) {
            const int ly = r - k; // weight row of output k (a constant after unrolling)
            if (ly >= 0 && ly < FSC) {
#pragma unroll
                for (int lx = 0; lx < FSC; ++lx)
                    acc[k] = fmaf(seg[lx], wwin[ly & 3][lx], acc[k]);
            }
        }
    }
    const PlanePtrs& pp = frame_ptrs(fsx);
    T* __restrict__ dst = static_cast<T*>(pp.dst[plane]);
    const long long dp = pp.dst_pitch[plane];
#pragma unroll
    for (int k = 0; k < SPT; ++k)
        dst[(long long)m[k].y * dp + m[k].x] = finish<T>(acc[k], fsx.peak);
}

// Strip block `sb` of the grid (planes are the slow dimension): one patch of PW x PH outputs, SPT per thread.  The
// source rectangle the patch reads (window origins are monotonic along both axes) is staged into shared memory as
// floats when it fits, so the global loads are coalesced, converted once and every window row is read from shared
// memory; otherwise every sample reads global memory directly.  A thread's SPT samples lie in one output row (wide
// strips) or one output column (narrow strips), a multiple of the phase period apart, so they normally share one weight
// block and run fused.  PERIOD > 0 (the exact-2x kernel: 2) makes them ADJACENT same-phase outputs (x, x + PERIOD, ...),
// whose window origins are STEP apart: their windows overlap, and strip_run_rows / strip_run_cols read every staged
// value once for all of them.
template <typename T, int FSC, int THREADS = STRIP_THREADS, int SPT = 1, int PERIOD = 0, int STEP = 0>
__device__ __forceinline__ void strip_block(const StripArgs& a, const FrameSet& fsx, unsigned sb, float* __restrict__ tile)
{
    static_assert((SPT & (SPT - 1)) == 0 && (THREADS & (THREADS - 1)) == 0, "powers of two");
    constexpr int SPT_L2 = SPT == 1 ? 0 : SPT == 2 ? 1 : SPT == 4 ? 2 : 3;
    const int fs = FSC > 0 ? FSC : a.fs;
    const unsigned plane = div_by(sb, a.blocks_per_plane_magic);
    const unsigned pid = sb - plane * a.blocks_per_plane;
    const int r = (int)(pid >= a.patch_begin[1]) + (int)(pid >= a.patch_begin[2]) + (int)(pid >= a.patch_begin[3]);
    const unsigned lp = pid - a.patch_begin[r];
    const unsigned pyi = div_by(lp, a.patches_x_magic[r]), pxi = lp - pyi * a.patches_x[r];
    const int pwl = a.pw_log2[r];
    const int ox0 = a.rect[r].x0 + (int)(pxi << pwl), oy0 = a.rect[r].y0 + (int)pyi * ((THREADS * SPT) >> pwl);
    const int nx = min(1 << pwl, a.rect[r].x1 - ox0), ny = min((THREADS * SPT) >> pwl, a.rect[r].y1 - oy0);

    // footprint corners and the tables of this thread's samples: one round of loads
    const int sx_lo = a.start_x[ox0], sy_lo = a.start_y[oy0];
    const int fw = a.start_x[ox0 + nx - 1] + fs - sx_lo, fh = a.start_y[oy0 + ny - 1] + fs - sy_lo;
    StripMeta meta[SPT];
    unsigned live = 0;
    const bool rows = a.row_mode[r] != 0;
    {
        // sample k of thread t: row mode (x, y) = (tx + k * dx, ty), column mode (tx, ty + k * dy), with dx = PW/SPT
        // (dy = PH/SPT) -- or, with PERIOD, the thread's samples PERIOD apart inside a group of SPT * PERIOD outputs.  The
        // live samples of a thread are a prefix (coordinates grow with k).  The axis tables are read once per distinct
        // coordinate: SPT + 1 positions instead of 2 SPT.
        const int txl = rows ? pwl - SPT_L2 : pwl; // log2 of the threads per patch row
        int tx = (int)threadIdx.x & ((1 << txl) - 1), ty = (int)threadIdx.x >> txl;
        int dx = rows ? 1 << txl : 0, dy = rows ? 0 : THREADS >> pwl;
        if (PERIOD > 0) {
            if (rows) {
                tx = (tx / PERIOD) * (SPT * PERIOD) + tx % PERIOD;
                dx = PERIOD;
            } else {
                ty = (ty / PERIOD) * (SPT * PERIOD) + ty % PERIOD;
                dy = PERIOD;
            }
        }
        const int fsp = (fs + 3) & ~3;
        int sxv[SPT], rxv[SPT], syv[SPT], ryv[SPT];
#pragma unroll
        for (int k = 0; k < SPT; ++k) {
            const int lx = tx + k * dx, ly = ty + k * dy;
            if (lx < nx && ly < ny) {
                live |= 1u << k;
                if (k == 0 || rows) {
                    sxv[k] = a.start_x[ox0 + lx];
                    rxv[k] = a.rank_x[ox0 + lx];
                } else {
                    sxv[k] = sxv[0];
                    rxv[k] = rxv[0];
                }
                if (k == 0 || !rows) {
                    syv[k] = a.start_y[oy0 + ly];
                    ryv[k] = a.rank_y[oy0 + ly];
                } else {
                    syv[k] = syv[0];
                    ryv[k] = ryv[0];
                }
            }
        }
#pragma unroll
        for (int k = 0; k < SPT; ++k) {
            if (!(live & (1u << k)))
                continue;
            StripMeta& m = meta[k];
            m.x = ox0 + tx + k * dx;
            m.y = oy0 + ty + k * dy;
            m.sx = sxv[k];
            m.sy = syv[k];
            if (rxv[k] >= 0 && ryv[k] >= 0) { // rank is -1 exactly on border coordinates
                const unsigned blk = (unsigned)(ryv[k] * a.n_rank_x + rxv[k]);
                m.w = a.weights_p ? a.weights_p + blk * (unsigned)(fs * fsp) : a.weights + blk * (unsigned)(fs * fs);
                m.wstride = a.weights_p ? fsp : fs;
            } else if (a.border_block) {
                m.w = a.border_wb + (unsigned)a.border_block[border_slot32(a.bg, m.x, m.y)] * (unsigned)(fs * fsp);
                m.wstride = fsp;
            } else {
                m.w = nullptr;
                m.wstride = 0;
            }
        }
    }
    const unsigned n = (unsigned)(fw * fh);
    const bool staged = tile != nullptr && n <= a.smem_floats; // the same for the whole block
    if (staged) {
        const PlanePtrs& pp = frame_ptrs(fsx);
        const int pitch = (int)pp.src_pitch[plane];
        const T* __restrict__ src = static_cast<const T*>(pp.src[plane]) + (long long)sy_lo * pitch + sx_lo;
        const unsigned magic = 0xFFFFFFFFu / (unsigned)fw + 1u; // floor(e / fw) = umulhi(e, magic) while e * fw < 2^32
        for (unsigned e0 = threadIdx.x; e0 < n; e0 += 4 * THREADS) {
            T v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) { // all four loads are issued before the first conversion
                const unsigned e = min(e0 + u * THREADS, n - 1);
                const unsigned row = __umulhi(e, magic);
                v[u] = __ldg(src + (int)(row * (unsigned)pitch + (e - row * (unsigned)fw)));
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (e0 + u * THREADS < n)
                    tile[e0 + u * THREADS] = sample_to_float(v[u]);
        }
        __syncthreads();
    }
    if (!(live & 1u))
        return; // live samples are a prefix
    if (SPT > 1 && staged) {
        // samples outside the rectangle repeat sample 0 (computed, not stored), so a partly live thread stays fused
        bool same = true, vec = true;
#pragma unroll
        for (int k = 0; k < SPT; ++k) {
            if (!(live & (1u << k)))
                meta[k] = meta[0];
            same = same && meta[k].w == meta[0].w;
            vec = vec && meta[k].wstride != 0 && (meta[k].wstride & 3) == 0 && meta[k].wstride == meta[0].wstride;
        }
        if (PERIOD > 0 && FSC > 0 && vec && same && live == (1u << SPT) - 1u) {
            // adjacent same-phase samples with regularly advancing origins: overlapping windows, every value read once
            bool run = true;
#pragma unroll
            for (int k = 1; k < SPT; ++k)
                run = run && (rows ? (meta[k].sy == meta[0].sy && meta[k].sx == meta[0].sx + k * STEP)
                                   : (meta[k].sx == meta[0].sx && meta[k].sy == meta[0].sy + k * STEP));
            if (run && rows) {
                strip_run_rows<T, (FSC > 0 ? FSC : 4), SPT, (STEP > 0 ? STEP : 1)>(fsx, meta, (int)plane, tile, fw, sx_lo, sy_lo);
                return;
            }
            if (run && STEP == 1 && SPT == 4 && FSC <= 9) { // the weight-row window of larger windows does not fit the registers
                strip_run_cols<T, (FSC > 0 && FSC <= 9 ? FSC : 4), 4>(fsx, reinterpret_cast<const StripMeta(&)[4]>(meta), (int)plane, tile, fw,
                                                                      sx_lo, sy_lo);
                return;
            }
        }
        if (vec) {
            if (same)
                strip_samples_fused<T, FSC, SPT, true>(a, fsx, meta, live, (int)plane, tile, fw, sx_lo, sy_lo);
            else
                strip_samples_fused<T, FSC, SPT, false>(a, fsx, meta, live, (int)plane, tile, fw, sx_lo, sy_lo);
            return;
        }
    }
#pragma unroll
    for (int k = 0; k < SPT; ++k) {
        if (!(live & (1u << k)))
            continue;
        if (staged && meta[k].wstride)
            strip_sample_staged<T, FSC>(a, fsx, meta[k], (int)plane, tile, fw, sx_lo, sy_lo);
        else
            strip_sample<T, FSC>(a, fsx, meta[k].x, meta[k].y, (int)plane);
    }
}

// ------------------------------------------------------------------------------------------ planned strip blocks
//
// Whole-frame launches of a table with a StripPlan (jinc_internal.h) run their strip blocks from it.  The plan cuts the
// border strips into its own patches and gives every thread up to SPT samples of ONE border row (wide strips) or column
// (tall strips) that are a phase period apart -- adjacent outputs of the same phase, so they normally share one weight
// block and their windows overlap.  A patch descriptor holds the source footprint, one 16-byte record per thread and
// sample holds the output coordinates, the window's offset in the staged footprint, the weight block and how the
// thread's samples are accumulated.  The distinct weight blocks of a patch (a handful: one per border row or column and
// phase) are packed next to each other by the table build and copied into shared memory with the footprint, so the
// accumulation loops read nothing from global memory (patches with too many blocks for that -- corners of wide windows --
// read the packed copy).  Every sample is accumulated in the same tap order as in strip_block (row-major, one fused
// multiply-add per tap): both paths give identical bits.

// De-interleaved footprint of a patch of row runs: the lanes of a warp are spt * step columns apart, so column c sits at
// (c % (spt * step)) * sub + c / (spt * step): the same element of consecutive lanes in consecutive words.  `sub` covers
// the widest patch (64 outputs) and is odd, which puts the two patch rows of a warp on different banks.
__host__ __device__ constexpr int plan_deint_sub(int step, int spt, int fs)
{
    return ((64 * step + fs + step + spt * step - 1) / (spt * step)) | 1;
}

template <bool WS>
__device__ __forceinline__ float4 plan_w4(const float* __restrict__ w)
{
    if (WS)
        return *reinterpret_cast<const float4*>(w); // shared memory
    return __ldg(reinterpret_cast<const float4*>(w));
}

// weight block of a record of a patch whose blocks are not staged: straight from the table (sel << 31 | block)
template <int FSC>
__device__ __forceinline__ const float* plan_block(const StripArgs& a, uint32_t z)
{
    constexpr int WBF = FSC * ((FSC + 3) & ~3);
    const float* __restrict__ base = (z >> 31) ? a.border_wb : (a.weights_p ? a.weights_p : a.weights);
    return base + (size_t)(z & 0x7fffffffu) * WBF;
}

template <bool WS, int FSP>
__device__ __forceinline__ void plan_weight_row(const float* __restrict__ w, float (&wr)[FSP])
{
#pragma unroll
    for (int q = 0; q < FSP / 4; ++q) {
        const float4 t = plan_w4<WS>(w + 4 * q);
        wr[4 * q] = t.x;
        wr[4 * q + 1] = t.y;
        wr[4 * q + 2] = t.z;
        wr[4 * q + 3] = t.w;
    }
}

// SPT same-block samples of one row whose window origins are STEP apart: a window row of FSC + (SPT-1)*STEP staged
// values is read once and feeds SPT x FSC FMAs.  DEINT: the footprint is staged de-interleaved (plan_deint_sub) and the
// thread's window starts on a multiple of SPT * STEP: every shared-memory offset is an immediate.
template <typename T, int FSC, int SPT, int STEP, bool WS, bool DEINT>
__device__ __forceinline__ void plan_run_rows(const float* __restrict__ s, int rs, const float* __restrict__ w, T* __restrict__ o, int xstep, float peak)
{
    constexpr int FSP = (FSC + 3) & ~3, SEG = FSC + (SPT - 1) * STEP, D = SPT * STEP, SUBC = plan_deint_sub(STEP, SPT, FSC);
    float acc[SPT];
#pragma unroll
    for (int k = 0; k < SPT; ++k)
        acc[k] = 0.f;
    if constexpr (FSC > 9 && !WS) {
        // wide windows, weights from global memory: the next weight row is in flight while this one is applied
        float4 wn[FSP / 4];
#pragma unroll
        for (int q = 0; q < FSP / 4; ++q)
            wn[q] = plan_w4<false>(w + 4 * q);
#pragma unroll 1
        for (int ly = 0; ly < FSC; ++ly) {
            float seg[SEG], wr[FSP];
#pragma unroll
            for (int q = 0; q < FSP / 4; ++q) {
                wr[4 * q] = wn[q].x;
                wr[4 * q + 1] = wn[q].y;
                wr[4 * q + 2] = wn[q].z;
                wr[4 * q + 3] = wn[q].w;
            }
            const float* __restrict__ wnext = w + min(ly + 1, FSC - 1) * FSP;
#pragma unroll
            for (int q = 0; q < FSP / 4; ++q)
                wn[q] = plan_w4<false>(wnext + 4 * q);
            const float* __restrict__ srow = s + ly * (DEINT ? D * SUBC : rs);
#pragma unroll
            for (int i = 0; i < SEG; ++i)
                seg[i] = DEINT ? srow[(i % D) * SUBC + i / D] : srow[i];
#pragma unroll
            for (int lx = 0; lx < FSC; ++lx)
#pragma unroll
                for (int k = 0; k < SPT; ++k)
                    acc[k] = fmaf(seg[lx + k * STEP], wr[lx], acc[k]);
        }
    } else {
#pragma unroll(FSC <= 9 ? FSC : 1)
        for (int ly = 0; ly < FSC; ++ly) {
            float seg[SEG], wr[FSP];
            plan_weight_row<WS, FSP>(w + ly * FSP, wr);
            const float* __restrict__ srow = s + ly * (DEINT ? D * SUBC : rs);
#pragma unroll
            for (int i = 0; i < SEG; ++i)
                seg[i] = DEINT ? srow[(i % D) * SUBC + i / D] : srow[i];
#pragma unroll
            for (int lx = 0; lx < FSC; ++lx)
#pragma unroll
                for (int k = 0; k < SPT; ++k)
                    acc[k] = fmaf(seg[lx + k * STEP], wr[lx], acc[k]);
        }
    }
#pragma unroll
    for (int k = 0; k < SPT; ++k)
        o[k * xstep] = finish<T>(acc[k], peak);
}

__device__ __forceinline__ void cp_async16(uint32_t smem_dst, const void* gsrc)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait()
{
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// plan_run_rows for wide windows whose weight block stays in the table (global memory): the sixteen threads of a half-warp
// share the block (the plan guarantees it), so its rows are streamed through a ring of JINC_PLAN_RING_DEPTH rows in shared
// memory with cp.async, DEPTH - 1 rows in flight -- the L2 round trip of a weight row is hidden behind several rows of
// FMAs instead of one -- and read back as broadcast LDS.128.  Same taps in the same order as plan_run_rows.
template <typename T, int FSC, int SPT, int STEP, bool DEINT>
__device__ __forceinline__ void plan_run_rows_ring(const float* __restrict__ s, int rs, const float* __restrict__ w, float* __restrict__ ring,
                                                   T* __restrict__ o, int xstep, float peak)
{
    constexpr int FSP = (FSC + 3) & ~3, NV = FSP / 4, SEG = FSC + (SPT - 1) * STEP, D = SPT * STEP, SUBC = plan_deint_sub(STEP, SPT, FSC);
    constexpr int DEPTH = JINC_PLAN_RING_DEPTH;
    static_assert(NV <= 16 && (DEPTH & (DEPTH - 1)) == 0, "one 16-byte copy per thread of the half-warp and row");
    const int j = threadIdx.x & 15;
    const uint32_t ring_s = (uint32_t)__cvta_generic_to_shared(ring);
    float acc[SPT];
#pragma unroll
    for (int k = 0; k < SPT; ++k)
        acc[k] = 0.f;
#pragma unroll
    for (int d = 0; d < DEPTH - 1; ++d) {
        if (d < FSC && j < NV)
            cp_async16(ring_s + (uint32_t)((d * FSP + 4 * j) * (int)sizeof(float)), w + d * FSP + 4 * j);
        cp_async_commit();
    }
#pragma unroll 1
    for (int ly = 0; ly < FSC; ++ly) {
        const int ahead = ly + DEPTH - 1;
        if (ahead < FSC && j < NV)
            cp_async16(ring_s + (uint32_t)((((ahead & (DEPTH - 1)) * FSP) + 4 * j) * (int)sizeof(float)), w + ahead * FSP + 4 * j);
        cp_async_commit();
        cp_async_wait<DEPTH - 1>(); // row ly has landed (this thread's part; the warp barrier publishes the others')
        __syncwarp();
        float seg[SEG], wr[FSP];
        plan_weight_row<true, FSP>(ring + (ly & (DEPTH - 1)) * FSP, wr);
        const float* __restrict__ srow = s + ly * (DEINT ? D * SUBC : rs);
#pragma unroll
        for (int i = 0; i < SEG; ++i)
            seg[i] = DEINT ? srow[(i % D) * SUBC + i / D] : srow[i];
#pragma unroll
        for (int lx = 0; lx < FSC; ++lx)
#pragma unroll
            for (int k = 0; k < SPT; ++k)
                acc[k] = fmaf(seg[lx + k * STEP], wr[lx], acc[k]);
        __syncwarp(); // the slot of row ly is overwritten by the next iteration's copy
    }
#pragma unroll
    for (int k = 0; k < SPT; ++k)
        o[k * xstep] = finish<T>(acc[k], peak);
}

// the same down one column (window origins STEP rows apart): a staged row of FSC values feeds up to SPT outputs, each
// with its own weight row
template <typename T, int FSC, int SPT, int STEP, bool WS>
__device__ __forceinline__ void plan_run_cols(const float* __restrict__ s, int fw, const float* __restrict__ w, T* __restrict__ o, long long ystep,
                                              float peak)
{
    constexpr int FSP = (FSC + 3) & ~3;
    float acc[SPT];
#pragma unroll
    for (int k = 0; k < SPT; ++k)
        acc[k] = 0.f;
    static_assert(FSC <= 9, "wide windows do not run down a column: one weight row for four source rows reads less (the planner agrees)");
#pragma unroll
    for (int r = 0; r < FSC + (SPT - 1) * STEP; ++r) {
        float seg[FSC];
#pragma unroll
        for (int i = 0; i < FSC; ++i)
            seg[i] = s[r * fw + i];
#pragma unroll
        for (int k = 0; k < SPT; ++k) {
            const int ly = r - k * STEP; // weight row of output k (a constant after unrolling)
            if (ly >= 0 && ly < FSC) {
                float wr[FSP];
                plan_weight_row<WS, FSP>(w + ly * FSP, wr);
#pragma unroll
                for (int lx = 0; lx < FSC; ++lx)
                    acc[k] = fmaf(seg[lx], wr[lx], acc[k]);
            }
        }
    }
#pragma unroll
    for (int k = 0; k < SPT; ++k)
        o[k * ystep] = finish<T>(acc[k], peak);
}

// SPT samples with separate windows, interleaved; SHARED: one weight block for all of them
template <typename T, int FSC, int SPT, bool SHARED, bool WS>
__device__ __forceinline__ void plan_fused(const StripArgs& a, const uint4 (&r)[SPT], unsigned live, const float* __restrict__ tile, int fw,
                                           const float* __restrict__ wbase, T* __restrict__ dst, long long dp, float peak)
{
    constexpr int FSP = (FSC + 3) & ~3, NW = SHARED ? 1 : SPT;
    const float* __restrict__ s[SPT];
    const float* __restrict__ w[NW];
    float acc[SPT];
#pragma unroll
    for (int k = 0; k < SPT; ++k) {
        s[k] = tile + (int)r[k].y;
        acc[k] = 0.f;
    }
#pragma unroll
    for (int k = 0; k < NW; ++k)
        w[k] = WS ? wbase + r[k].z : plan_block<FSC>(a, r[k].z);
    if constexpr (SHARED && FSC > 9 && !WS) {
        // wide windows, one block read from global memory: the next weight row is in flight while this one is applied
        float4 wn[FSP / 4];
#pragma unroll
        for (int q = 0; q < FSP / 4; ++q)
            wn[q] = plan_w4<false>(w[0] + 4 * q);
#pragma unroll 1
        for (int ly = 0; ly < FSC; ++ly) {
            float4 wc[FSP / 4];
#pragma unroll
            for (int q = 0; q < FSP / 4; ++q)
                wc[q] = wn[q];
            const float* __restrict__ wnext = w[0] + min(ly + 1, FSC - 1) * FSP;
#pragma unroll
            for (int q = 0; q < FSP / 4; ++q)
                wn[q] = plan_w4<false>(wnext + 4 * q);
#pragma unroll
            for (int q = 0; q < FSP / 4; ++q) {
                const int lx = 4 * q;
#pragma unroll
                for (int k = 0; k < SPT; ++k) {
                    acc[k] = fmaf(s[k][lx], wc[q].x, acc[k]);
                    if (lx + 1 < FSC)
                        acc[k] = fmaf(s[k][lx + 1], wc[q].y, acc[k]);
                    if (lx + 2 < FSC)
                        acc[k] = fmaf(s[k][lx + 2], wc[q].z, acc[k]);
                    if (lx + 3 < FSC)
                        acc[k] = fmaf(s[k][lx + 3], wc[q].w, acc[k]);
                }
            }
#pragma unroll
            for (int k = 0; k < SPT; ++k)
                s[k] += fw;
        }
    } else {
#pragma unroll 1
        for (int ly = 0; ly < FSC; ++ly) {
#pragma unroll
            for (int q = 0; q < FSP / 4; ++q) {
                float4 t[NW];
#pragma unroll
                for (int k = 0; k < NW; ++k)
                    t[k] = plan_w4<WS>(w[k] + 4 * q);
                const int lx = 4 * q;
#pragma unroll
                for (int k = 0; k < SPT; ++k) {
                    const float4& tk = t[SHARED ? 0 : k];
                    acc[k] = fmaf(s[k][lx], tk.x, acc[k]);
                    if (lx + 1 < FSC)
                        acc[k] = fmaf(s[k][lx + 1], tk.y, acc[k]);
                    if (lx + 2 < FSC)
                        acc[k] = fmaf(s[k][lx + 2], tk.z, acc[k]);
                    if (lx + 3 < FSC)
                        acc[k] = fmaf(s[k][lx + 3], tk.w, acc[k]);
                }
            }
#pragma unroll
            for (int k = 0; k < NW; ++k)
                w[k] += FSP;
#pragma unroll
            for (int k = 0; k < SPT; ++k)
                s[k] += fw;
        }
    }
#pragma unroll
    for (int k = 0; k < SPT; ++k)
        if (live & (1u << k))
            dst[(long long)(r[k].x >> 16) * dp + (r[k].x & 0xffffu)] = finish<T>(acc[k], peak);
}

// SPT border pixels that each keep their own weights (ratios whose positions never repeat exactly: no class blocks), stored
// [slot / 32][tap][slot % 32]: the lanes of a warp are neighbouring pixels, so a tap's weights are one contiguous line; the
// windows come from the staged footprint.  Same tap order as strip_sample.
template <typename T, int FSC, int SPT>
__device__ __forceinline__ void plan_per_pixel(const StripArgs& a, const uint4 (&r)[SPT], unsigned live, const float* __restrict__ tile, int fw,
                                               T* __restrict__ dst, long long dp, float peak)
{
    const float* __restrict__ s[SPT];
    const float* __restrict__ w[SPT];
    float acc[SPT];
#pragma unroll
    for (int k = 0; k < SPT; ++k) {
        s[k] = tile + (int)r[k].y;
        w[k] = a.border_w + (size_t)(r[k].z >> 5) * (size_t)(FSC * FSC * 32) + (r[k].z & 31u);
        acc[k] = 0.f;
    }
#pragma unroll 1
    for (int ly = 0; ly < FSC; ++ly) {
#pragma unroll
        for (int lx = 0; lx < FSC; ++lx)
#pragma unroll
            for (int k = 0; k < SPT; ++k)
                acc[k] = fmaf(s[k][lx], __ldg(w[k] + lx * 32), acc[k]);
#pragma unroll
        for (int k = 0; k < SPT; ++k) {
            s[k] += fw;
            w[k] += FSC * 32;
        }
    }
#pragma unroll
    for (int k = 0; k < SPT; ++k)
        if (live & (1u << k))
            dst[(long long)(r[k].x >> 16) * dp + (r[k].x & 0xffffu)] = finish<T>(acc[k], peak);
}

// the prologue path as a real function (row-band launches and tables without a plan)
template <typename T, int FSC, int THREADS, int SPT, int PERIOD, int STEP>
__device__ __noinline__ void strip_block_unplanned(const StripArgs& a, const FrameSet& fsx, unsigned sb, float* __restrict__ tile)
{
    strip_block<T, FSC, THREADS, SPT, PERIOD, STEP>(a, fsx, sb, tile);
}

template <typename T, int FSC, int THREADS, int SPT, int STEP, bool WS>
__device__ __forceinline__ void plan_accumulate(const StripArgs& a, const FrameSet& fsx, unsigned plane, const uint4& r0, const uint4* __restrict__ recs,
                                                const float* __restrict__ tile, int rs, bool deint, const float* __restrict__ wbase,
                                                float* __restrict__ ring)
{
    const unsigned kind = r0.w & 0xffu, live = r0.w >> 8;
    const PlanePtrs& pp = frame_ptrs(fsx);
    T* __restrict__ dst = static_cast<T*>(pp.dst[plane]);
    const long long dp = pp.dst_pitch[plane];
    const float* __restrict__ w0 = WS ? wbase + r0.z : plan_block<FSC>(a, r0.z); // sample 0's weight block
    if (kind == JINC_SK_RUN_ROWS) {
        T* __restrict__ o = dst + (long long)(r0.x >> 16) * dp + (r0.x & 0xffffu);
        if constexpr (FSC > 9 && !WS) {
            if (ring) { // the whole patch is half-warps of row runs sharing a block: weight rows through the ring
                float* __restrict__ mine = ring + (threadIdx.x >> 4) * (JINC_PLAN_RING_DEPTH * ((FSC + 3) & ~3));
                if (STEP > 1 && deint)
                    plan_run_rows_ring<T, FSC, SPT, STEP, (STEP > 1)>(tile + (int)r0.y, rs, w0, mine, o, a.plan_px, fsx.peak);
                else
                    plan_run_rows_ring<T, FSC, SPT, STEP, false>(tile + (int)r0.y, rs, w0, mine, o, a.plan_px, fsx.peak);
                return;
            }
        }
        if (STEP > 1 && deint)
            plan_run_rows<T, FSC, SPT, STEP, WS, (STEP > 1)>(tile + (int)r0.y, rs, w0, o, a.plan_px, fsx.peak);
        else
            plan_run_rows<T, FSC, SPT, STEP, WS, false>(tile + (int)r0.y, rs, w0, o, a.plan_px, fsx.peak);
        return;
    }
    if constexpr (FSC <= 9) {
        if (kind == JINC_SK_RUN_COLS) {
            plan_run_cols<T, FSC, SPT, STEP, WS>(tile + (int)r0.y, rs, w0, dst + (long long)(r0.x >> 16) * dp + (r0.x & 0xffffu),
                                                 (long long)a.plan_py * dp, fsx.peak);
            return;
        }
    }
    uint4 r[SPT];
    r[0] = r0;
#pragma unroll
    for (int k = 1; k < SPT; ++k)
        r[k] = __ldg(recs + k * THREADS);
    if (kind == JINC_SK_FUSED_SHARED) {
        plan_fused<T, FSC, SPT, true, WS>(a, r, live, tile, rs, wbase, dst, dp, fsx.peak);
    } else if (kind == JINC_SK_FUSED_SEP) {
        plan_fused<T, FSC, SPT, false, WS>(a, r, live, tile, rs, wbase, dst, dp, fsx.peak);
    } else if (kind == JINC_SK_PER_PIXEL) {
        plan_per_pixel<T, FSC, SPT>(a, r, live, tile, rs, dst, dp, fsx.peak);
    } else { // JINC_SK_PER_SAMPLE: no vector-readable block (per-pixel border weights): straight from global memory
#pragma unroll 1
        for (int k = 0; k < SPT; ++k)
            if (live & (1u << k))
                strip_sample<T, FSC>(a, fsx, (int)(r[k].x & 0xffffu), (int)(r[k].x >> 16), (int)plane);
    }
}

template <typename T, int FSC, int THREADS, int SPT, int STEP>
__device__ __forceinline__ void strip_block_planned(const StripArgs& a, const FrameSet& fsx, unsigned sb, float* __restrict__ tile)
{
    static_assert(FSC > 0, "planned strips need a compile-time window size");
    static_assert(sizeof(StripPlanPatch) == 48, "three 16-byte loads");
    constexpr int FSP = (FSC + 3) & ~3, WB4 = FSC * FSP / 4;
    const unsigned plane = div_by(sb, a.blocks_per_plane_magic);
    const unsigned pid = sb - plane * a.blocks_per_plane;
    const int4* __restrict__ pd = reinterpret_cast<const int4*>(a.plan_patches + pid);
    const int4 pa = __ldg(pd);     // sx_lo, sy_lo, fw, fh
    const int4 pb = __ldg(pd + 1); // magic, n_wb, wdata_off, tile_floats
    const int4 pc = __ldg(pd + 2); // row_stride, sub, deint, ring
    const uint4* __restrict__ recs = a.plan_threads + (size_t)pid * (unsigned)(SPT * THREADS) + threadIdx.x;
    const uint4 r0 = __ldg(recs);
    const PlanePtrs& pp = frame_ptrs(fsx);
    constexpr int D = SPT * STEP, SUBC = plan_deint_sub(STEP, SPT, FSC);
    const int fw = pa.z, rs = pc.x;
    const bool deint = STEP > 1 && pc.z != 0; // then rs == D * SUBC
    const bool ws = pb.y >= 0; // the patch's weight blocks are staged
    float* __restrict__ wsm = tile + pb.w;
    const float* __restrict__ wglobal = a.plan_wdata + (unsigned)pb.z;
    {
        // the patch's weight blocks (packed in plan order: a straight copy) and its source footprint, converted to float.
        // The first round of both is loaded before anything is stored: one memory round trip for the usual patch.
        const float4* __restrict__ wsrc = reinterpret_cast<const float4*>(wglobal);
        float4* __restrict__ wdst = reinterpret_cast<float4*>(wsm);
        const int nw4 = max(pb.y, 0) * WB4;
        const int pitch = (int)pp.src_pitch[plane];
        const T* __restrict__ src = static_cast<const T*>(pp.src[plane]) + (long long)pa.y * pitch + pa.x;
        const unsigned n = (unsigned)(fw * pa.w), magic = (unsigned)pb.x;
        float4 wv[2];
#pragma unroll
        for (int u = 0; u < 2; ++u)
            wv[u] = __ldg(wsrc + min((int)threadIdx.x + u * THREADS, max(nw4 - 1, 0)));
        // wide windows have footprints of thousands of samples: sixteen loads per thread in flight instead of four
        constexpr int U = FSC > 9 ? 16 : 4;
        for (unsigned e0 = threadIdx.x; e0 < n; e0 += U * THREADS) {
            T v[U];
            unsigned at[U];
#pragma unroll
            for (int u = 0; u < U; ++u) { // all loads of a round are issued before the first conversion
                const unsigned e = min(e0 + u * THREADS, n - 1);
                const unsigned row = __umulhi(e, magic), col = e - row * (unsigned)fw;
                v[u] = __ldg(src + (int)(row * (unsigned)pitch + col));
                at[u] = deint ? row * (unsigned)(D * SUBC) + (col % (unsigned)D) * (unsigned)SUBC + col / (unsigned)D : e;
            }
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (e0 + u * THREADS < n)
                    tile[at[u]] = sample_to_float(v[u]);
        }
#pragma unroll
        for (int u = 0; u < 2; ++u)
            if ((int)threadIdx.x + u * THREADS < nw4)
                wdst[threadIdx.x + u * THREADS] = wv[u];
        for (int i = threadIdx.x + 2 * THREADS; i < nw4; i += THREADS)
            wdst[i] = __ldg(wsrc + i);
    }
    __syncthreads();
    if ((r0.w & 0xffu) == JINC_SK_NONE)
        return;
    if (ws)
        plan_accumulate<T, FSC, THREADS, SPT, STEP, true>(a, fsx, plane, r0, recs, tile, rs, deint, wsm, nullptr);
    else
        plan_accumulate<T, FSC, THREADS, SPT, STEP, false>(a, fsx, plane, r0, recs, tile, rs, deint, nullptr, pc.w > 0 ? tile + pc.w : nullptr);
}

// Role of block b in a merged grid of interior tile blocks and `strips` strip blocks: strip block k sits at grid
// position k << shift (their latency-bound work then hides under the FMA-bound tiles sharing the SM) instead of
// trailing the grid.  Returns true for a strip block and its index in `id`, else the tile index.  32-bit shifts only:
// this runs in every block's prologue.
__device__ __forceinline__ bool block_role(unsigned b, unsigned strips, int shift, unsigned& id)
{
    const unsigned k = b >> shift;
    if ((b & ((1u << shift) - 1u)) == 0u && k < strips) {
        id = k;
        return true;
    }
    id = b - min(k + 1u, strips);
    return false;
}

// largest shift with (strips - 1) << shift < interior + strips, i.e. every strip block has a grid position
inline int strip_role_shift(long long interior, long long strips)
{
    int shift = 0;
    if (strips > 0)
        while (shift < 30 && (strips << (shift + 1)) <= interior + strips)
            ++shift;
    return shift;
}

// Cuts the rectangles into patches of `outputs` samples (one strip block each), at most `max_pw` wide; returns the
// number of strip blocks per plane.
inline long long set_strip_rects(StripArgs& a, const Rect* rects, int n_rects, int outputs, int max_pw, size_t smem_bytes)
{
    unsigned total = 0;
    int k = 0;
    max_pw = std::min(max_pw, outputs);
    for (int r = 0; r < n_rects; ++r) {
        const long long w = rects[r].x1 - rects[r].x0, h = rects[r].y1 - rects[r].y0;
        if (w <= 0 || h <= 0)
            continue;
        int pwl = 3; // patches are at least 8 wide
        while ((1 << pwl) < w && (1 << pwl) < max_pw)
            ++pwl;
        const long long pw = 1ll << pwl, ph = outputs / pw;
        a.rect[k] = rects[r];
        a.row_mode[k] = w >= h ? 1 : 0; // top/bottom strips are wide, left/right strips are tall
        a.pw_log2[k] = pwl;
        a.patches_x[k] = (unsigned)((w + pw - 1) / pw);
        a.patches_x_magic[k] = div_magic(a.patches_x[k]);
        a.patch_begin[k] = total;
        total += a.patches_x[k] * (unsigned)((h + ph - 1) / ph);
        ++k;
    }
    for (int j = k; j < 4; ++j) {
        a.rect[j] = Rect{0, 0, 1, 1};
        a.row_mode[j] = 1;
        a.pw_log2[j] = 3;
        a.patches_x[j] = 1;
        a.patches_x_magic[j] = div_magic(1);
        a.patch_begin[j] = total;
    }
    a.patch_begin[4] = total;
    a.blocks_per_plane = total;
    a.blocks_per_plane_magic = div_magic(total);
    a.smem_floats = (unsigned)(smem_bytes / sizeof(float));
    return total;
}

// ------------------------------------------------------------------------------------------ exact-2x kernel

constexpr int UP_TX = 4;                     // cells per thread along x
constexpr int UP_WARPS = 4;
constexpr int UP_THREADS = UP_WARPS * 32;
constexpr int UP_CW = 32 * UP_TX;            // cells per tile row (128 -> 256 output samples)
// cell-row pairs per warp: the smallest window (tap 3) takes twice as tall a tile -- its tiles are short-lived, and the halo
// rows, the staging round trip and the block start-up weigh most there -- at five instead of six blocks per SM
constexpr int up_rpw(int fs) { return fs <= 7 ? 4 : 2; }
constexpr int up_ch(int fs) { return 2 * UP_WARPS * up_rpw(fs); } // cell rows per tile (16 -> 32 output rows, or 32 -> 64)
constexpr int UP_STRIP_SPT = 4;              // strip role: outputs per thread (patches of 1024 outputs, up to 256 wide)
constexpr int UP_STRIP_MAX_PW = 64;   // wide strips are cut into 64 x 8 patches: the rows of a strip share most of their source rows

template <int FS>
struct UpGeom {
    static constexpr int FSP = (FS + 3) & ~3;       // weight row stride (16-byte rows)
    static constexpr int NSEG = UP_TX + 1 + FS - 1; // pair columns a thread reads per row (ox1 <= 1)
    static constexpr int NC = UP_CW + FS;           // pair columns per tile row (CW + ox1 + FS - 1)
    static constexpr int NCP = (NC + 3) & ~3;
    static constexpr int SUB = NCP / 4;             // columns are de-interleaved by (c & 3): 4 sub-rows of SUB
    static constexpr int RPW = up_rpw(FS), CH = up_ch(FS);
    static constexpr int NR = CH + 1 + FS - 1;      // pair rows per tile (CH + oy1 + FS - 1)
    static constexpr size_t SMEM = (size_t)NR * NCP * sizeof(float2);
};

template <int FS>
struct alignas(16) UpWeights {
    float w[2][2][FS][UpGeom<FS>::FSP]; // [py][px][ly][lx]
};

struct UpArgs {
    FrameSet fr;
    StripArgs st;         // border strips around the interior (run by the blocks after the interior tiles)
    int src_w, src_h;
    int x0, y0, ncx;      // output origin of the periodic interior, cells per row
    int sx0, sy0;         // window origin of cell (0,0), phase (0,0)
    int cy_begin, cy_end; // cell rows to produce (row-band split)
    int tiles_x, tiles_per_plane, interior_blocks; // interior_blocks = tiles_per_plane * n_planes
    unsigned tiles_x_magic, tiles_per_plane_magic; // div_magic of the two tile divisors
    int strip_blocks, strip_shift;
};

inline bool up2x_supported(int fs) { return fs == 7 || fs == 9 || fs == 11 || fs == 13 || fs == 15 || fs == 17; } // taps 3..8

inline size_t up2x_smem_bytes(int fs)
{
    switch (fs) {
    case 7: return UpGeom<7>::SMEM;
    case 9: return UpGeom<9>::SMEM;
    case 11: return UpGeom<11>::SMEM;
    case 13: return UpGeom<13>::SMEM;
    case 15: return UpGeom<15>::SMEM;
    case 17: return UpGeom<17>::SMEM;
    default: return 0;
    }
}

// ------------------------------------------------------------------------------------------ integer-ratio downscale kernel
//
// Output (x,y) of the interior reads the FS x FS window at (sx0 + Q*x, sy0 + Q*y) with ONE weight block for every
// pixel (config 5: Q = 4, FS = 50, 2500 taps per sample).  All threads apply the same weight at the same time, so
// weights again come from the constant bank through uniform registers.  Three ideas shape the kernel:
//   * polyphase columns: lx = Q*m + p turns the x-sum into Q stride-1 convolutions over the de-interleaved sequences
//     S_p[j] = S[Q*j + p]; a thread that owns NX consecutive outputs reads a span of NX+MT-1 values per (row, p) and
//     uses each for up to NX outputs, and one weight fetch feeds NX FFMA2s;
//   * tap pairing: one packed FFMA2 multiplies the vertical sample pair {S[r][c], S[r+1][c]} with the weight pair
//     {w[ly][lx], w[ly+1][lx]} into the two halves of ONE output's accumulator (even-row and odd-row partial sums,
//     added in the epilogue).  With an even Q every output row of the thread sees the same pairing and a staged pair
//     is reused for both output rows of the thread; with an odd Q (1/3, and the passes of the periodic 2:3 / 4:3
//     paths, where each phase pair's sub-lattice is a ratio-3 problem written with an output stride) the second row
//     starts on an odd source row, so its window is taken one row early with a leading zero weight -- a second weight
//     set {w[2k-1], w[2k]}, still warp-uniform;
//   * raw sample pairs in shared memory for integer formats (two 16-bit samples per 32-bit word; u8 is widened while
//     staging), so a 64x32-output tile with its 302x174-sample footprint fits twice per SM.  The float value is made
//     after the shared-memory load.  For depths up to 15 bits that costs ONE byte permute per sample: staging stores
//     x << (15 - bits), and PRMT drops those 16 bits into mantissa bits [22:8] of 0x3F000000, i.e. f = 0.5 + x' / 65536
//     exactly.  The kernel accumulates sum(w * f) and the epilogue removes the 0.5 * sum(w) bias (host-computed per
//     accumulator half) and rescales by a power of two.  Precision matches a direct float sum of 15-bit samples (the
//     accumulator's ulp relative to one input LSB is the same).  16-bit samples use I2F instead (XU pipe).
// Columns are de-interleaved by c mod (Q*NX) so a warp's loads are bank-conflict free.
constexpr int DN_TW = 64;  // output columns per tile
constexpr int DN_TH = 32;  // output rows per tile (integer formats; float tiles are half as tall)

constexpr int DN_STRIP_SPT = 4;    // strip role: outputs per thread (four independent accumulator chains), patches at most 64 wide (the windows are wide)
constexpr int DN_STRIP_MAX_PW = 64;

enum { DN_CVT_I2F = 0, DN_CVT_PRMT = 1, DN_CVT_FLOAT = 2 };

template <typename T, int FS, int Q, int NX, int NY>
struct DownGeom {
    static constexpr bool IS_FLOAT = is_float_sample<T>::value; // float and half planes: float pairs, half-height tiles
    using Word = typename std::conditional<IS_FLOAT, float2, uint32_t>::type; // {row 2k, row 2k+1}
    static constexpr int LX = DN_TW / NX;               // lanes along x
    static constexpr int LY = 32 / LX;                  // lanes along y
    static constexpr int TH = IS_FLOAT ? DN_TH / 2 : DN_TH;
    static constexpr int WARPS = TH / (LY * NY);
    static constexpr int THREADS = 32 * WARPS;
    static constexpr int FSE = (FS + 1) & ~1;           // window rows rounded up to whole pairs
    static constexpr bool ODD = (Q & 1) != 0;
    // Row pairs are formed from the tile origin.  With an odd ratio the second output row of a thread starts on an odd
    // source row: its window is taken one row early with a leading zero weight (weight set 1: {w[2k-1], w[2k]}), so it
    // still reads whole pairs, OFF1 pairs below the first row.
    static constexpr int NKW = FSE / 2;                 // weight row pairs of output row 0 (set 0: {w[2k], w[2k+1]})
    static constexpr int NKW1 = ODD ? (FS + 2) / 2 : NKW; // weight row pairs of output row 1
    static constexpr int OFF1 = ODD ? (Q - 1) / 2 : Q / 2; // row pairs between output rows 0 and 1 of a thread
    static constexpr int MT = (FS + Q - 1) / Q;         // taps per polyphase component
    static constexpr int SPAN = NX + MT - 1;            // values a thread reads per (row pair, p)
    static constexpr int D = Q * NX;                    // column de-interleave modulus
    static constexpr int NCOL = Q * (DN_TW - 1) + Q * (MT - 1) + Q; // columns a tile row can be asked for
    static constexpr int SUB = (NCOL + D - 1) / D;
    static constexpr int NROWS = Q * (TH - 1) + 2 * NKW1;
    static constexpr int NROWP = (NROWS + 1) / 2;       // row pairs per tile
    static constexpr int NK = OFF1 * (NY - 1) + NKW1;   // row pairs a thread walks
    static constexpr int HALF = NY * Q / 2;             // row pairs between lane groups that differ in y
    static constexpr int rs_pad()
    {
        for (int pad = 0; pad < 32; ++pad) // lane group g lands on banks [g*LX, g*LX + LX)
            if (((D * SUB + pad) * HALF) % 32 == LX % 32)
                return pad;
        return 0;
    }
    static constexpr int RS = D * SUB + rs_pad();       // row-pair stride in words
    static constexpr size_t SMEM = (size_t)NROWP * RS * sizeof(Word);
    static_assert(NY == 2, "the thread's two output rows carry the pairing parity");
    static_assert(TH % (LY * NY) == 0 && WARPS >= 1, "tile rows must split evenly over the warps");
    static_assert(LX - 1 + (Q * (SPAN - 1) + Q - 1) / D < SUB, "span reaches past the tile row");
};

template <int FS, int Q>
struct alignas(16) DownWeights {
    static constexpr int MT = (FS + Q - 1) / Q;
    static constexpr int NSET = (Q & 1) ? 2 : 1;                        // odd ratios: a second set shifted by one row
    static constexpr int NKWMAX = (Q & 1) ? (FS + 2) / 2 : ((FS + 1) & ~1) / 2;
    float2 w[NSET][NKWMAX][Q][MT]; // set 0: [k][p][m] = {w[2k][Q*m+p], w[2k+1][Q*m+p]}; set 1: {w[2k-1][..], w[2k][..]}; outside the window 0
};

// the weight blocks of all passes of one launch (1 for an integer ratio; P*P for the periodic paths: blockIdx.z = pass)
template <int FS, int Q, int NPASS>
struct alignas(16) DownWeightsN {
    DownWeights<FS, Q> pass[NPASS];
};

constexpr int DN_MAX_PASSES = 16;

// what differs between the passes of a launch
struct DownPass {
    int tsx0, tsy0;       // window origin of output (x0, y0)
    int out_x0, out_y0;   // plane coordinates of (x0, y0)
    float bias_x[2], bias_y[2]; // PRMT conversion, output row j of a thread: out = ((acc.x - bias_x[j]) + (acc.y - bias_y[j])) * out_scale
};

struct DownArgs {
    FrameSet fr;
    StripArgs st;
    int src_w, src_h;
    int x0, y0, x1, y1;  // output rectangle produced by the tiles (y0..y1 already cut to the row band); for the periodic
                         // paths these count CELLS of a pass's sub-lattice
    int out_stride;      // distance between neighbouring outputs in the plane (1, or P for a periodic pass)
    int n_passes;
    DownPass pass[DN_MAX_PASSES];
    int tiles_x, tiles_per_plane, interior_blocks, strip_blocks, strip_shift;
    unsigned tiles_x_magic, tiles_per_plane_magic; // div_magic of the two tile divisors
    int pre_shift;       // PRMT conversion: samples are staged as x << pre_shift
    float out_scale;     // PRMT conversion: power-of-two rescale of the de-biased sum
    bool want_strip_plan; // host only: a whole-frame launch, the strips may run from the table's plan
};

// ---- launch entry points, one explicit instantiation per sample type (jinc_up2x_*.cu, jinc_down_*.cu)
// 0 launched, 1 unsupported filter size, <0 error
template <typename T>
int launch_up2x(const jinc_table* t, UpArgs& a, long long strip_blocks, int n_frames, cudaStream_t st);
// 0 launched, 2 nothing to do, 1 unsupported geometry, <0 error
template <typename T>
int launch_down(const jinc_table* t, DownArgs& a, int q, const int* wblocks, bool want_strips, int n_frames, cudaStream_t st,
                const Rect* rects, int n_rects);

// ------------------------------------------------------------------------------------------ chunked-cells kernel (jinc_cells.cuh)

constexpr int CL_STRIP_SPT = 4;    // strip role of the cells kernel: outputs per thread, widest patch
constexpr int CL_STRIP_MAX_PW = 64;

struct CellsArgs {
    FrameSet fr;
    StripArgs st;
    const int32_t* cx_cell; // per x-chunk: first cell of its group, first live cell, live cells; per residue: origin, phase rank
    const int32_t* cx_i0;
    const int32_t* cx_n;
    const int32_t* cx_org;
    const int32_t* cx_rank;
    const int32_t* cy_cell;
    const int32_t* cy_i0;
    const int32_t* cy_n;
    const int32_t* cy_org;
    const int32_t* cy_rank;
    const float* wblocks; // phase blocks [block][FS][wstride]
    int wstride;
    int Px, Py, x0, y0, n_rank_x;
    int n_cx;                   // x-chunks
    int cyk_begin, cyk_end;     // y-chunks of this launch (row band)
    int cell_y_begin, cell_y_end; // cell rows to produce
    int src_w, src_h;
    int tiles_x, tiles_per_plane, interior_blocks, strip_blocks, strip_shift;
    unsigned tiles_x_magic, tiles_per_plane_magic;
    bool want_strip_plan; // host only: a whole-frame launch, the strips may run from the table's plan
};

// defined in jinc_cells.cuh, instantiated in jinc_cells_<type>_q<Q>.cu (one source step Q per translation unit)
template <typename T, int Q>
int launch_cells_q(const jinc_table* t, CellsArgs& a, int n_frames, cudaStream_t st, const Rect* rects, int n_rects);

// Q = 1: 3x, 4x, 5x ... and shifts at 1:1;  Q = 2: 3:2 (720p -> 1080p, 1440p -> 2160p), 5:2, 9:2;  Q = 3: 4:3 (1080p -> 1440p),
// 5:3;  Q = 4: 5:4, 9:4 (480p -> 1080p), and the 3:4 downscale (1440p -> 1080p)
template <typename T>
int launch_cells(const jinc_table* t, CellsArgs& a, int n_frames, cudaStream_t st, const Rect* rects, int n_rects)
{
    switch (t->cells.Q) {
    case 1: return launch_cells_q<T, 1>(t, a, n_frames, st, rects, n_rects);
    case 2: return launch_cells_q<T, 2>(t, a, n_frames, st, rects, n_rects);
    case 3: return launch_cells_q<T, 3>(t, a, n_frames, st, rects, n_rects);
    case 4: return launch_cells_q<T, 4>(t, a, n_frames, st, rects, n_rects);
    default: return 1;
    }
}

inline bool periodic_supported(const jinc_table* t)
{
    const PeriodicPlan& u = t->periodic;
    if (!u.ok)
        return false;
    if (u.P == 2 && u.Q == 3)
        return t->sc.fs == 10 || t->sc.fs == 13; // taps 3 and 4 at 2:3 (1080p -> 720p)
    if (u.P == 4 && (u.Q == 3 || u.Q == 1))
        return t->sc.fs == 7 || t->sc.fs == 9;   // taps 3 and 4 at 4:3 (1080p -> 1440p) and at 4x (540p -> 2160p)
    return false;
}

inline bool down_supported(const jinc_table* t)
{
    if (!t->down.ok || t->down.qx != t->down.qy)
        return false;
    switch (t->down.qx * 1000 + t->sc.fs) {
    case 2013: case 2017: case 2025: case 2033: case 3020: case 4026: case 4034: case 4050: return true;
    default: return false;
    }
}

} // namespace jinc_rs

#endif
