// jinc_resize.cu -- the general (any ratio) resample kernel and the launcher that picks a kernel family per table.
//
// Replaces JincResize::resize_plane_c<T,thr,subsampled> (src/JincResize.cpp:536-601) and the three SIMD copies of
// its inner loop.  The layout of the kernels, the block roles of a merged launch and the strip role for border pixels
// are described once, in jinc_resample.cuh; the kernel families live in jinc_up2x.cuh (exact 2x), jinc_down.cuh
// (integer-ratio downscale and the exactly periodic 2:3 path) and jinc_cells.cuh (rational ratios with piecewise-periodic
// phases), each instantiated once per sample type in its own translation unit so that the build runs in parallel.
#include <chrono>
#include <cstdio>
#include <cstdlib>

#include "jinc_resample.cuh"

using namespace jinc_rs;

namespace {

struct GeneralArgs {
    FrameSet fr;
    StripArgs st;
};

constexpr int GEN_SPT = 4;                  // outputs per thread of the general kernel
constexpr int GEN_MAX_PW = 128;             // its patches are 128 x 8 outputs: a warp covers ONE output row (consecutive lanes read nearly consecutive shared-memory words)
constexpr size_t GEN_SMEM = (size_t)96 << 10; // staging space (two blocks per SM)

// General kernel: one block = one patch of 64 x 16 outputs of ALL NP planes that share the table.  Every output has its
// own phase block (that is what "general ratio" means), so the weight stream from L1/L2 is the bottleneck: a thread
// owns 4 outputs of one row and applies each float4 of weights to the same output of all NP planes (and the 4 outputs
// run interleaved), which divides the weight traffic per sample by NP.  Falls back to the per-plane strip role when
// the NP source footprints do not fit in shared memory or a sample has no vector-readable block.
// FSC > 0 fixes the window size at compile time (taps 3 and 4 at upscale ratios): the weight row of an output is then
// read with back-to-back vector loads -- both halves of every 32-byte sector are consumed at once instead of coming back
// from L2 a second time after the other streams of the block have pushed it out of L1 -- and the tap loops unroll.
template <typename T, int NP, int FSC>
__global__ void __launch_bounds__(STRIP_THREADS) resample_strips(const __grid_constant__ GeneralArgs ga)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* __restrict__ tile = reinterpret_cast<float*>(smem_raw);
    const StripArgs& a = ga.st;
    constexpr int SPT = GEN_SPT, THREADS = STRIP_THREADS;
    const int fs = FSC > 0 ? FSC : a.fs;
    const unsigned pid = blockIdx.x;
    const unsigned pyi = div_by(pid, a.patches_x_magic[0]), pxi = pid - pyi * a.patches_x[0];
    const int pwl = a.pw_log2[0];
    const int ox0 = a.rect[0].x0 + (int)(pxi << pwl), oy0 = a.rect[0].y0 + (int)pyi * ((THREADS * SPT) >> pwl);
    const int nx = min(1 << pwl, a.rect[0].x1 - ox0), ny = min((THREADS * SPT) >> pwl, a.rect[0].y1 - oy0);
    const int sx_lo = a.start_x[ox0], sy_lo = a.start_y[oy0];
    const int fw = a.start_x[ox0 + nx - 1] + fs - sx_lo, fh = a.start_y[oy0 + ny - 1] + fs - sy_lo;
    const unsigned n = (unsigned)(fw * fh);

    // this thread's outputs: (tx + k * PW/SPT, ty); live ones are a prefix
    const int txl = pwl - 2;
    const int tx = (int)threadIdx.x & ((1 << txl) - 1), ty = (int)threadIdx.x >> txl;
    StripMeta meta[SPT];
    unsigned live = 0;
    bool vec = true;
#pragma unroll
    for (int k = 0; k < SPT; ++k) {
        const int lx = tx + (k << txl);
        if (lx < nx && ty < ny) {
            meta[k] = strip_meta<0>(a, ox0 + lx, oy0 + ty);
            live |= 1u << k;
            vec = vec && meta[k].wstride != 0 && (meta[k].wstride & 3) == 0;
        }
    }
    // the whole block takes one path: block-wide vote (every thread reaches it)
    const bool fast = NP * n <= a.smem_floats && __syncthreads_and(vec ? 1 : 0) != 0;
    if (!fast) {
        for (int pl = 0; pl < NP; ++pl) {
            __syncthreads(); // the previous plane's staged footprint is no longer read
            strip_block<T, 0, THREADS, SPT>(a, ga.fr, (unsigned)pl * a.blocks_per_plane + pid, tile);
        }
        return;
    }

    const PlanePtrs& pp = frame_ptrs(ga.fr);
    {
        const unsigned magic = 0xFFFFFFFFu / (unsigned)fw + 1u; // floor(e / fw) = umulhi(e, magic) while e * fw < 2^32
#pragma unroll
        for (int pl = 0; pl < NP; ++pl) {
            const int pitch = (int)pp.src_pitch[pl];
            const T* __restrict__ src = static_cast<const T*>(pp.src[pl]) + (long long)sy_lo * pitch + sx_lo;
            float* __restrict__ tp = tile + pl * n;
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
                        tp[e0 + u * THREADS] = sample_to_float(v[u]);
            }
        }
    }
    __syncthreads();
    if (!(live & 1u))
        return;
#pragma unroll
    for (int k = 1; k < SPT; ++k)
        if (!(live & (1u << k)))
            meta[k] = meta[0]; // computed, not stored

    const float* __restrict__ sp[SPT];
    const float4* __restrict__ w4[SPT];
    float acc[SPT][NP];
#pragma unroll
    for (int k = 0; k < SPT; ++k) {
        sp[k] = tile + (meta[k].sy - sy_lo) * fw + (meta[k].sx - sx_lo);
        w4[k] = reinterpret_cast<const float4*>(meta[k].w);
#pragma unroll
        for (int pl = 0; pl < NP; ++pl)
            acc[k][pl] = 0.f;
    }
    const int wq = meta[0].wstride / 4; // the same for every block of the table
    if constexpr (FSC > 0) {
        constexpr int WQ = (FSC + 3) / 4;
#pragma unroll 1
        for (int ly = 0; ly < FSC; ++ly) {
#pragma unroll
            for (int k = 0; k < SPT; ++k) {
                float4 t[WQ]; // the whole weight row of output k: consecutive vector loads
#pragma unroll
                for (int q = 0; q < WQ; ++q)
                    t[q] = __ldg(w4[k] + q);
#pragma unroll
                for (int q = 0; q < WQ; ++q) {
                    const int lx = 4 * q;
#pragma unroll
                    for (int pl = 0; pl < NP; ++pl) {
                        const float* __restrict__ s = sp[k] + pl * n + lx;
                        float v = acc[k][pl];
                        v = fmaf(s[0], t[q].x, v);
                        if (lx + 1 < FSC)
                            v = fmaf(s[1], t[q].y, v);
                        if (lx + 2 < FSC)
                            v = fmaf(s[2], t[q].z, v);
                        if (lx + 3 < FSC)
                            v = fmaf(s[3], t[q].w, v);
                        acc[k][pl] = v;
                    }
                }
                w4[k] += WQ;
                sp[k] += fw;
            }
        }
    } else {
        for (int ly = 0; ly < fs; ++ly) {
            for (int q = 0; q < wq; ++q) {
                float4 t[SPT];
#pragma unroll
                for (int k = 0; k < SPT; ++k)
                    t[k] = __ldg(w4[k] + q);
                const int lx = 4 * q;
#pragma unroll
                for (int k = 0; k < SPT; ++k) {
#pragma unroll
                    for (int pl = 0; pl < NP; ++pl) {
                        const float* __restrict__ s = sp[k] + pl * n + lx;
                        float v = acc[k][pl];
                        v = fmaf(s[0], t[k].x, v);
                        if (lx + 1 < fs)
                            v = fmaf(s[1], t[k].y, v);
                        if (lx + 2 < fs)
                            v = fmaf(s[2], t[k].z, v);
                        if (lx + 3 < fs)
                            v = fmaf(s[3], t[k].w, v);
                        acc[k][pl] = v;
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < SPT; ++k) {
                w4[k] += wq;
                sp[k] += fw;
            }
        }
    }
#pragma unroll
    for (int pl = 0; pl < NP; ++pl) {
        T* __restrict__ dst = static_cast<T*>(pp.dst[pl]);
        const long long dp = pp.dst_pitch[pl];
#pragma unroll
        for (int k = 0; k < SPT; ++k)
            if (live & (1u << k))
                dst[(long long)meta[k].y * dp + meta[k].x] = finish<T>(acc[k][pl], ga.fr.peak);
    }
}

template <typename T, int NP, int FSC>
cudaError_t launch_general_fs(const GeneralArgs& ga, unsigned blocks, int n_frames, cudaStream_t st)
{
    cudaError_t e = cudaFuncSetAttribute(resample_strips<T, NP, FSC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GEN_SMEM);
    if (e != cudaSuccess)
        return e;
    resample_strips<T, NP, FSC><<<dim3(blocks, n_frames), STRIP_THREADS, GEN_SMEM, st>>>(ga);
    return cudaGetLastError();
}

template <typename T, int NP>
cudaError_t launch_general_np(const GeneralArgs& ga, unsigned blocks, int n_frames, cudaStream_t st)
{
    // the unrolled variants need the padded weight rows (16-byte vectors) the table build provides for these sizes
    if (ga.st.weights_p && ga.st.fs == 7)
        return launch_general_fs<T, NP, 7>(ga, blocks, n_frames, st);
    if (ga.st.weights_p && ga.st.fs == 9)
        return launch_general_fs<T, NP, 9>(ga, blocks, n_frames, st);
    return launch_general_fs<T, NP, 0>(ga, blocks, n_frames, st);
}

// weights of one output pixel exactly as the reference defines them (introspection for parity tests)
__global__ void pixel_weights_kernel(StripArgs a, int x, int y, float* out)
{
    const int fs = a.fs;
    const int rx = a.rank_x[x], ry = a.rank_y[y];
    if (rx >= 0 && ry >= 0) {
        const float* w = a.weights + (size_t)(ry * a.n_rank_x + rx) * fs * fs;
        for (int t = threadIdx.x; t < fs * fs; t += blockDim.x)
            out[t] = w[t];
        return;
    }
    if (a.border_block) {
        // what the resample kernels apply: the block of this border pixel's class
        const int fsp = (fs + 3) & ~3;
        const float* w = a.border_wb + (size_t)a.border_block[jinc_border_slot(a.bg, x, y)] * (unsigned)(fs * fsp);
        for (int t = threadIdx.x; t < fs * fs; t += blockDim.x)
            out[t] = w[(t / fs) * fsp + t % fs];
        return;
    }
    const int sx = a.start_x[x], sy = a.start_y[y];
    const float px = a.pos_x[x], py = a.pos_y[y];
    const float sum = a.border_sum[jinc_border_slot(a.bg, x, y)];
    for (int t = threadIdx.x; t < fs * fs; t += blockDim.x) {
        const int ly = t / fs, lx = t - ly * fs;
        const double dy2 = jinc_tap_dist2(py, a.src_h, sy + ly, a.step_y);
        const double dx2 = jinc_tap_dist2(px, a.src_w, sx + lx, a.step_x);
        out[t] = __fdiv_rn(jinc_lut_weight(a.lut, __dadd_rn(dx2, dy2), a.radius2, a.idx_scale), sum);
    }
}

} // namespace

void jinc_rs::fill_strip_args(const jinc_table* t, StripArgs& a)
{
    memset(&a, 0, sizeof(a));
    a.start_x = t->ax[0].start;
    a.start_y = t->ax[1].start;
    a.rank_x = t->ax[0].rank;
    a.rank_y = t->ax[1].rank;
    a.pos_x = t->ax[0].pos;
    a.pos_y = t->ax[1].pos;
    a.weights = t->d_weights;
    a.weights_p = t->d_weights_p;
    a.lut = t->d_lut;
    a.border_sum = t->d_border_sum;
    a.border_w = t->d_border_w;
    a.border_block = t->d_border_block;
    a.border_wb = t->d_border_wb;
    a.bg = t->bgeom;
    a.fs = t->sc.fs;
    a.n_rank_x = t->ax[0].n_rank;
    a.src_w = t->sc.src_w;
    a.src_h = t->sc.src_h;
    a.step_x = t->sc.filt_step[0];
    a.step_y = t->sc.filt_step[1];
    a.radius2 = t->sc.radius2;
    a.idx_scale = t->sc.idx_scale;
}

namespace {

// ------------------------------------------------------------------------------------------ launcher

template <typename T>
int launch_typed(const jinc_table* t, const FrameSet& fr, int n_frames, int y_begin, int y_end, cudaStream_t st, int* launches,
                 int parts)
{
    const int W = t->sc.dst_w;
    StripArgs sa;
    fill_strip_args(t, sa);
    Rect rects[4];
    int n_rects = 0;

    if (t->fast_path == JINC_PATH_UP2X && up2x_supported(t->sc.fs)) {
        const Up2xPlan& u = t->up2x;
        // cell rows whose 2 output rows lie inside [y_begin, y_end)
        const int cb = (std::max(y_begin, u.y0) - u.y0 + 1) / 2;
        const int ce = (std::min(y_end, u.y0 + 2 * u.ncy) - u.y0) / 2;
        if (ce > cb) {
            const int fy0 = u.y0 + 2 * cb, fy1 = u.y0 + 2 * ce;
            if (parts & JINC_PART_BORDER) {
                rects[n_rects++] = Rect{0, y_begin, W, fy0};  // top strip
                rects[n_rects++] = Rect{0, fy1, W, y_end};    // bottom strip
                rects[n_rects++] = Rect{0, fy0, t->ix0, fy1}; // left strip
                rects[n_rects++] = Rect{t->ix1, fy0, W, fy1}; // right strip
            }
            UpArgs a;
            memset(&a, 0, sizeof(a));
            a.fr = fr;
            a.st = sa;
            long long strip_blocks =
                set_strip_rects(a.st, rects, n_rects, UP_THREADS * UP_STRIP_SPT, UP_STRIP_MAX_PW, up2x_smem_bytes(t->sc.fs)) * fr.n_planes;
            if (n_rects == 4 && y_begin == 0 && y_end == t->sc.dst_h && attach_strip_plan(t, a.st, UP_THREADS, UP_STRIP_SPT))
                strip_blocks = (long long)a.st.blocks_per_plane * fr.n_planes; // whole frame: the strip blocks run from the table's plan
            a.src_w = t->sc.src_w;
            a.src_h = t->sc.src_h;
            a.x0 = u.x0;
            a.y0 = u.y0;
            a.ncx = u.ncx;
            a.sx0 = u.sx0;
            a.sy0 = u.sy0;
            a.cy_begin = cb;
            a.cy_end = ce;
            a.tiles_x = (u.ncx + UP_CW - 1) / UP_CW;
            a.tiles_per_plane = a.tiles_x * ((ce - cb + up_ch(t->sc.fs) - 1) / up_ch(t->sc.fs));
            a.tiles_x_magic = div_magic((unsigned)a.tiles_x);
            a.tiles_per_plane_magic = div_magic((unsigned)a.tiles_per_plane);
            a.interior_blocks = (parts & JINC_PART_INTERIOR) ? a.tiles_per_plane * fr.n_planes : 0;
            if (a.interior_blocks + strip_blocks == 0)
                return JINC_OK;
            const int rc = launch_up2x<T>(t, a, strip_blocks, n_frames, st);
            if (rc <= 0) {
                if (rc == 0)
                    ++*launches;
                return rc;
            }
        }
    }
    if (t->fast_path == JINC_PATH_CELLS && t->cells.ok) {
        const CellsAxis &ax = t->cells.ax[0], &ay = t->cells.ax[1];
        // cell rows whose Py output rows lie inside [y_begin, y_end)
        const int cb = (std::max(y_begin, ay.first) - ay.first + ay.P - 1) / ay.P;
        const int ce = (std::min(y_end, ay.first + ay.P * ay.ncells) - ay.first) / ay.P;
        if (ce > cb) {
            const int fy0 = ay.first + ay.P * cb, fy1 = ay.first + ay.P * ce;
            if (parts & JINC_PART_BORDER) {
                rects[n_rects++] = Rect{0, y_begin, W, fy0};
                rects[n_rects++] = Rect{0, fy1, W, y_end};
                rects[n_rects++] = Rect{0, fy0, t->ix0, fy1};
                rects[n_rects++] = Rect{t->ix1, fy0, W, fy1};
            }
            CellsArgs a;
            memset(&a, 0, sizeof(a));
            a.fr = fr;
            a.st = sa;
            a.cx_cell = ax.d_cell;
            a.cx_i0 = ax.d_i0;
            a.cx_n = ax.d_n;
            a.cx_org = ax.d_org;
            a.cx_rank = ax.d_rank;
            a.cy_cell = ay.d_cell;
            a.cy_i0 = ay.d_i0;
            a.cy_n = ay.d_n;
            a.cy_org = ay.d_org;
            a.cy_rank = ay.d_rank;
            a.wblocks = t->d_weights_p ? t->d_weights_p : t->d_weights;
            a.wstride = t->d_weights_p ? ((t->sc.fs + 3) & ~3) : t->sc.fs;
            a.Px = ax.P;
            a.Py = ay.P;
            a.x0 = ax.first;
            a.y0 = ay.first;
            a.n_rank_x = t->ax[0].n_rank;
            a.n_cx = ax.n_chunks;
            // y-chunks holding cell rows of [cb, ce): chunk k covers cells [cell[k] + i0[k], cell[k] + i0[k] + n[k])
            int k0 = 0, k1 = ay.n_chunks;
            while (k0 < k1 && ay.cell[k0] + ay.i0[k0] + ay.n[k0] <= cb)
                ++k0;
            while (k1 > k0 && ay.cell[k1 - 1] + ay.i0[k1 - 1] >= ce)
                --k1;
            a.cyk_begin = k0;
            a.cyk_end = k1;
            a.cell_y_begin = cb;
            a.cell_y_end = ce;
            a.src_w = t->sc.src_w;
            a.src_h = t->sc.src_h;
            a.interior_blocks = (parts & JINC_PART_INTERIOR) ? 1 : 0; // resolved to the tile count by the launcher
            a.want_strip_plan = n_rects == 4 && y_begin == 0 && y_end == t->sc.dst_h;
            const int rc = launch_cells<T>(t, a, n_frames, st, rects, n_rects);
            if (rc != 1) {
                if (rc == 0)
                    ++*launches;
                return rc == 2 ? JINC_OK : rc;
            }
            n_rects = 0;
        }
    }
    if (t->fast_path == JINC_PATH_PERIODIC && periodic_supported(t)) {
        const PeriodicPlan& u = t->periodic;
        // cells whose P output rows lie inside [y_begin, y_end)
        const int cb = (std::max(y_begin, u.y0) - u.y0 + u.P - 1) / u.P;
        const int ce = (std::min(y_end, u.y0 + u.P * u.ncy) - u.y0) / u.P;
        if (ce > cb) {
            const int fy0 = u.y0 + u.P * cb, fy1 = u.y0 + u.P * ce;
            if (parts & JINC_PART_BORDER) {
                rects[n_rects++] = Rect{0, y_begin, W, fy0};
                rects[n_rects++] = Rect{0, fy1, W, y_end};
                rects[n_rects++] = Rect{0, fy0, t->ix0, fy1};
                rects[n_rects++] = Rect{t->ix1, fy0, W, fy1};
            }
            // one launch, one pass (blockIdx.z) per phase pair: an integer-ratio-Q problem over the cells, written with
            // stride P; the border strips ride on pass 0
            DownArgs a;
            memset(&a, 0, sizeof(a));
            a.fr = fr;
            a.st = sa;
            a.src_w = t->sc.src_w;
            a.src_h = t->sc.src_h;
            a.x0 = 0;
            a.x1 = u.ncx;
            a.y0 = cb;
            a.y1 = ce;
            a.out_stride = u.P;
            a.n_passes = u.P * u.P;
            int wblocks[DN_MAX_PASSES];
            for (int py = 0; py < u.P; ++py)
                for (int px = 0; px < u.P; ++px) {
                    DownPass& ps = a.pass[py * u.P + px];
                    ps.tsx0 = u.sx0 + u.ox[px];
                    ps.tsy0 = u.sy0 + u.oy[py] + u.Q * cb;
                    ps.out_x0 = u.x0 + px;
                    ps.out_y0 = u.y0 + u.P * cb + py;
                    wblocks[py * u.P + px] = u.wblock[py][px];
                }
            a.interior_blocks = (parts & JINC_PART_INTERIOR) ? 1 : 0;
            const int rc = launch_down<T>(t, a, u.Q, wblocks, n_rects > 0, n_frames, st, rects, n_rects);
            if (rc < 0 || rc == 1)
                return rc < 0 ? rc : jinc_fail(JINC_E_UNSUPPORTED, "resize: periodic passes not instantiated (fs %d)", t->sc.fs);
            if (rc == 0)
                ++*launches;
            return JINC_OK;
        }
    }
    if (t->fast_path == JINC_PATH_DOWN_INT && down_supported(t)) {
        const DownPlan& d = t->down;
        const int fy0 = std::max(y_begin, d.y0), fy1 = std::min(y_end, d.y0 + d.ny);
        if (fy1 > fy0) {
            if (parts & JINC_PART_BORDER) {
                rects[n_rects++] = Rect{0, y_begin, W, fy0};
                rects[n_rects++] = Rect{0, fy1, W, y_end};
                rects[n_rects++] = Rect{0, fy0, t->ix0, fy1};
                rects[n_rects++] = Rect{t->ix1, fy0, W, fy1};
            }
            DownArgs a;
            memset(&a, 0, sizeof(a));
            a.fr = fr;
            a.st = sa;
            a.src_w = t->sc.src_w;
            a.src_h = t->sc.src_h;
            a.x0 = d.x0;
            a.x1 = d.x0 + d.nx;
            a.y0 = fy0;
            a.y1 = fy1;
            a.n_passes = 1;
            a.out_stride = 1;
            a.pass[0].tsx0 = d.sx0;
            a.pass[0].tsy0 = d.sy0 + d.qy * (fy0 - d.y0);
            a.pass[0].out_x0 = a.x0;
            a.pass[0].out_y0 = a.y0;
            a.interior_blocks = (parts & JINC_PART_INTERIOR) ? 1 : 0; // resolved to the tile count by the launcher
            a.want_strip_plan = n_rects == 4 && y_begin == 0 && y_end == t->sc.dst_h;
            const int rc = launch_down<T>(t, a, d.qx, &d.wblock, n_rects > 0, n_frames, st, rects, n_rects);
            if (rc != 1) {
                if (rc == 0)
                    ++*launches;
                return rc == 2 ? JINC_OK : rc;
            }
            n_rects = 0;
        }
    }
    if (!(parts & JINC_PART_BORDER))
        return JINC_OK;
    // no fast path for this geometry (or band): every sample goes through the strip role
    GeneralArgs ga;
    ga.fr = fr;
    ga.st = sa;
    rects[0] = Rect{0, y_begin, W, y_end};
    const long long blocks = set_strip_rects(ga.st, rects, 1, STRIP_THREADS * GEN_SPT, GEN_MAX_PW, GEN_SMEM);
    if (blocks == 0)
        return JINC_OK;
    cudaError_t e = cudaSuccess;
    switch (fr.n_planes) { // one block covers the patch in every plane of the table
    case 1: e = launch_general_np<T, 1>(ga, (unsigned)blocks, n_frames, st); break;
    case 2: e = launch_general_np<T, 2>(ga, (unsigned)blocks, n_frames, st); break;
    case 3: e = launch_general_np<T, 3>(ga, (unsigned)blocks, n_frames, st); break;
    default: e = launch_general_np<T, 4>(ga, (unsigned)blocks, n_frames, st); break;
    }
    if (e != cudaSuccess)
        return jinc_fail(JINC_E_CUDA, "resample_strips launch failed: %s", cudaGetErrorString(e));
    ++*launches;
    return JINC_OK;
}

int check_and_fill(PlanePtrs& pl, int sample, int n_planes, const void* const* d_src, const ptrdiff_t* src_pitch,
                   void* const* d_dst, const ptrdiff_t* dst_pitch)
{
    memset(&pl, 0, sizeof(pl));
    if (!jinc_sample_valid(sample))
        return jinc_fail(JINC_E_INVALID, "resize: sample_bytes must be 1, 2, 4 or JINC_SAMPLE_F16");
    const int sample_bytes = jinc_sample_size(sample);
    for (int i = 0; i < n_planes; ++i) {
        if (!d_src[i] || !d_dst[i])
            return jinc_fail(JINC_E_INVALID, "resize: null plane pointer");
        if (src_pitch[i] % sample_bytes || dst_pitch[i] % sample_bytes)
            return jinc_fail(JINC_E_INVALID, "resize: pitch must be a multiple of the sample size");
        if (reinterpret_cast<uintptr_t>(d_dst[i]) % 16 || dst_pitch[i] % 16)
            return jinc_fail(JINC_E_INVALID, "resize: device destination planes must be 16-byte aligned (base and pitch)");
        pl.src[i] = d_src[i];
        pl.dst[i] = d_dst[i];
        pl.src_pitch[i] = src_pitch[i] / sample_bytes;
        pl.dst_pitch[i] = dst_pitch[i] / sample_bytes;
    }
    return JINC_OK;
}

int dispatch(const jinc_table* t, int sample, const FrameSet& fr, int n_frames, int y_begin, int y_end, cudaStream_t stream,
             int* launches, int parts)
{
    y_begin = std::max(y_begin, 0);
    y_end = std::min(y_end, t->sc.dst_h);
    if (y_end <= y_begin || n_frames <= 0)
        return JINC_OK;
    int dummy = 0;
    if (!launches)
        launches = &dummy;
    switch (sample) {
    case 1: return launch_typed<uint8_t>(t, fr, n_frames, y_begin, y_end, stream, launches, parts);
    case 2: return launch_typed<uint16_t>(t, fr, n_frames, y_begin, y_end, stream, launches, parts);
    case 4: return launch_typed<float>(t, fr, n_frames, y_begin, y_end, stream, launches, parts);
    case JINC_SAMPLE_F16: return launch_typed<__half>(t, fr, n_frames, y_begin, y_end, stream, launches, parts);
    default: return jinc_fail(JINC_E_INVALID, "resize: sample_bytes must be 1, 2, 4 or JINC_SAMPLE_F16");
    }
}

} // namespace

size_t jinc_plane_ptrs_size() { return sizeof(PlanePtrs); }

void jinc_free_strip_plan(jinc_table* t)
{
    StripPlan& sp = t->strip_plan;
    cudaFree(sp.d_patches);
    cudaFree(sp.d_threads);
    cudaFree(sp.d_wdata);
    sp = StripPlan{};
}

// Host side of the plan.  The strips (up to four rectangles) are cut into patches: 64 outputs wide in the wide strips,
// 8 in the tall ones, as tall as the block has threads for.  In a wide strip a thread takes up to SPT outputs of one row
// that are px apart (one residue class of the row), in a tall strip up to SPT outputs of one column that are py apart;
// how they are accumulated is decided here, by the rules of strip_block.
struct StripPlanParams {
    int threads, spt;
    int px, py;   // phase period of the outputs along x and y
    int step;     // distance of the window origins of same-phase neighbours (both axes)
    unsigned smem_floats;
};

struct StripPlanHost {
    std::vector<StripPlanPatch> patches;
    std::vector<uint4> recs;
    std::vector<uint32_t> wlist; // sel << 31 | block, in packing order
    unsigned n_staged = 0;       // patches whose weight blocks fit in shared memory
    bool ok = false;
};

inline void build_strip_plan_host(const jinc_table* t, const Rect* rects, int n_rects, const StripPlanParams& pp, StripPlanHost& out)
{
    const int fs = t->sc.fs, fsp = (fs + 3) & ~3, wbf = fs * fsp;
    const int THREADS = pp.threads, SPT = pp.spt;
    const std::vector<int32_t>&start_x = t->h_start[0], &start_y = t->h_start[1], &rank_x = t->h_rank[0], &rank_y = t->h_rank[1];
    const bool have_classes = !t->h_border_block.empty();
    const int phase_stride = t->d_weights_p ? fsp : fs;
    const int n_rank_x = t->ax[0].n_rank;
    out = StripPlanHost{};
    out.recs.reserve((size_t)SPT * THREADS * 256);
    struct Meta {
        int x, y, sx, sy, wstride;
        uint32_t wkey; // sel << 31 | block; only meaningful when wstride != 0 (per-pixel weights: the border slot)
        bool perpix;   // a border pixel with its own resident weights
    };
    struct Item {
        int x[8], y[8], n;
    };
    std::vector<Meta> meta((size_t)SPT);
    std::vector<Item> items;
    std::vector<uint32_t> keys; // distinct weight blocks of the patch, in first-use order
    if (SPT > 8)
        return;
    // Ratios whose positions never repeat exactly have no class blocks: every border pixel keeps its own weights, stored so
    // that neighbouring pixels lie next to each other.  Their threads take pixels a quarter of a patch row apart (the
    // prologue path's mapping: the lanes of a warp are neighbouring pixels), not same-phase neighbours.
    const bool scatter = !have_classes && t->bgeom.total > 0;
    if (scatter && !t->d_border_w)
        return; // border weights over the residency budget are rebuilt per tap from the LUT: the prologue path
    for (int ri = 0; ri < n_rects; ++ri) {
        const Rect rc = rects[ri];
        const int w = rc.x1 - rc.x0, h = rc.y1 - rc.y0;
        if (w <= 0 || h <= 0)
            continue;
        const bool rows = w >= h; // top/bottom strips are wide, left/right strips are tall
        const int pw = rows ? 64 : 8;
        for (int ox0 = rc.x0; ox0 < rc.x1; ox0 += pw) {
            const int nx = std::min(pw, rc.x1 - ox0);
            // patch height: as many rows as the block has threads for
            int ph;
            if (rows && scatter) {
                ph = std::max(1, THREADS / ((nx + SPT - 1) / SPT));
            } else if (!rows && scatter) {
                ph = std::max(1, THREADS / nx) * SPT;
            } else if (rows) {
                int per_row = 0;
                for (int p = 0; p < pp.px; ++p) {
                    int cnt = 0;
                    for (int x = ox0; x < ox0 + nx; ++x)
                        cnt += (x % pp.px) == p;
                    per_row += (cnt + SPT - 1) / SPT;
                }
                ph = std::max(1, THREADS / std::max(per_row, 1));
                if (per_row > THREADS)
                    return; // cannot happen for 64-wide patches
            } else {
                const int m = THREADS / (nx * pp.py); // groups of SPT * py rows
                if (m < 1)
                    return;
                ph = m * SPT * pp.py;
            }
            for (int oy0 = rc.y0; oy0 < rc.y1; oy0 += ph) {
                const int ny = std::min(ph, rc.y1 - oy0);
                const int sx_lo = start_x[ox0], sy_lo = start_y[oy0];
                const int fw = start_x[ox0 + nx - 1] + fs - sx_lo, fh = start_y[oy0 + ny - 1] + fs - sy_lo;
                if ((long long)fw * fh > (long long)pp.smem_floats)
                    return; // footprints of the planned kernel families always fit; otherwise no plan at all
                // the work items of the patch
                items.clear();
                if (rows && scatter) {
                    const int dx = (nx + SPT - 1) / SPT;
                    for (int y = oy0; y < oy0 + ny; ++y)
                        for (int tx = 0; tx < dx; ++tx) {
                            Item it{};
                            for (int k = 0; k < SPT && tx + k * dx < nx; ++k) {
                                it.x[it.n] = ox0 + tx + k * dx;
                                it.y[it.n] = y;
                                ++it.n;
                            }
                            items.push_back(it);
                        }
                } else if (rows) {
                    for (int y = oy0; y < oy0 + ny; ++y)
                        for (int p = 0; p < pp.px; ++p) {
                            Item it{};
                            for (int x = ox0; x < ox0 + nx; ++x) {
                                if (x % pp.px != p)
                                    continue;
                                it.x[it.n] = x;
                                it.y[it.n] = y;
                                if (++it.n == SPT) {
                                    items.push_back(it);
                                    it.n = 0;
                                }
                            }
                            if (it.n)
                                items.push_back(it);
                        }
                } else if (fs > 9 || scatter) {
                    // wide windows never run down a column (see below): a thread's samples need not be neighbours, so
                    // neighbouring lanes take neighbouring rows (window rows `step` apart: different banks) and a thread's
                    // samples lie a quarter of the patch apart -- the prologue path's mapping
                    const int tyn = std::max(1, THREADS / nx), dy = (ny + SPT - 1) / SPT;
                    for (int ty = 0; ty < std::min(tyn, dy); ++ty)
                        for (int x = ox0; x < ox0 + nx; ++x) {
                            Item it{};
                            for (int k = 0; k < SPT; ++k) {
                                const int y = oy0 + ty + k * dy;
                                if (y < oy0 + ny) {
                                    it.x[it.n] = x;
                                    it.y[it.n] = y;
                                    ++it.n;
                                }
                            }
                            if (it.n)
                                items.push_back(it);
                        }
                } else {
                    // groups of one residue class down a column; neighbouring lanes take neighbouring columns (their windows
                    // start in the same source rows: no bank conflicts between them)
                    for (int g = 0;; ++g) {
                        bool any = false;
                        for (int p = 0; p < pp.py; ++p)
                            for (int x = ox0; x < ox0 + nx; ++x) {
                                Item it{};
                                int seen = 0;
                                for (int y = oy0; y < oy0 + ny; ++y) {
                                    if (y % pp.py != p)
                                        continue;
                                    if (seen / SPT == g) {
                                        it.x[it.n] = x;
                                        it.y[it.n] = y;
                                        ++it.n;
                                    }
                                    ++seen;
                                }
                                if (it.n) {
                                    items.push_back(it);
                                    any = true;
                                }
                            }
                        if (!any)
                            break;
                    }
                }
                if ((int)items.size() > THREADS)
                    return;
                StripPlanPatch pd{};
                pd.sx_lo = sx_lo;
                pd.sy_lo = sy_lo;
                pd.fw = fw;
                pd.fh = fh;
                pd.magic = 0xFFFFFFFFu / (unsigned)fw + 1u;
                pd.row_stride = fw;
                pd.sub = 0;
                pd.deint = 0;
                pd.ring = 0;
                const size_t rec0 = out.recs.size();
                out.recs.resize(rec0 + (size_t)SPT * THREADS, make_uint4(0, 0, 0, 0));
                uint4* prec = out.recs.data() + rec0;
                keys.clear();
                size_t last_key = 0;
                for (size_t tid = 0; tid < items.size(); ++tid) {
                    const Item& it = items[tid];
                    const unsigned live = (1u << it.n) - 1u;
                    for (int k = 0; k < it.n; ++k) {
                        Meta& m = meta[k];
                        m.x = it.x[k];
                        m.y = it.y[k];
                        m.sx = start_x[m.x];
                        m.sy = start_y[m.y];
                        const int rx = rank_x[m.x], ry = rank_y[m.y];
                        if (rx >= 0 && ry >= 0) {
                            m.wkey = (uint32_t)(ry * n_rank_x + rx);
                            m.wstride = phase_stride;
                        } else if (have_classes) {
                            m.wkey = 0x80000000u | (uint32_t)t->h_border_block[(size_t)jinc_border_slot(t->bgeom, m.x, m.y)];
                            m.wstride = fsp;
                        } else {
                            m.wkey = scatter ? (uint32_t)jinc_border_slot(t->bgeom, m.x, m.y) : 0u;
                            m.wstride = 0;
                        }
                        m.perpix = scatter && !(rx >= 0 && ry >= 0);
                    }
                    bool same = true, vec = true, perpix = true;
                    for (int k = 0; k < SPT; ++k) {
                        if (k >= it.n)
                            meta[k] = meta[0]; // computed, not stored
                        same = same && meta[k].wstride == meta[0].wstride && (meta[k].wstride == 0 || meta[k].wkey == meta[0].wkey);
                        vec = vec && meta[k].wstride != 0 && (meta[k].wstride & 3) == 0 && meta[k].wstride == meta[0].wstride;
                        perpix = perpix && meta[k].perpix;
                    }
                    unsigned kind = perpix ? JINC_SK_PER_PIXEL : JINC_SK_PER_SAMPLE;
                    if (vec) {
                        kind = same ? JINC_SK_FUSED_SHARED : JINC_SK_FUSED_SEP;
                        if (same && it.n == SPT) {
                            bool run = true;
                            for (int k = 1; k < SPT; ++k)
                                run = run && (rows ? (meta[k].sy == meta[0].sy && meta[k].sx == meta[0].sx + k * pp.step)
                                                   : (meta[k].sx == meta[0].sx && meta[k].sy == meta[0].sy + k * pp.step));
                            if (run && rows)
                                kind = JINC_SK_RUN_ROWS;
                            else if (run && fs <= 9) // wide windows down a column: one weight row for four source rows reads less
                                kind = JINC_SK_RUN_COLS;
                        }
                    }
                    for (int k = 0; k < SPT; ++k) {
                        const Meta& m = meta[k];
                        uint32_t slot = kind == JINC_SK_PER_PIXEL ? m.wkey : 0u;
                        if (kind != JINC_SK_PER_SAMPLE && kind != JINC_SK_PER_PIXEL) {
                            size_t j = last_key < keys.size() && keys[last_key] == m.wkey ? last_key : 0; // neighbours share blocks
                            while (j < keys.size() && keys[j] != m.wkey)
                                ++j;
                            last_key = j;
                            if (j == keys.size())
                                keys.push_back(m.wkey);
                            slot = (uint32_t)j * (uint32_t)wbf;
                        }
                        prec[(size_t)k * THREADS + tid] = make_uint4((uint32_t)m.x | ((uint32_t)m.y << 16),
                                                                     (uint32_t)((m.sy - sy_lo) * fw + (m.sx - sx_lo)), slot, k == 0 ? (kind | (live << 8)) : 0u);
                    }
                }
                // a patch of row runs whose windows all start on a multiple of spt * step is staged de-interleaved
                if (pp.step > 1 && !items.empty()) {
                    const int d = SPT * pp.step, sub = plan_deint_sub(pp.step, SPT, fs), rs = d * sub;
                    bool pure = fw <= rs;
                    for (size_t tid = 0; tid < items.size() && pure; ++tid) {
                        const uint4& r0 = prec[tid];
                        pure = (r0.w & 0xffu) == JINC_SK_RUN_ROWS && ((int)r0.y % fw) % d == 0;
                    }
                    if (pure && (long long)rs * fh <= (long long)pp.smem_floats) {
                        pd.deint = 1;
                        pd.sub = sub;
                        pd.row_stride = rs;
                        for (size_t tid = 0; tid < items.size(); ++tid) {
                            uint4& r0 = prec[tid];
                            const int row = (int)r0.y / fw, col = (int)r0.y % fw;
                            r0.y = (uint32_t)(row * rs + col / d);
                        }
                    }
                }
                pd.tile_floats = ((unsigned)(pd.row_stride * fh) + 3u) & ~3u;
                const bool staged = (unsigned long long)pd.tile_floats + (unsigned long long)keys.size() * wbf <= pp.smem_floats;
                pd.n_wb = staged ? (int32_t)keys.size() : -1;
                pd.wdata_off = (uint32_t)(out.wlist.size() * (size_t)wbf);
                if (staged) {
                    out.wlist.insert(out.wlist.end(), keys.begin(), keys.end());
                } else {
                    // too many blocks for shared memory: the records name the table's own blocks (shared by every patch, so
                    // they stay in the caches) instead of slots of a packed copy
                    for (int k = 0; k < SPT; ++k)
                        for (size_t tid = 0; tid < items.size(); ++tid) {
                            uint4& rk = prec[(size_t)k * THREADS + tid];
                            if ((prec[tid].w & 0xffu) != JINC_SK_PER_SAMPLE && (prec[tid].w & 0xffu) != JINC_SK_PER_PIXEL)
                                rk.z = keys[rk.z / (uint32_t)wbf];
                        }
                }
                // Wide windows whose blocks stay in the table: when every half-warp of the patch is sixteen row runs with one
                // weight block (a 64-wide patch row), the block's rows are streamed through a shared-memory ring, several
                // rows in flight (plan_run_rows_ring), instead of being loaded a row ahead into registers.
                if (!staged && fs > 9 && items.size() % 16 == 0 && !items.empty()) {
                    bool uniform = true;
                    for (size_t h0 = 0; h0 < items.size() && uniform; h0 += 16)
                        for (size_t tid = h0; tid < h0 + 16 && uniform; ++tid)
                            uniform = (prec[tid].w & 0xffu) == JINC_SK_RUN_ROWS && prec[tid].z == prec[h0].z;
                    const unsigned long long ring_floats = (unsigned long long)(THREADS / 16) * JINC_PLAN_RING_DEPTH * fsp;
                    if (uniform && pd.tile_floats + ring_floats <= pp.smem_floats)
                        pd.ring = (int32_t)pd.tile_floats;
                }
                out.n_staged += staged ? 1u : 0u;
                out.patches.push_back(pd);
            }
        }
    }
    out.ok = !out.patches.empty();
}

// whole-frame launches: the strip blocks of a table with a plan run from it (its own patches)
bool jinc_rs::attach_strip_plan(const jinc_table* t, StripArgs& st, int threads, int spt)
{
    const StripPlan& sp = t->strip_plan;
    if (!sp.ok || sp.threads != threads || sp.spt != spt)
        return false;
    st.plan_patches = sp.d_patches;
    st.plan_threads = sp.d_threads;
    st.plan_wdata = sp.d_wdata;
    st.plan_px = sp.px;
    st.plan_py = sp.py;
    st.blocks_per_plane = sp.n_patches;
    st.blocks_per_plane_magic = div_magic(sp.n_patches);
    return true;
}

// Strip plan of the exact-2x and chunked-cells tables (the upscale ratios): see StripPlan in jinc_internal.h.  Tables
// without a plan (other kernel families, planes wider than the 16-bit coordinates of a record) keep the prologue path.
int jinc_build_strip_plan(jinc_table* t)
{
    StripPlan& sp = t->strip_plan;
    sp = StripPlan{};
    const char* off = getenv("JINCRESIZE_B200_STRIP_PLAN");
    if (off && off[0] == '0')
        return JINC_OK;
    if (t->sc.dst_w > 65535 || t->sc.dst_h > 65535)
        return JINC_OK;
    const int fs = t->sc.fs, wbf = fs * ((fs + 3) & ~3);
    StripPlanParams pp{};
    if (t->fast_path == JINC_PATH_UP2X && up2x_supported(fs)) {
        pp = StripPlanParams{UP_THREADS, UP_STRIP_SPT, 2, 2, 1, (unsigned)(up2x_smem_bytes(fs) / sizeof(float))};
    } else if (t->fast_path == JINC_PATH_CELLS && t->cells.ok && jinc_cells_instantiated(t->cells.Q, fs)) {
        const int q = t->cells.Q, warps = jinc_cells_warps(q, fs);
        const int d = q * JINC_CELLS_NX, fwc = jinc_cells_footprint(q, fs, JINC_CELLS_NX, 32), fhc = jinc_cells_footprint(q, fs, JINC_CELLS_NY, warps);
        const size_t smem = (size_t)fhc * (size_t)(d * ((fwc + d - 1) / d)) * sizeof(float); // CellsGeom<FS, Q>::SMEM
        pp = StripPlanParams{32 * warps, CL_STRIP_SPT, t->cells.ax[0].P, t->cells.ax[1].P, q, (unsigned)(smem / sizeof(float))};
    } else if (t->fast_path == JINC_PATH_DOWN_INT && down_supported(t)) {
        // DownGeom<T, FS, Q, 8, 2> of the integer sample types (128 threads per block; float and half planes run 64-thread
        // blocks and keep the prologue path): a lower bound of its shared memory (the row padding left out)
        const int q = t->down.qx;
        const int nkw1 = (q & 1) ? (fs + 2) / 2 : ((fs + 1) & ~1) / 2;
        const int nrowp = (q * (DN_TH - 1) + 2 * nkw1 + 1) / 2, mt = (fs + q - 1) / q, d = q * 8;
        const int ncol = q * (DN_TW - 1) + q * (mt - 1) + q, sub = (ncol + d - 1) / d;
        pp = StripPlanParams{128, DN_STRIP_SPT, 1, 1, q, (unsigned)((size_t)nrowp * d * sub)};
    } else {
        return JINC_OK;
    }
    const int W = t->sc.dst_w, H = t->sc.dst_h;
    // the whole-frame strips around the interior, as launch_typed cuts them
    const Rect rects[4] = {Rect{0, 0, W, t->iy0}, Rect{0, t->iy1, W, H}, Rect{0, t->iy0, t->ix0, t->iy1}, Rect{t->ix1, t->iy0, W, t->iy1}};
    StripPlanHost h;
    const auto t_begin = std::chrono::steady_clock::now();
    build_strip_plan_host(t, rects, 4, pp, h);
    if (!h.ok)
        return JINC_OK;
    const auto t_host = std::chrono::steady_clock::now();
    cudaStream_t st = t->ctx->stream;
    JINC_CUDA(cudaSetDevice(t->ctx->device));
    JINC_CUDA(cudaMalloc(reinterpret_cast<void**>(&sp.d_patches), h.patches.size() * sizeof(StripPlanPatch)));
    JINC_CUDA(cudaMalloc(reinterpret_cast<void**>(&sp.d_threads), h.recs.size() * sizeof(uint4)));
    JINC_CUDA(cudaMalloc(reinterpret_cast<void**>(&sp.d_wdata), (h.wlist.size() + 1) * wbf * sizeof(float)));
    JINC_CUDA(cudaMemcpyAsync(sp.d_patches, h.patches.data(), h.patches.size() * sizeof(StripPlanPatch), cudaMemcpyHostToDevice, st));
    JINC_CUDA(cudaMemcpyAsync(sp.d_threads, h.recs.data(), h.recs.size() * sizeof(uint4), cudaMemcpyHostToDevice, st));
    if (!h.wlist.empty()) {
        uint32_t* d_list = nullptr;
        JINC_CUDA(cudaMalloc(reinterpret_cast<void**>(&d_list), h.wlist.size() * sizeof(uint32_t)));
        cudaError_t e = cudaMemcpyAsync(d_list, h.wlist.data(), h.wlist.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) {
            e = jinc_gather_blocks(sp.d_wdata, d_list, (unsigned)h.wlist.size(), t->d_weights_p ? t->d_weights_p : t->d_weights, t->d_border_wb,
                                   wbf, st);
        }
        if (e == cudaSuccess)
            e = cudaStreamSynchronize(st); // the host vectors and the list are temporaries
        cudaFree(d_list);
        if (e != cudaSuccess)
            return jinc_fail(JINC_E_CUDA, "strip plan: %s", cudaGetErrorString(e));
    } else {
        JINC_CUDA(cudaStreamSynchronize(st));
    }
    if (const char* e = getenv("JINCRESIZE_B200_PLAN_TIMING"); e && e[0] == '1') {
        const auto t_end = std::chrono::steady_clock::now();
        fprintf(stderr, "strip plan %dx%d: %zu patches (%u staged), %zu packed blocks; host %.2f ms, upload %.2f ms\n", W, H, h.patches.size(),
                h.n_staged, h.wlist.size(), std::chrono::duration<double, std::milli>(t_host - t_begin).count(),
                std::chrono::duration<double, std::milli>(t_end - t_host).count());
    }
    sp.threads = pp.threads;
    sp.spt = pp.spt;
    sp.px = pp.px;
    sp.py = pp.py;
    sp.n_patches = (unsigned)h.patches.size();
    sp.n_staged = h.n_staged;
    sp.ok = true;
    return JINC_OK;
}

int jinc_pack_plane_ptrs(void* out, int sample, int n_planes, const void* const* d_src, const ptrdiff_t* src_pitch,
                         void* const* d_dst, const ptrdiff_t* dst_pitch)
{
    if (n_planes < 1 || n_planes > JINC_MAX_PLANES)
        return jinc_fail(JINC_E_INVALID, "resize: n_planes must be 1..4");
    return check_and_fill(*static_cast<PlanePtrs*>(out), sample, n_planes, d_src, src_pitch, d_dst, dst_pitch);
}

int jinc_launch_resize_planes(jinc_ctx* ctx, const jinc_table* t, int sample, float peak, int n_planes,
                              const void* const* d_src, const ptrdiff_t* src_pitch, void* const* d_dst,
                              const ptrdiff_t* dst_pitch, int y_begin, int y_end, cudaStream_t stream, int* launches,
                              int parts)
{
    (void)ctx;
    FrameSet fr;
    memset(&fr, 0, sizeof(fr));
    if (int rc = jinc_pack_plane_ptrs(&fr.one, sample, n_planes, d_src, src_pitch, d_dst, dst_pitch))
        return rc;
    fr.frames = nullptr;
    fr.n_planes = n_planes;
    fr.peak = peak;
    return dispatch(t, sample, fr, 1, y_begin, y_end, stream, launches, parts);
}

int jinc_launch_resize_batch(jinc_ctx* ctx, const jinc_table* t, int sample, float peak, int n_planes,
                             const void* d_frame_ptrs, int n_frames, cudaStream_t stream, int* launches, int parts)
{
    (void)ctx;
    FrameSet fr;
    memset(&fr, 0, sizeof(fr));
    fr.frames = static_cast<const PlanePtrs*>(d_frame_ptrs);
    fr.n_planes = n_planes;
    fr.peak = peak;
    return dispatch(t, sample, fr, n_frames, 0, t->sc.dst_h, stream, launches, parts);
}

int jinc_launch_resize(jinc_ctx* ctx, const jinc_table* t, int sample, float peak, const void* d_src,
                       ptrdiff_t src_pitch, void* d_dst, ptrdiff_t dst_pitch, int y_begin, int y_end, cudaStream_t stream,
                       int* launches)
{
    return jinc_launch_resize_planes(ctx, t, sample, peak, 1, &d_src, &src_pitch, &d_dst, &dst_pitch, y_begin, y_end,
                                     stream, launches, JINC_PART_ALL);
}

// Probe words of a freshly uploaded source buffer, read back so the host can compare them with the caller's memory
// (stale-registration check of the frame pipeline; no pixel is computed here).
__global__ void probe_kernel(const uint32_t* __restrict__ buf, uint32_t n_words, uint32_t seed, uint32_t* __restrict__ out)
{
    out[threadIdx.x] = buf[jinc_probe_index(seed, threadIdx.x, n_words)];
}

int jinc_launch_probe(const void* d_buf, uint32_t n_words, uint32_t seed, uint32_t* d_out, cudaStream_t stream)
{
    probe_kernel<<<1, JINC_PROBE_WORDS, 0, stream>>>(static_cast<const uint32_t*>(d_buf), n_words, seed, d_out);
    JINC_CUDA(cudaGetLastError());
    return JINC_OK;
}

int jinc_debug_pixel_weights(const jinc_table* t, int x, int y, float* out)
{
    JINC_CUDA(cudaSetDevice(t->ctx->device));
    StripArgs a;
    fill_strip_args(t, a);
    const size_t n = (size_t)t->sc.fs * t->sc.fs;
    float* d = nullptr;
    JINC_CUDA(cudaMalloc(&d, n * sizeof(float)));
    pixel_weights_kernel<<<1, 128, 0, t->ctx->stream>>>(a, x, y, d);
    cudaError_t e = cudaMemcpyAsync(out, d, n * sizeof(float), cudaMemcpyDeviceToHost, t->ctx->stream);
    if (e == cudaSuccess)
        e = cudaStreamSynchronize(t->ctx->stream);
    cudaFree(d);
    if (e != cudaSuccess)
        return jinc_fail(JINC_E_CUDA, "pixel_weights: %s", cudaGetErrorString(e));
    return JINC_OK;
}

extern "C" int jinc_resize_plane_device(jinc_ctx* ctx, const jinc_table* t, int sample_bytes, float peak, const void* d_src,
                                        ptrdiff_t src_pitch, void* d_dst, ptrdiff_t dst_pitch, void* stream)
{
    if (!ctx || !t)
        return jinc_fail(JINC_E_INVALID, "jinc_resize_plane_device: null argument");
    JINC_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    return jinc_launch_resize(ctx, t, sample_bytes, peak, d_src, src_pitch, d_dst, dst_pitch, 0, t->sc.dst_h, st, nullptr);
}

extern "C" int jinc_resize_planes_device(jinc_ctx* ctx, const jinc_table* t, int sample_bytes, float peak, int n_planes,
                                         const void* d_src, ptrdiff_t src_pitch, ptrdiff_t src_plane_stride, void* d_dst,
                                         ptrdiff_t dst_pitch, ptrdiff_t dst_plane_stride, void* stream)
{
    if (!ctx || !t || !d_src || !d_dst)
        return jinc_fail(JINC_E_INVALID, "jinc_resize_planes_device: null argument");
    if (n_planes < 1)
        return jinc_fail(JINC_E_INVALID, "jinc_resize_planes_device: n_planes must be at least 1");
    if (!jinc_sample_valid(sample_bytes))
        return jinc_fail(JINC_E_INVALID, "jinc_resize_planes_device: sample_bytes must be 1, 2, 4 or JINC_SAMPLE_F16");
    if (reinterpret_cast<uintptr_t>(d_dst) % 16 || dst_pitch % 16 || (n_planes > 1 && dst_plane_stride % 16))
        return jinc_fail(JINC_E_INVALID, "jinc_resize_planes_device: device destination planes must be 16-byte aligned (base, pitch and "
                                         "plane stride)");
    JINC_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    // records of up to four planes each (one block then serves the patch in all of them), grid.y = record
    int per = JINC_MAX_PLANES;
    while (n_planes % per)
        --per;
    const int n_rec = n_planes / per;
    const size_t rec = sizeof(PlanePtrs);
    constexpr int kMaxRecords = 65535; // grid.y limit
    std::vector<unsigned char> host;
    for (int r0 = 0; r0 < n_rec; r0 += kMaxRecords) {
        const int nr = std::min(kMaxRecords, n_rec - r0);
        host.assign(rec * nr, 0);
        for (int r = 0; r < nr; ++r) {
            const void* src[JINC_MAX_PLANES];
            void* dst[JINC_MAX_PLANES];
            ptrdiff_t sp[JINC_MAX_PLANES], dp[JINC_MAX_PLANES];
            for (int k = 0; k < per; ++k) {
                const long long i = (long long)(r0 + r) * per + k;
                src[k] = static_cast<const unsigned char*>(d_src) + i * src_plane_stride;
                dst[k] = static_cast<unsigned char*>(d_dst) + i * dst_plane_stride;
                sp[k] = src_pitch;
                dp[k] = dst_pitch;
            }
            if (int rc = jinc_pack_plane_ptrs(host.data() + rec * r, sample_bytes, per, src, sp, dst, dp))
                return rc;
        }
        const int rc = jinc_ring_launch(ctx, host.data(), host.size(), st, [&](const void* dbuf) {
            return jinc_launch_resize_batch(ctx, t, sample_bytes, peak, per, dbuf, nr, st, nullptr, JINC_PART_ALL);
        });
        if (rc != JINC_OK)
            return rc;
    }
    return JINC_OK;
}

extern "C" int jinc_table_strip_plan(const jinc_table* t, int* staged)
{
    if (staged)
        *staged = t && t->strip_plan.ok ? (int)t->strip_plan.n_staged : 0;
    return t && t->strip_plan.ok ? (int)t->strip_plan.n_patches : 0;
}

extern "C" int jinc_table_launches_per_plane(const jinc_table* t)
{
    return t ? 1 : 0; // interior tiles and border strips of all planes sharing the table go out in one launch
}

