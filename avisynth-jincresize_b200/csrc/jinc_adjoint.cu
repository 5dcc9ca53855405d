// jinc_adjoint.cu -- the adjoint (transpose) of the resampler: float32 output gradients -> float32 source gradients.
//
// The resampler is a fixed linear map, out = A * src, with the weights of the table (jinc_table_pixel_weights).  The
// adjoint of one output-gradient plane g is grad_src[sy][sx] = sum of w_{x,y}[sy - start_y[y]][sx - start_x[x]] * g[y][x]
// over the outputs (x, y) whose window covers (sx, sy), accumulated in ONE canonical order: output rows y ascending, in a
// row x ascending, acc = fmaf(w, g, acc) from 0.  Both kernels below use that order, so a source sample's bits do not
// depend on which kernel, tile or batch position computed it (DESIGN.md 4.8).
//
// The outputs whose window covers source column sx form one contiguous range: start_x is non-decreasing (the positions
// are accumulated with positive float steps and the origin is built from monotone functions, jinc_table.cu).  So the
// range is [lower_bound(start_x, sx - fs + 1), lower_bound(start_x, sx + 1)), found by binary search on the table's device
// array; the table build is unchanged.
//
//   adjoint_general   any table.  A block takes 32 x 8 source samples, finds each column's and row's covering range once,
//                     stages those outputs' start and rank and the g rectangle they span in shared memory (the rectangle is
//                     read through L1 when it does not fit), and a thread sums its sample over the covering outputs.  The
//                     weights come from the same four places the forward strip role reads (strip_sample): the shared phase
//                     block, the border class block, the resident per-pixel border block, or the LUT rebuilt from pos.
//   adjoint_up2x      exact-2x tables, the source samples all of whose covering outputs are interior cells of the table's
//                     Up2xPlan.  The adjoint of the polyphase 2x upscale is four stride-1 correlations of the phase
//                     sub-lattices of g with the flipped phase blocks: sample u of a row receives cell c = u - j with tap j
//                     of phase px = 0 and tap j - ox1 of phase px = 1.  The g tile is staged once per block as float4
//                     {g[2c], g[2c+2], g[2c+1], g[2c+3]} per cell, so one LDS.128 feeds both phases of two neighbouring
//                     samples (cells c and c + 1 at the same tap) and one packed FFMA2 updates both samples with a weight
//                     from the constant bank.  A thread owns 4 neighbouring columns x RY rows.
// The 2x kernel runs first; the general kernel then takes the source samples around its rectangle in a second launch on
// the same stream.
#include <climits>

#include "jinc_resample.cuh"

using namespace jinc_rs;

namespace {

struct AdjPlanes {
    const float* g; // output-gradient planes, pitch / plane stride in floats
    long long g_pitch, g_stride;
    float* out; // source-gradient planes
    long long o_pitch, o_stride;
    int n_planes;
};

// first index in [0, n) whose value is >= v (n when none); a is non-decreasing
__device__ __forceinline__ int lower_bound_i32(const int32_t* __restrict__ a, int n, int v)
{
    int lo = 0, hi = n;
    while (lo < hi) {
        const int m = (lo + hi) >> 1;
        if (__ldg(a + m) < v)
            lo = m + 1;
        else
            hi = m;
    }
    return lo;
}

// ------------------------------------------------------------------------------------------ general kernel

constexpr int AG_TW = 32, AG_TH = 8, AG_THREADS = AG_TW * AG_TH;
constexpr int AG_MAX_N = 512;                 // outputs per axis whose start and rank a block stages
constexpr int AG_G_FLOATS = 8192;             // g rectangle staged in shared memory (32 KB)

struct AdjGeneralArgs {
    StripArgs st; // table arrays and geometry (no strips)
    AdjPlanes pl;
    int dst_w, dst_h;
    Rect rect[4];             // source rectangles to produce
    unsigned tile_begin[5];   // prefix sums of the tiles per rectangle
    unsigned tiles_x[4];
};

// Weight of output (x, y) at tap (ly, lx), source sample (sx, sy) = (start_x[x] + lx, start_y[y] + ly): the value the
// forward strip role multiplies (strip_sample), taken from the same storage in the same order of preference.
__device__ __forceinline__ float adj_weight(const StripArgs& a, int x, int y, int rx, int ry, int lx, int ly, int sx, int sy)
{
    const int fs = a.fs;
    if (rx >= 0 && ry >= 0)
        return __ldg(a.weights + (unsigned)(ry * a.n_rank_x + rx) * (unsigned)(fs * fs) + (unsigned)(ly * fs + lx));
    const long long slot = jinc_border_slot(a.bg, x, y);
    if (a.border_block) {
        const int fsp = (fs + 3) & ~3;
        return __ldg(a.border_wb + (size_t)a.border_block[slot] * (unsigned)(fs * fsp) + (unsigned)(ly * fsp + lx));
    }
    if (a.border_w)
        return __ldg(a.border_w + (size_t)(slot >> 5) * (size_t)(fs * fs * 32) + (unsigned)(ly * fs + lx) * 32u + (unsigned)(slot & 31));
    const double dy2 = jinc_tap_dist2(a.pos_y[y], a.src_h, sy, a.step_y);
    const double dx2 = jinc_tap_dist2(a.pos_x[x], a.src_w, sx, a.step_x);
    return __fdiv_rn(jinc_lut_weight(a.lut, __dadd_rn(dx2, dy2), a.radius2, a.idx_scale), a.border_sum[slot]);
}

__global__ void __launch_bounds__(AG_THREADS) adjoint_general(const __grid_constant__ AdjGeneralArgs a)
{
    __shared__ int s_xlo[AG_TW], s_xhi[AG_TW], s_ylo[AG_TH], s_yhi[AG_TH];
    __shared__ int32_t s_sx[AG_MAX_N], s_rx[AG_MAX_N], s_sy[AG_MAX_N], s_ry[AG_MAX_N];
    extern __shared__ float s_g[]; // [ny][nx] when it fits

    const unsigned b = blockIdx.x;
    int r = 0;
    while (r < 3 && b >= a.tile_begin[r + 1])
        ++r;
    const Rect rc = a.rect[r];
    const unsigned tb = b - a.tile_begin[r], tyi = tb / a.tiles_x[r], txi = tb - tyi * a.tiles_x[r];
    const int x0 = rc.x0 + (int)txi * AG_TW, y0 = rc.y0 + (int)tyi * AG_TH;
    const int tw = min(AG_TW, rc.x1 - x0), th = min(AG_TH, rc.y1 - y0);
    const StripArgs& st = a.st;
    const int fs = st.fs;
    const int tid = threadIdx.x;
    if (tid < tw) {
        s_xlo[tid] = lower_bound_i32(st.start_x, a.dst_w, x0 + tid - fs + 1);
        s_xhi[tid] = lower_bound_i32(st.start_x, a.dst_w, x0 + tid + 1);
    } else if (tid >= 32 && tid - 32 < th) {
        s_ylo[tid - 32] = lower_bound_i32(st.start_y, a.dst_h, y0 + tid - 32 - fs + 1);
        s_yhi[tid - 32] = lower_bound_i32(st.start_y, a.dst_h, y0 + tid - 32 + 1);
    }
    __syncthreads();
    const int X0 = s_xlo[0], Y0 = s_ylo[0];
    const int nx = max(s_xhi[tw - 1] - X0, 0), ny = max(s_yhi[th - 1] - Y0, 0);
    const bool stage_axes = nx <= AG_MAX_N && ny <= AG_MAX_N; // block-uniform
    if (stage_axes) {
        for (int i = tid; i < nx; i += AG_THREADS) {
            s_sx[i] = __ldg(st.start_x + X0 + i);
            s_rx[i] = __ldg(st.rank_x + X0 + i);
        }
        for (int i = tid; i < ny; i += AG_THREADS) {
            s_sy[i] = __ldg(st.start_y + Y0 + i);
            s_ry[i] = __ldg(st.rank_y + Y0 + i);
        }
    }
    const bool stage_g = nx * ny <= AG_G_FLOATS; // block-uniform (nx, ny <= dst size)
    const int txl = tid % AG_TW, tyl = tid / AG_TW;
    const int sx = x0 + txl, sy = y0 + tyl;
    const bool live = txl < tw && tyl < th;
    __syncthreads();
    const int xl = live ? s_xlo[txl] : 0, xh = live ? s_xhi[txl] : 0;
    const int yl = live ? s_ylo[tyl] : 0, yh = live ? s_yhi[tyl] : 0;

    for (int plane = blockIdx.y; plane < a.pl.n_planes; plane += gridDim.y) {
        const float* __restrict__ g = a.pl.g + (long long)plane * a.pl.g_stride;
        if (stage_g) {
            __syncthreads(); // the previous plane's rectangle is no longer read
            for (int e = tid; e < nx * ny; e += AG_THREADS) {
                const int row = e / nx, col = e - row * nx;
                s_g[e] = __ldg(g + (long long)(Y0 + row) * a.pl.g_pitch + X0 + col);
            }
            __syncthreads();
        }
        if (!live)
            continue;
        float acc = 0.f;
        for (int y = yl; y < yh; ++y) {
            const int j = y - Y0;
            const int ly = sy - (stage_axes ? s_sy[j] : __ldg(st.start_y + y));
            const int ry = stage_axes ? s_ry[j] : __ldg(st.rank_y + y);
            const float* __restrict__ grow = stage_g ? s_g + j * nx - X0 : g + (long long)y * a.pl.g_pitch;
            for (int x = xl; x < xh; ++x) {
                const int i = x - X0;
                const int lx = sx - (stage_axes ? s_sx[i] : __ldg(st.start_x + x));
                const int rx = stage_axes ? s_rx[i] : __ldg(st.rank_x + x);
                const float gv = stage_g ? grow[x] : __ldg(grow + x);
                acc = fmaf(adj_weight(st, x, y, rx, ry, lx, ly, sx, sy), gv, acc);
            }
        }
        a.pl.out[(long long)plane * a.pl.o_stride + (long long)sy * a.pl.o_pitch + sx] = acc;
    }
}

// ------------------------------------------------------------------------------------------ exact-2x kernel

constexpr int AU_TX = 4; // source columns per thread

template <int FS>
struct AdjUpGeom {
    static constexpr int WARPS = FS <= 9 ? 4 : 8;
    static constexpr int THREADS = 32 * WARPS;
    static constexpr int RY = FS <= 9 ? 4 : 2;      // source rows per thread
    static constexpr int TW = 32 * AU_TX;           // 128 source columns per tile
    static constexpr int TH = WARPS * RY;           // 16 source rows per tile
    static constexpr int NC = TW + FS + 3;          // cells per staged g row (4 * lane + m, m < FS + 3)
    static constexpr int NCP = (NC + 3) & ~3;
    static constexpr int SUB = NCP / 4;             // cells are de-interleaved by (c & 3): conflict-free LDS.128
    static constexpr int NR = 2 * (TH + FS);        // staged g rows: both phase rows of TH + FS - 1 + oy1 cell rows
    static constexpr size_t SMEM = (size_t)NR * NCP * sizeof(float4);
};

struct AdjUpArgs {
    AdjPlanes pl;
    int dst_w, dst_h;
    int x0, y0, sx0, sy0; // Up2xPlan: output origin of cell (0,0) and its window origin
    int ux0, ux1, uy0, uy1; // source rectangle this kernel produces
    int tiles_x, tiles;
};

template <int FS, int OX1, int OY1>
__global__ void __launch_bounds__(AdjUpGeom<FS>::THREADS, 1)
    adjoint_up2x(const __grid_constant__ AdjUpArgs a, const __grid_constant__ UpWeights<FS> W)
{
    using G = AdjUpGeom<FS>;
    constexpr int NSEG = FS + 2 + OX1; // cells a thread reads per g row: m = 2p - j + FS - 1 + OX1
    constexpr int NK = G::RY + FS - 1 + OY1; // g cell rows a thread's RY source rows read
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float4* tile = reinterpret_cast<float4*>(smem_raw); // [NR][4][SUB]

    const int tyi = blockIdx.x / a.tiles_x, txi = blockIdx.x - tyi * a.tiles_x;
    const int ts = a.ux0 + txi * G::TW, tv = a.uy0 + tyi * G::TH; // first source column / row of the tile
    const int uc0 = ts - a.sx0 - (FS - 1 + OX1);                 // cell of tile column 0
    const int vc0 = tv - a.sy0 - (FS - 1 + OY1);                 // cell row of tile g row pair 0
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    for (int plane = blockIdx.y; plane < a.pl.n_planes; plane += gridDim.y) {
        const float* __restrict__ g = a.pl.g + (long long)plane * a.pl.g_stride;
        __syncthreads(); // the previous plane's tile is no longer read
        // ---- stage: tile row gr = 2 * (cell row) + py, column tc -> {g[Y][X], g[Y][X+2], g[Y][X+1], g[Y][X+3]}, X = x0 + 2c.
        //      Cells outside the plane are clamped: they only feed samples this kernel does not store.
        for (int e = threadIdx.x; e < G::NR * G::NCP; e += G::THREADS) {
            const int gr = e / G::NCP, tc = e - gr * G::NCP;
            const int Y = min(max(a.y0 + 2 * (vc0 + (gr >> 1)) + (gr & 1), 0), a.dst_h - 1);
            const int X = a.x0 + 2 * (uc0 + tc);
            const float* __restrict__ row = g + (long long)Y * a.pl.g_pitch;
            float4 q;
            q.x = __ldg(row + min(max(X, 0), a.dst_w - 1));
            q.y = __ldg(row + min(max(X + 2, 0), a.dst_w - 1));
            q.z = __ldg(row + min(max(X + 1, 0), a.dst_w - 1));
            q.w = __ldg(row + min(max(X + 3, 0), a.dst_w - 1));
            tile[gr * G::NCP + (tc & 3) * G::SUB + (tc >> 2)] = q;
        }
        __syncthreads();

        float2 acc[G::RY][2]; // [row][sample pair]: samples 4 lane + 2p, + 1
#pragma unroll
        for (int iy = 0; iy < G::RY; ++iy)
            acc[iy][0] = acc[iy][1] = make_float2(0.f, 0.f);
        const float4* __restrict__ tl = tile + lane;

        // g cell rows ascending (kk); sample row iy takes cell row kk with k = FS - 1 + OY1 + iy - kk: phase row 0 at tap row
        // k, phase row 1 at k - OY1; within a g row the cells ascend (j descending), phase 0 before phase 1
        auto g_row = [&](int kk, int py) {
            const float4* __restrict__ trow = tl + (size_t)(2 * (warp * G::RY + kk) + py) * G::NCP;
            float4 seg[NSEG];
#pragma unroll
            for (int m = 0; m < NSEG; ++m)
                seg[m] = trow[(m & 3) * G::SUB + (m >> 2)];
#pragma unroll
            for (int iy = 0; iy < G::RY; ++iy) {
                const int ly = FS - 1 + OY1 + iy - kk - py * OY1;
                if (ly < 0 || ly >= FS)
                    continue;
#pragma unroll
                for (int j = FS - 1 + OX1; j >= 0; --j) {
                    if (j < FS) {
                        const float w0 = W.w[py][0][ly][j];
#pragma unroll
                        for (int p = 0; p < 2; ++p) {
                            const float4 s = seg[2 * p - j + FS - 1 + OX1];
                            acc[iy][p] = __ffma2_rn(make_float2(s.x, s.y), make_float2(w0, w0), acc[iy][p]);
                        }
                    }
                    if (j - OX1 >= 0 && j - OX1 < FS) {
                        const float w1 = W.w[py][1][ly][j - OX1];
#pragma unroll
                        for (int p = 0; p < 2; ++p) {
                            const float4 s = seg[2 * p - j + FS - 1 + OX1];
                            acc[iy][p] = __ffma2_rn(make_float2(s.z, s.w), make_float2(w1, w1), acc[iy][p]);
                        }
                    }
                }
            }
        };
        if constexpr (FS <= 9) {
#pragma unroll
            for (int kk = 0; kk < NK; ++kk) {
                g_row(kk, 0);
                g_row(kk, 1);
            }
        } else {
#pragma unroll 1
            for (int kk = 0; kk < NK; ++kk) {
                g_row(kk, 0);
                g_row(kk, 1);
            }
        }

        float* __restrict__ out = a.pl.out + (long long)plane * a.pl.o_stride;
        const int sx = ts + AU_TX * lane;
#pragma unroll
        for (int iy = 0; iy < G::RY; ++iy) {
            const int sy = tv + warp * G::RY + iy;
            if (sy >= a.uy1)
                continue;
            float* o = out + (long long)sy * a.pl.o_pitch;
            const float v[4] = {acc[iy][0].x, acc[iy][0].y, acc[iy][1].x, acc[iy][1].y};
#pragma unroll
            for (int i = 0; i < AU_TX; ++i)
                if (sx + i < a.ux1)
                    o[sx + i] = v[i];
        }
    }
}

template <int FS>
int launch_adjoint_up2x_fs(const jinc_table* t, const AdjUpArgs& a, int grid_y, cudaStream_t st)
{
    using G = AdjUpGeom<FS>;
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
    void (*kern)(AdjUpArgs, UpWeights<FS>) = u.ox1 ? (u.oy1 ? adjoint_up2x<FS, 1, 1> : adjoint_up2x<FS, 1, 0>)
                                                   : (u.oy1 ? adjoint_up2x<FS, 0, 1> : adjoint_up2x<FS, 0, 0>);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G::SMEM);
    if (e != cudaSuccess)
        return jinc_fail(JINC_E_CUDA, "cudaFuncSetAttribute(adjoint_up2x smem %zu): %s", G::SMEM, cudaGetErrorString(e));
    kern<<<dim3((unsigned)a.tiles, (unsigned)grid_y), G::THREADS, G::SMEM, st>>>(a, w);
    e = cudaGetLastError();
    if (e != cudaSuccess)
        return jinc_fail(JINC_E_CUDA, "adjoint_up2x launch failed: %s", cudaGetErrorString(e));
    return JINC_OK;
}

int launch_adjoint_up2x(const jinc_table* t, AdjUpArgs& a, int grid_y, cudaStream_t st)
{
    int th = 0;
    switch (t->sc.fs) {
    case 7: th = AdjUpGeom<7>::TH; break;
    case 9: th = AdjUpGeom<9>::TH; break;
    default: th = AdjUpGeom<11>::TH; break;
    }
    a.tiles_x = (a.ux1 - a.ux0 + AdjUpGeom<7>::TW - 1) / AdjUpGeom<7>::TW;
    a.tiles = a.tiles_x * ((a.uy1 - a.uy0 + th - 1) / th);
    switch (t->sc.fs) {
    case 7: return launch_adjoint_up2x_fs<7>(t, a, grid_y, st);   // tap 3
    case 9: return launch_adjoint_up2x_fs<9>(t, a, grid_y, st);   // tap 4
    case 11: return launch_adjoint_up2x_fs<11>(t, a, grid_y, st); // tap 5
    case 13: return launch_adjoint_up2x_fs<13>(t, a, grid_y, st); // tap 6
    case 15: return launch_adjoint_up2x_fs<15>(t, a, grid_y, st); // tap 7
    case 17: return launch_adjoint_up2x_fs<17>(t, a, grid_y, st); // tap 8
    default: return jinc_fail(JINC_E_UNSUPPORTED, "adjoint_up2x: no kernel for fs %d", t->sc.fs);
    }
}

// Source samples [lo, hi) along one axis that the 2x kernel takes: every output covering the sample (from the table's
// start array) lies in the plan's cells [0, nc), and every cell u - j (tap j of phase 0, j - o1 of phase 1) exists.
void up2x_source_range(const std::vector<int32_t>& start, int fs, int n_src, int out0, int nc, int s0, int o1, int& lo, int& hi)
{
    const int n = (int)start.size();
    lo = INT_MAX;
    hi = INT_MIN;
    int a = 0, b = 0; // covering outputs of sample s: [a, b)
    for (int s = 0; s < n_src; ++s) {
        while (a < n && start[a] <= s - fs)
            ++a;
        while (b < n && start[b] <= s)
            ++b;
        const int u = s - s0;
        if (a >= out0 && b <= out0 + 2 * nc && b > a && u >= fs - 1 + o1 && u <= nc - 1) {
            lo = std::min(lo, s);
            hi = s + 1;
        }
    }
    if (lo >= hi)
        lo = hi = 0;
}

} // namespace

int jinc_launch_adjoint(const jinc_table* t, int n_planes, const float* g, long long g_pitch, long long g_stride, float* out,
                        long long out_pitch, long long out_stride, cudaStream_t st, int* launches)
{
    const int W = t->sc.src_w, H = t->sc.src_h;
    const int grid_y = std::min(n_planes, 65535);
    AdjPlanes pl{g, g_pitch, g_stride, out, out_pitch, out_stride, n_planes};
    int ux0 = 0, ux1 = 0, uy0 = 0, uy1 = 0;
    const Up2xPlan& u = t->up2x;
    if (t->fast_path == JINC_PATH_UP2X && u.ok && up2x_supported(t->sc.fs)) {
        up2x_source_range(t->h_start[0], t->sc.fs, W, u.x0, u.ncx, u.sx0, u.ox1, ux0, ux1);
        up2x_source_range(t->h_start[1], t->sc.fs, H, u.y0, u.ncy, u.sy0, u.oy1, uy0, uy1);
        if (ux1 > ux0 && uy1 > uy0) {
            AdjUpArgs a;
            memset(&a, 0, sizeof(a));
            a.pl = pl;
            a.dst_w = t->sc.dst_w;
            a.dst_h = t->sc.dst_h;
            a.x0 = u.x0;
            a.y0 = u.y0;
            a.sx0 = u.sx0;
            a.sy0 = u.sy0;
            a.ux0 = ux0;
            a.ux1 = ux1;
            a.uy0 = uy0;
            a.uy1 = uy1;
            if (int rc = launch_adjoint_up2x(t, a, grid_y, st))
                return rc;
            ++*launches;
        } else {
            ux0 = ux1 = uy0 = uy1 = 0;
        }
    }
    // every other source sample: the frame around the 2x rectangle (all of it when there is none)
    AdjGeneralArgs ga;
    memset(&ga, 0, sizeof(ga));
    fill_strip_args(t, ga.st);
    ga.pl = pl;
    ga.dst_w = t->sc.dst_w;
    ga.dst_h = t->sc.dst_h;
    Rect rects[4];
    int n_rects = 0;
    if (ux1 > ux0) {
        rects[n_rects++] = Rect{0, 0, W, uy0};
        rects[n_rects++] = Rect{0, uy1, W, H};
        rects[n_rects++] = Rect{0, uy0, ux0, uy1};
        rects[n_rects++] = Rect{ux1, uy0, W, uy1};
    } else {
        rects[n_rects++] = Rect{0, 0, W, H};
    }
    unsigned total = 0;
    int k = 0;
    for (int r = 0; r < n_rects; ++r) {
        const int w = rects[r].x1 - rects[r].x0, h = rects[r].y1 - rects[r].y0;
        if (w <= 0 || h <= 0)
            continue;
        ga.rect[k] = rects[r];
        ga.tiles_x[k] = (unsigned)((w + AG_TW - 1) / AG_TW);
        ga.tile_begin[k] = total;
        total += ga.tiles_x[k] * (unsigned)((h + AG_TH - 1) / AG_TH);
        ++k;
    }
    for (int j = k; j < 4; ++j) {
        ga.rect[j] = Rect{0, 0, 1, 1};
        ga.tiles_x[j] = 1;
        ga.tile_begin[j] = total;
    }
    ga.tile_begin[4] = total;
    if (total == 0)
        return JINC_OK;
    adjoint_general<<<dim3(total, (unsigned)grid_y), AG_THREADS, AG_G_FLOATS * sizeof(float), st>>>(ga);
    JINC_CUDA(cudaGetLastError());
    ++*launches;
    return JINC_OK;
}

extern "C" int jinc_resize_adjoint_planes_device(jinc_ctx* ctx, const jinc_table* t, int n_planes, const float* d_grad_dst,
                                                 ptrdiff_t grad_dst_pitch, ptrdiff_t grad_dst_plane_stride, float* d_grad_src,
                                                 ptrdiff_t grad_src_pitch, ptrdiff_t grad_src_plane_stride, void* stream)
{
    if (!ctx || !t || !d_grad_dst || !d_grad_src)
        return jinc_fail(JINC_E_INVALID, "jinc_resize_adjoint_planes_device: null argument");
    if (n_planes < 1)
        return jinc_fail(JINC_E_INVALID, "jinc_resize_adjoint_planes_device: n_planes must be at least 1");
    if ((reinterpret_cast<uintptr_t>(d_grad_dst) | reinterpret_cast<uintptr_t>(d_grad_src)) % 4)
        return jinc_fail(JINC_E_INVALID, "jinc_resize_adjoint_planes_device: planes must be 4-byte aligned");
    const long long dw = t->sc.dst_w, dh = t->sc.dst_h, sw = t->sc.src_w, sh = t->sc.src_h;
    if (grad_dst_pitch < dw * 4 || grad_dst_pitch % 4 || grad_src_pitch < sw * 4 || grad_src_pitch % 4)
        return jinc_fail(JINC_E_INVALID, "jinc_resize_adjoint_planes_device: pitches must be multiples of 4 bytes and hold a row");
    if (n_planes > 1 && (grad_dst_plane_stride < dh * grad_dst_pitch || grad_dst_plane_stride % 4 || grad_src_plane_stride < sh * grad_src_pitch ||
                         grad_src_plane_stride % 4))
        return jinc_fail(JINC_E_INVALID, "jinc_resize_adjoint_planes_device: plane strides must be multiples of 4 bytes and hold a plane");
    const uintptr_t g0 = reinterpret_cast<uintptr_t>(d_grad_dst), o0 = reinterpret_cast<uintptr_t>(d_grad_src);
    const uintptr_t g1 = g0 + (uintptr_t)((n_planes - 1) * (long long)grad_dst_plane_stride + (dh - 1) * grad_dst_pitch + dw * 4);
    const uintptr_t o1 = o0 + (uintptr_t)((n_planes - 1) * (long long)grad_src_plane_stride + (sh - 1) * grad_src_pitch + sw * 4);
    if (g0 < o1 && o0 < g1)
        return jinc_fail(JINC_E_INVALID, "jinc_resize_adjoint_planes_device: d_grad_src must not overlap d_grad_dst");
    JINC_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    int launches = 0;
    return jinc_launch_adjoint(t, n_planes, d_grad_dst, grad_dst_pitch / 4, grad_dst_plane_stride / 4, d_grad_src, grad_src_pitch / 4,
                               grad_src_plane_stride / 4, st, &launches);
}
