// jinc_table.cu -- coefficient-table generation on the device.
//
// Replaces generate_coeff_table_c (src/JincResize.cpp:336-533).  The reference walks all dst_w*dst_h output
// pixels serially and stores {start_x,start_y,coeff_meta} per pixel plus one fs x coeff_stride weight block per
// unique quantised phase AND per border pixel (hundreds of MB).  Two facts make a much smaller parallel table
// exact:
//   * positions are separable: xpos depends only on x (it restarts every row, :528), ypos only on y (:527);
//     window origin, border flag and quantised phase are therefore per-axis quantities;
//   * the block shared by all interior pixels of phase (qy,qx) is the one computed at the FIRST such pixel in
//     row-major order (:431-435,517-518) = (first interior row with phase qy, first interior column with qx).
// So the device table is: per-axis arrays (pos, start, phase, border, rank) + one block per used phase pair.
// Border pixels get their weights on the fly in the resample kernel from the same LUT (jinc_weights.cuh).
//
// Bit-exactness rules (SURVEY.md 7.3): positions are a sequential float accumulation (one thread per axis),
// every float/double operation uses an explicit round-to-nearest intrinsic so nvcc cannot contract a*b+c into
// an FMA, and the block normaliser is a sequential float sum in row-major order.
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <unordered_map>

#include "jinc_internal.h"
#include "jinc_up2x_taps.h"
#include "jinc_weights.cuh"

namespace {

constexpr int kAxisThreads = 1024;
constexpr size_t kBorderWeightBudget = (size_t)8 << 30; // resident per-pixel border weights per table
constexpr size_t kPaddedWeightBudget = (size_t)1 << 30; // second copy of the phase blocks with 16-byte rows

struct AxisKernelArgs {
    float* pos;
    int32_t* start;
    int32_t* qint;
    int32_t* phase;
    int32_t* rank;
    uint8_t* border;
    int32_t* rep;
    int32_t* rank_of;
    double* rep_d2;
    int32_t* n_rank_out;
    int n, src_n, quant, fs;
    float pos0, pos_step, support;
    double filt_step;
};

// K1+K2: one block per axis.
__global__ void __launch_bounds__(kAxisThreads) axis_kernel(AxisKernelArgs ax0, AxisKernelArgs ax1)
{
    const AxisKernelArgs a = blockIdx.x == 0 ? ax0 : ax1;
    __shared__ int s_rep[256];
    __shared__ int s_rank_of[256];
    const int tid = threadIdx.x;

    if (tid < 256)
        s_rep[tid] = INT_MAX;
    if (tid == 0) {
        // xpos += x_step / ypos += y_step (:524,527): sequential float accumulation, NOT pos0 + i*step
        float p = a.pos0;
        for (int i = 0; i < a.n; ++i) {
            a.pos[i] = p;
            p = __fadd_rn(p, a.pos_step);
        }
    }
    __syncthreads();

    for (int i = tid; i < a.n; i += kAxisThreads) {
        const float p = a.pos[i];
        int border = 0;
        int end = __float2int_rz(__fadd_rn(p, a.support)); // :392-393 truncation, not floor
        if (end >= a.src_n) {
            end = a.src_n - 1;
            border = 1;
        }
        int begin = end - a.fs + 1;
        if (begin < 0) {
            begin = 0;
            border = 1;
        }
        const int qi = __float2int_rz(__fmul_rn(p, (float)a.quant)); // :424-425
        const int ph = qi % a.quant;                                 // C remainder (:426-427)
        a.start[i] = begin;
        a.border[i] = (uint8_t)border;
        a.qint[i] = qi;
        a.phase[i] = ph;
        if (!border)
            atomicMin(&s_rep[ph], i); // first interior index holding this phase (:431,517)
    }
    __syncthreads();

    if (tid < 256) {
        int r = -1;
        if (tid < a.quant && s_rep[tid] != INT_MAX) {
            r = 0;
            for (int v = 0; v < tid; ++v)
                r += s_rep[v] != INT_MAX;
        }
        s_rank_of[tid] = r;
        if (tid < a.quant) {
            a.rep[tid] = s_rep[tid];
            a.rank_of[tid] = r;
        }
    }
    if (tid == 0) {
        int c = 0;
        for (int v = 0; v < a.quant; ++v)
            c += s_rep[v] != INT_MAX;
        *a.n_rank_out = c;
    }
    __syncthreads();

    for (int i = tid; i < a.n; i += kAxisThreads)
        a.rank[i] = a.border[i] ? -1 : s_rank_of[a.phase[i]];

    // squared scaled tap distances of every phase representative (:446-451,485-486): the weights' own window
    // comes from the QUANTISED position, while meta.start above came from the unquantised one.
    const int total = a.quant * a.fs;
    for (int e = tid; e < total; e += kAxisThreads) {
        const int v = e / a.fs, l = e - v * a.fs;
        const int r = s_rank_of[v];
        if (r < 0)
            continue;
        const int irep = s_rep[v];
        const float qpos = __fdiv_rn((float)a.qint[irep], (float)a.quant); // :428-429
        const int begin = __float2int_rz(__fadd_rn(qpos, a.support)) - a.fs + 1;
        a.rep_d2[r * a.fs + l] = jinc_tap_dist2(qpos, a.src_n, begin + l, a.filt_step);
    }
}

// weight rows padded to 16 bytes (pad = 0)
__global__ void __launch_bounds__(256) pad_rows_kernel(float* __restrict__ out, const float* __restrict__ in, size_t rows, int fs, int fsp)
{
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= rows * fsp)
        return;
    const size_t r = i / fsp;
    const int c = (int)(i - r * fsp);
    out[i] = c < fs ? in[r * fs + c] : 0.f;
}

// K3: one block per used phase pair (ry, rx).
__global__ void __launch_bounds__(128) phase_blocks_kernel(float* __restrict__ weights, const double* __restrict__ dx2,
                                                           const double* __restrict__ dy2,
                                                           const float* __restrict__ lut, int n_rank_x, int fs,
                                                           double radius2, double idx_scale)
{
    const int b = blockIdx.x;
    const int ry = b / n_rank_x, rx = b - ry * n_rank_x;
    const int taps = fs * fs;
    float* w = weights + (size_t)b * taps;
    __shared__ float s_sum;

    for (int t = threadIdx.x; t < taps; t += blockDim.x) {
        const int ly = t / fs, lx = t - ly * fs;
        const double d2 = __dadd_rn(dx2[rx * fs + lx], dy2[ry * fs + ly]);
        w[t] = jinc_lut_weight(lut, d2, radius2, idx_scale); // :488-492
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f; // divider: float running sum in row-major tap order (:439,493)
        for (int t = 0; t < taps; ++t)
            s = __fadd_rn(s, w[t]);
        s_sum = s;
    }
    __syncthreads();
    const float s = s_sum;
    for (int t = threadIdx.x; t < taps; t += blockDim.x)
        w[t] = __fdiv_rn(w[t], s); // :505-514
}

// Normaliser of every border pixel: the float running sum of its window's LUT factors in row-major tap order
// (:439,493), from the UNquantised position and the clamped window origin (:443-451 are skipped for border pixels).
struct BorderSumArgs {
    BorderGeom g;
    const float* pos_x;
    const float* pos_y;
    const int32_t* start_x;
    const int32_t* start_y;
    const float* lut;
    float* sums;
    float* weights; // [g.total / 32][fs*fs][32] normalised per-pixel weights (neighbouring pixels coalesce, tap stride 32), or null
    int fs, src_w, src_h;
    double step_x, step_y, radius2, idx_scale;
};

__global__ void __launch_bounds__(256) border_sum_kernel(BorderSumArgs a)
{
    const long long slot = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= a.g.total)
        return;
    // invert jinc_border_slot
    int x, y;
    const BorderGeom& g = a.g;
    if (slot < g.off_bottom) {
        y = (int)(slot / g.W);
        x = (int)(slot - (long long)y * g.W);
    } else if (slot < g.off_left) {
        const long long r = slot - g.off_bottom;
        y = g.by1 + (int)(r / g.W);
        x = (int)(r % g.W);
    } else if (slot < g.off_right) {
        const long long r = slot - g.off_left;
        y = g.by0 + (int)(r / g.bx0);
        x = (int)(r % g.bx0);
    } else {
        const long long r = slot - g.off_right;
        const int w = g.W - g.bx1;
        y = g.by0 + (int)(r / w);
        x = g.bx1 + (int)(r % w);
    }
    const float px = a.pos_x[x], py = a.pos_y[y];
    const int sx = a.start_x[x], sy = a.start_y[y];
    float sum = 0.f;
    for (int ly = 0; ly < a.fs; ++ly) {
        const double dy2 = jinc_tap_dist2(py, a.src_h, sy + ly, a.step_y);
        for (int lx = 0; lx < a.fs; ++lx) {
            const double dx2 = jinc_tap_dist2(px, a.src_w, sx + lx, a.step_x);
            sum = __fadd_rn(sum, jinc_lut_weight(a.lut, __dadd_rn(dx2, dy2), a.radius2, a.idx_scale));
        }
    }
    a.sums[slot] = sum;
    if (!a.weights)
        return;
    float* w = a.weights + (size_t)(slot >> 5) * (size_t)(a.fs * a.fs * 32) + (slot & 31);
    for (int ly = 0; ly < a.fs; ++ly) {
        const double dy2 = jinc_tap_dist2(py, a.src_h, sy + ly, a.step_y);
        for (int lx = 0; lx < a.fs; ++lx) {
            const double dx2 = jinc_tap_dist2(px, a.src_w, sx + lx, a.step_x);
            *w = __fdiv_rn(jinc_lut_weight(a.lut, __dadd_rn(dx2, dy2), a.radius2, a.idx_scale), sum); // :505-514
            w += 32;
        }
    }
}

// Weight block of one border class, from its representative pixel: factor / divider (:488-514), row-major taps.
__global__ void __launch_bounds__(128) border_class_kernel(BorderSumArgs a, const int2* __restrict__ reps, float* __restrict__ out)
{
    const int2 r = reps[blockIdx.x];
    const float px = a.pos_x[r.x], py = a.pos_y[r.y];
    const int sx = a.start_x[r.x], sy = a.start_y[r.y];
    const float sum = a.sums[jinc_border_slot(a.g, r.x, r.y)];
    const int fsp = (a.fs + 3) & ~3; // rows padded to 16 bytes (the pad stays 0 from the memset)
    float* w = out + (size_t)blockIdx.x * a.fs * fsp;
    for (int t = threadIdx.x; t < a.fs * a.fs; t += blockDim.x) {
        const int ly = t / a.fs, lx = t - ly * a.fs;
        const double dy2 = jinc_tap_dist2(py, a.src_h, sy + ly, a.step_y);
        const double dx2 = jinc_tap_dist2(px, a.src_w, sx + lx, a.step_x);
        w[ly * fsp + lx] = __fdiv_rn(jinc_lut_weight(a.lut, __dadd_rn(dx2, dy2), a.radius2, a.idx_scale), sum);
    }
}

// packs the weight blocks a strip plan names (sel << 31 | block) next to each other: one thread block per weight block.
// Lives here, not next to the planner in jinc_resize.cu: that module (the general kernels) is large and would be loaded
// just for this launch, 20 ms on the first table of a process.
__global__ void __launch_bounds__(128) gather_blocks_kernel(float* __restrict__ out, const uint32_t* __restrict__ list, const float* __restrict__ phase_blocks,
                                                            const float* __restrict__ border_blocks, int block_floats)
{
    const uint32_t e = list[blockIdx.x];
    const float* __restrict__ src = ((e >> 31) ? border_blocks : phase_blocks) + (size_t)(e & 0x7fffffffu) * block_floats;
    float* __restrict__ dst = out + (size_t)blockIdx.x * block_floats;
    for (int i = threadIdx.x; i < block_floats; i += blockDim.x)
        dst[i] = src[i];
}

template <typename T>
int dev_alloc(T** p, size_t count)
{
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T));
    if (e != cudaSuccess)
        return jinc_fail(JINC_E_NOMEM, "cudaMalloc(%zu bytes) failed: %s", count * sizeof(T), cudaGetErrorString(e));
    return JINC_OK;
}

double dmin(double a, double b) { return a < b ? a : b; }

// Host-side scalars in the reference's own expression shapes and precisions (:349-364).
void derive_scalars(const jinc_table_params& p, TableScalars& s)
{
    s.quant_x = p.quant_x;
    s.quant_y = p.quant_y;
    s.src_w = p.src_w;
    s.src_h = p.src_h;
    s.dst_w = p.dst_w;
    s.dst_h = p.dst_h;
    s.filt_step[0] = dmin(static_cast<double>(p.dst_w) / p.crop_w, 1.0);
    s.filt_step[1] = dmin(static_cast<double>(p.dst_h) / p.crop_h, 1.0);
    const float sup_x = static_cast<float>(p.radius / s.filt_step[0]);
    const float sup_y = static_cast<float>(p.radius / s.filt_step[1]);
    s.support = sup_x > sup_y ? sup_x : sup_y;
    const int fx = static_cast<int>(std::ceil(sup_x * 2.0)), fy = static_cast<int>(std::ceil(sup_y * 2.0));
    s.fs = fx > fy ? fx : fy;
    s.pos0[0] = static_cast<float>(p.crop_left + (p.crop_w / p.dst_w - 1.0) / 2.0);
    s.pos0[1] = static_cast<float>(p.crop_top + (p.crop_h - p.dst_h) / static_cast<double>(p.dst_h * static_cast<int64_t>(2)));
    s.pos_step[0] = static_cast<float>(p.crop_w / p.dst_w);
    s.pos_step[1] = static_cast<float>(p.crop_h / p.dst_h);
    s.radius2 = p.radius * p.radius;
    s.idx_scale = (JINC_LUT_SAMPLES - 1) / s.radius2;
}

// The run [a,b) of non-border indices.  Border flags are monotone along an axis (windows are clamped only at the two ends:
// src/JincResize.cpp:395-418), so the first run found is the only one.
void interior_run(const std::vector<uint8_t>& border, int& a, int& b)
{
    const int n = static_cast<int>(border.size());
    a = 0;
    while (a < n && border[a])
        ++a;
    b = a;
    while (b < n && !border[b])
        ++b;
}

int round_up(int v, int m) { return (v + m - 1) / m * m; }

// Exact-2x structure on one axis over [a,b): start[i+2]==start[i]+1 and rank[i+2]==rank[i].
bool axis_is_up2x(const std::vector<int32_t>& start, const std::vector<int32_t>& rank, int a, int b)
{
    if (b - a < 4)
        return false;
    for (int i = a; i + 2 < b; ++i)
        if (start[i + 2] != start[i] + 1 || rank[i + 2] != rank[i])
            return false;
    const int d = start[a + 1] - start[a];
    return d == 0 || d == 1;
}

// Integer-ratio downscale on one axis: start[i+1]==start[i]+q (q>=2), single rank.
int axis_down_ratio(const std::vector<int32_t>& start, const std::vector<int32_t>& rank, int a, int b)
{
    if (b - a < 2)
        return 0;
    const int q = start[a + 1] - start[a];
    if (q < 2)
        return 0;
    for (int i = a; i + 1 < b; ++i)
        if (start[i + 1] != start[i] + q || rank[i + 1] != rank[a])
            return 0;
    return q;
}

// Periodic axis: start[i+P] == start[i] + Q and rank[i+P] == rank[i] over the interior run; smallest P in 2..4.
bool axis_periodic(const std::vector<int32_t>& start, const std::vector<int32_t>& rank, int a, int b, int& P, int& Q)
{
    for (P = 2; P <= 4; ++P) {
        if (b - a < 4 * P)
            continue;
        Q = start[a + P] - start[a];
        if (Q < 1)
            continue;
        bool ok = true;
        for (int i = a; ok && i + P < b; ++i)
            ok = start[i + P] == start[i] + Q && rank[i + P] == rank[i];
        if (ok)
            return true;
    }
    return false;
}

// Piecewise-periodic structure of one axis over the interior run [a,b): the smallest P <= 16 (cell = P outputs) for which
// start[i+P] - start[i] is one constant Q almost everywhere, then chunks of up to N cells inside which every residue
// keeps its rank and its origins advance by exactly Q per cell.  False when the axis has no such structure or the
// chunks come out too short to be worth a thread each.
bool build_cells_axis(const std::vector<int32_t>& start, const std::vector<int32_t>& rank, int a, int b, int N, CellsAxis& out)
{
    for (int P = 1; P <= 16; ++P) { // 9:4 (480p -> 1080p) has P = 9
        const int n = b - a - P;
        if (n < 8 * P)
            continue;
        std::unordered_map<int, int> hist;
        for (int i = a; i + P < b; ++i)
            ++hist[start[i + P] - start[i]];
        int Q = 0, best = 0;
        for (auto& kv : hist)
            if (kv.second > best) {
                best = kv.second;
                Q = kv.first;
            }
        if (Q < 1 || best < n - n / 50)
            continue;
        out = CellsAxis();
        out.P = P;
        out.Q = Q;
        out.first = a;
        out.ncells = (b - a) / P;
        // Chunks live on a REGULAR grid of N-cell groups: a group inside which some residue changes its rank (or an
        // origin steps irregularly) becomes several chunks, each with the group's origin extrapolated back to the group's
        // first cell.  A thread computes all N cells of its group and stores the ones of its chunk, so every lane of a warp
        // reads the same shared-memory alignment (neighbouring lanes of a split group read the same words: a broadcast).
        for (int c0 = 0; c0 < out.ncells; c0 += N) {
            const int c1 = std::min(out.ncells, c0 + N);
            int c = c0;
            while (c < c1) {
                int len = 1;
                while (c + len < c1) {
                    bool same = true;
                    for (int p = 0; p < P && same; ++p) {
                        const int i0 = a + P * (c + len - 1) + p, i1 = i0 + P;
                        same = rank[i1] == rank[i0] && start[i1] == start[i0] + Q;
                    }
                    if (!same)
                        break;
                    ++len;
                }
                out.cell.push_back(c0);
                out.i0.push_back(c - c0);
                out.n.push_back(len);
                for (int p = 0; p < P; ++p) {
                    out.org.push_back(start[a + P * c + p] - Q * (c - c0));
                    out.rank.push_back(rank[a + P * c + p]);
                }
                c += len;
            }
        }
        out.n_chunks = static_cast<int>(out.cell.size());
        const long long groups = (out.ncells + N - 1) / N;
        return out.ncells >= 8 && static_cast<long long>(out.n_chunks) * 3 <= groups * 4 + 8;
    }
    return false;
}

// every window of `per_tile` consecutive chunks (tiles start anywhere on the y axis: row bands) must fit the footprint the
// kernel stages: from the smallest origin of the first chunk to the end of the last window a thread READS -- a thread
// always walks all N cells of its chunk, also the ones a short chunk does not have
bool cells_footprints_fit(const CellsAxis& ax, int fs, int N, int per_tile, int limit, bool any_start)
{
    for (int k0 = 0; k0 < ax.n_chunks; k0 += any_start ? 1 : per_tile) {
        const int k1 = std::min(ax.n_chunks, k0 + per_tile);
        int lo = INT_MAX, hi = INT_MIN;
        for (int p = 0; p < ax.P; ++p)
            lo = std::min(lo, ax.org[(size_t)k0 * ax.P + p]);
        for (int k = k0; k < k1; ++k)
            for (int p = 0; p < ax.P; ++p) {
                const int o = ax.org[(size_t)k * ax.P + p];
                if (o < lo)
                    return false; // origins must not run backwards inside a tile
                hi = std::max(hi, o + ax.Q * (N - 1) + fs);
            }
        if (hi - lo > limit)
            return false;
    }
    return true;
}

int upload_cells_axis(CellsAxis& ax, cudaStream_t st)
{
    int rc = dev_alloc(&ax.d_cell, ax.cell.size());
    rc = rc ? rc : dev_alloc(&ax.d_i0, ax.i0.size());
    rc = rc ? rc : dev_alloc(&ax.d_n, ax.n.size());
    rc = rc ? rc : dev_alloc(&ax.d_org, ax.org.size());
    rc = rc ? rc : dev_alloc(&ax.d_rank, ax.rank.size());
    if (rc)
        return rc;
    JINC_CUDA(cudaMemcpyAsync(ax.d_cell, ax.cell.data(), ax.cell.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    JINC_CUDA(cudaMemcpyAsync(ax.d_i0, ax.i0.data(), ax.i0.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    JINC_CUDA(cudaMemcpyAsync(ax.d_n, ax.n.data(), ax.n.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    JINC_CUDA(cudaMemcpyAsync(ax.d_org, ax.org.data(), ax.org.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    JINC_CUDA(cudaMemcpyAsync(ax.d_rank, ax.rank.data(), ax.rank.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    return JINC_OK;
}

void plan_fast_paths(jinc_table* t)
{
    int ax_a[2], ax_b[2];
    for (int k = 0; k < 2; ++k)
        interior_run(t->h_border[k], ax_a[k], ax_b[k]);
    t->fast_path = JINC_PATH_GENERAL;
    t->ix0 = t->ix1 = t->iy0 = t->iy1 = 0;

    const int nrx = t->ax[0].n_rank;
    if (axis_is_up2x(t->h_start[0], t->h_rank[0], ax_a[0], ax_b[0]) &&
        axis_is_up2x(t->h_start[1], t->h_rank[1], ax_a[1], ax_b[1])) {
        Up2xPlan& u = t->up2x;
        u.x0 = round_up(ax_a[0], 8); // 8-pixel alignment keeps the kernel's row stores vector-aligned
        u.y0 = round_up(ax_a[1], 2);
        u.ncx = (ax_b[0] - u.x0) / 2;
        u.ncy = (ax_b[1] - u.y0) / 2;
        if (u.ncx >= 8 && u.ncy >= 2) {
            u.sx0 = t->h_start[0][u.x0];
            u.sy0 = t->h_start[1][u.y0];
            u.ox1 = t->h_start[0][u.x0 + 1] - u.sx0;
            u.oy1 = t->h_start[1][u.y0 + 1] - u.sy0;
            for (int py = 0; py < 2; ++py)
                for (int px = 0; px < 2; ++px)
                    u.wblock[py][px] = t->h_rank[1][u.y0 + py] * nrx + t->h_rank[0][u.x0 + px];
            u.ok = (u.ox1 == 0 || u.ox1 == 1) && (u.oy1 == 0 || u.oy1 == 1);
            if (u.ok) {
                t->fast_path = JINC_PATH_UP2X;
                t->ix0 = u.x0;
                t->ix1 = u.x0 + 2 * u.ncx;
                t->iy0 = u.y0;
                t->iy1 = u.y0 + 2 * u.ncy;
                return;
            }
        }
    }
    const int qx = axis_down_ratio(t->h_start[0], t->h_rank[0], ax_a[0], ax_b[0]);
    const int qy = axis_down_ratio(t->h_start[1], t->h_rank[1], ax_a[1], ax_b[1]);
    if (qx >= 2 && qy >= 2) {
        DownPlan& d = t->down;
        d.x0 = round_up(ax_a[0], 4);
        d.y0 = ax_a[1];
        d.nx = ax_b[0] - d.x0;
        d.ny = ax_b[1] - d.y0;
        if (d.nx >= 8 && d.ny >= 2) {
            d.sx0 = t->h_start[0][d.x0];
            d.sy0 = t->h_start[1][d.y0];
            d.qx = qx;
            d.qy = qy;
            d.wblock = t->h_rank[1][d.y0] * nrx + t->h_rank[0][d.x0];
            d.ok = true;
            // the polyphase kernel is selected in jinc_resize.cu when it supports this (fs, qx, qy)
            t->fast_path = JINC_PATH_DOWN_INT;
            t->ix0 = d.x0;
            t->ix1 = d.x0 + d.nx;
            t->iy0 = d.y0;
            t->iy1 = d.y0 + d.ny;
        }
        return; // an integer ratio also looks periodic (P = 2, Q = 2q): it is the polyphase kernel's own case
    }
    // rational ratios with piecewise-periodic phases (exactly periodic ones included): chunked cells
    {
        CellsPlan& u = t->cells;
        const int fs = t->sc.fs;
        if (build_cells_axis(t->h_start[0], t->h_rank[0], ax_a[0], ax_b[0], JINC_CELLS_NX, u.ax[0]) &&
            build_cells_axis(t->h_start[1], t->h_rank[1], ax_a[1], ax_b[1], JINC_CELLS_NY, u.ax[1]) && u.ax[0].Q == u.ax[1].Q &&
            jinc_cells_instantiated(u.ax[0].Q, fs) &&
            cells_footprints_fit(u.ax[0], fs, JINC_CELLS_NX, 32, jinc_cells_footprint(u.ax[0].Q, fs, JINC_CELLS_NX, 32), false) &&
            cells_footprints_fit(u.ax[1], fs, JINC_CELLS_NY, jinc_cells_warps(u.ax[1].Q, fs),
                                 jinc_cells_footprint(u.ax[1].Q, fs, JINC_CELLS_NY, jinc_cells_warps(u.ax[1].Q, fs)), true)) {
            u.Q = u.ax[0].Q;
            u.ok = true;
            t->fast_path = JINC_PATH_CELLS;
            t->ix0 = u.ax[0].first;
            t->ix1 = u.ax[0].first + u.ax[0].P * u.ax[0].ncells;
            t->iy0 = u.ax[1].first;
            t->iy1 = u.ax[1].first + u.ax[1].P * u.ax[1].ncells;
            return;
        }
    }
    int Px = 0, Qx = 0, Py = 0, Qy = 0;
    if (axis_periodic(t->h_start[0], t->h_rank[0], ax_a[0], ax_b[0], Px, Qx) &&
        axis_periodic(t->h_start[1], t->h_rank[1], ax_a[1], ax_b[1], Py, Qy) && Px == Py && Qx == Qy && !(Px == 2 && Qx == 1)) {
        PeriodicPlan& u = t->periodic;
        u.P = Px;
        u.Q = Qx;
        u.x0 = ax_a[0];
        u.y0 = ax_a[1];
        u.ncx = (ax_b[0] - u.x0) / u.P;
        u.ncy = (ax_b[1] - u.y0) / u.P;
        if (u.ncx >= 8 && u.ncy >= 2) {
            u.sx0 = t->h_start[0][u.x0];
            u.sy0 = t->h_start[1][u.y0];
            for (int p = 0; p < u.P; ++p) {
                u.ox[p] = t->h_start[0][u.x0 + p] - u.sx0;
                u.oy[p] = t->h_start[1][u.y0 + p] - u.sy0;
            }
            for (int py = 0; py < u.P; ++py)
                for (int px = 0; px < u.P; ++px)
                    u.wblock[py][px] = t->h_rank[1][u.y0 + py] * nrx + t->h_rank[0][u.x0 + px];
            u.ok = true;
            // the polyphase kernel is selected in jinc_resize.cu when it supports this (fs, P, Q)
            t->fast_path = JINC_PATH_PERIODIC;
            t->ix0 = u.x0;
            t->ix1 = u.x0 + u.P * u.ncx;
            t->iy0 = u.y0;
            t->iy1 = u.y0 + u.P * u.ncy;
        }
    }
}

// Tightest tap-mask variant of fs whose (ox1, oy1) is the table's and whose live columns contain every non-zero weight
template <int FS, int M = 1>
void pick_up2x_taps(const uint32_t (&nz)[2][2][FS], Up2xPlan& u)
{
    if constexpr (M < jinc_rs::UP_TAP_VARIANTS) {
        using K = jinc_rs::UpTaps<FS, M>;
        bool fits = K::OX1 == u.ox1 && K::OY1 == u.oy1;
        int live = 0;
        for (int py = 0; py < 2; ++py)
            for (int px = 0; px < 2; ++px)
                for (int ly = 0; ly < FS; ++ly) {
                    fits = fits && (nz[py][px][ly] & ~K::cols(py, px, ly)) == 0;
                    live += __builtin_popcount(K::cols(py, px, ly));
                }
        if (fits && live < u.live_taps) {
            u.taps = M;
            u.live_taps = live;
        }
        pick_up2x_taps<FS, M + 1>(nz, u);
    }
}

template <int FS>
void plan_up2x_taps_fs(const jinc_table* t, Up2xPlan& u)
{
    uint32_t nz[2][2][FS] = {}; // [py][px][ly]: bit lx set when that weight is not exactly zero
    for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px) {
            const float* blk = t->h_weights.data() + (size_t)u.wblock[py][px] * FS * FS;
            for (int ly = 0; ly < FS; ++ly)
                for (int lx = 0; lx < FS; ++lx)
                    nz[py][px][ly] |= (blk[ly * FS + lx] != 0.f ? 1u : 0u) << lx;
        }
    pick_up2x_taps<FS>(nz, u);
}

// The exact-2x kernel of integer planes skips the taps a compiled mask marks as zero (jinc_up2x_taps.h).  A mask is
// used only when every weight it skips is exactly zero in this table, so the choice can cost speed but never change a
// result.  JINCRESIZE_B200_UP2X_ZERO_TAPS=0 keeps every tap (the byte-identity reference of the tests).
void plan_up2x_taps(jinc_table* t)
{
    Up2xPlan& u = t->up2x;
    const int fs = t->sc.fs;
    u.taps = 0;
    u.live_taps = 4 * fs * fs;
    if (t->fast_path != JINC_PATH_UP2X || t->h_weights.empty())
        return;
    const char* off = getenv("JINCRESIZE_B200_UP2X_ZERO_TAPS");
    if (off && off[0] == '0')
        return;
    if (fs == 7)
        plan_up2x_taps_fs<7>(t, u);
    else if (fs == 9)
        plan_up2x_taps_fs<9>(t, u);
}

} // namespace

int jinc_table_build_device(jinc_table* t, const double* lut)
{
    const TableScalars& s = t->sc;
    cudaStream_t st = t->ctx->stream;
    JINC_CUDA(cudaSetDevice(t->ctx->device));

    // LUT as the float values Lut::GetFactor returns (:277-282)
    float lut_f[JINC_LUT_SAMPLES];
    for (int i = 0; i < JINC_LUT_SAMPLES; ++i)
        lut_f[i] = static_cast<float>(lut[i]);
    if (int rc = dev_alloc(&t->d_lut, JINC_LUT_SAMPLES))
        return rc;
    JINC_CUDA(cudaMemcpyAsync(t->d_lut, lut_f, sizeof(lut_f), cudaMemcpyHostToDevice, st));

    int32_t* d_nrank = nullptr;
    if (int rc = dev_alloc(&d_nrank, 2))
        return rc;
    struct FreeOnExit {
        int32_t*& p;
        ~FreeOnExit() { cudaFree(p); }
    } free_nrank{d_nrank};
    const int n_of[2] = {s.dst_w, s.dst_h}, src_of[2] = {s.src_w, s.src_h}, quant_of[2] = {s.quant_x, s.quant_y};
    AxisKernelArgs args[2];
    for (int k = 0; k < 2; ++k) {
        AxisArrays& a = t->ax[k];
        a.n = n_of[k];
        int rc = 0;
        rc = rc ? rc : dev_alloc(&a.pos, a.n);
        rc = rc ? rc : dev_alloc(&a.start, a.n);
        rc = rc ? rc : dev_alloc(&a.qint, a.n);
        rc = rc ? rc : dev_alloc(&a.phase, a.n);
        rc = rc ? rc : dev_alloc(&a.rank, a.n);
        rc = rc ? rc : dev_alloc(&a.border, a.n);
        rc = rc ? rc : dev_alloc(&a.rep, 256);
        rc = rc ? rc : dev_alloc(&a.rank_of, 256);
        rc = rc ? rc : dev_alloc(&a.rep_d2, (size_t)quant_of[k] * s.fs);
        if (rc)
            return rc;
        args[k] = AxisKernelArgs{a.pos, a.start, a.qint, a.phase, a.rank, a.border, a.rep, a.rank_of, a.rep_d2,
                                 d_nrank + k, a.n, src_of[k], quant_of[k], s.fs, s.pos0[k], s.pos_step[k], s.support,
                                 s.filt_step[k]};
    }
    axis_kernel<<<2, kAxisThreads, 0, st>>>(args[0], args[1]);
    JINC_CUDA(cudaGetLastError());

    int32_t h_nrank[2] = {0, 0};
    JINC_CUDA(cudaMemcpyAsync(h_nrank, d_nrank, sizeof(h_nrank), cudaMemcpyDeviceToHost, st));
    for (int k = 0; k < 2; ++k) {
        const int n = n_of[k];
        t->h_start[k].resize(n);
        t->h_phase[k].resize(n);
        t->h_rank[k].resize(n);
        t->h_qint[k].resize(n);
        t->h_border[k].resize(n);
        t->h_pos[k].resize(n);
        JINC_CUDA(cudaMemcpyAsync(t->h_start[k].data(), t->ax[k].start, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        JINC_CUDA(cudaMemcpyAsync(t->h_phase[k].data(), t->ax[k].phase, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        JINC_CUDA(cudaMemcpyAsync(t->h_rank[k].data(), t->ax[k].rank, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        JINC_CUDA(cudaMemcpyAsync(t->h_qint[k].data(), t->ax[k].qint, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        JINC_CUDA(cudaMemcpyAsync(t->h_border[k].data(), t->ax[k].border, n * sizeof(uint8_t), cudaMemcpyDeviceToHost, st));
        JINC_CUDA(cudaMemcpyAsync(t->h_pos[k].data(), t->ax[k].pos, n * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    JINC_CUDA(cudaStreamSynchronize(st));
    t->ax[0].n_rank = h_nrank[0];
    t->ax[1].n_rank = h_nrank[1];

    const size_t n_blocks = (size_t)h_nrank[0] * h_nrank[1];
    const size_t taps = (size_t)s.fs * s.fs;
    if (n_blocks > 0) {
        if (int rc = dev_alloc(&t->d_weights, n_blocks * taps))
            return rc;
        phase_blocks_kernel<<<(unsigned)n_blocks, 128, 0, st>>>(t->d_weights, t->ax[0].rep_d2, t->ax[1].rep_d2, t->d_lut,
                                                               h_nrank[0], s.fs, s.radius2, s.idx_scale);
        JINC_CUDA(cudaGetLastError());
    }
    // border strips and their per-pixel normalisers
    {
        int ax_a[2], ax_b[2];
        for (int k = 0; k < 2; ++k)
            interior_run(t->h_border[k], ax_a[k], ax_b[k]);
        BorderGeom& g = t->bgeom;
        g.W = s.dst_w;
        g.H = s.dst_h;
        g.bx0 = ax_a[0];
        g.bx1 = ax_b[0];
        g.by0 = ax_a[1];
        g.by1 = ax_b[1];
        const long long core_h = g.by1 - g.by0;
        g.off_bottom = (long long)g.by0 * g.W;
        g.off_left = g.off_bottom + (long long)(g.H - g.by1) * g.W;
        g.off_right = g.off_left + core_h * g.bx0;
        g.total = g.off_right + core_h * (g.W - g.bx1);
        if (g.total > 0) {
            if (int rc = dev_alloc(&t->d_border_sum, (size_t)g.total))
                return rc;
            // Border weights are frame-invariant: keep them resident (what the reference's table holds on the host).
            // First try to fold the border pixels into classes of identical blocks.  A tap's distance is
            // fl(c - (start + l)) with c the clamped position (:485-486); c - start is exactly representable
            // (0 <= c - start <= c, a multiple of ulp(c)), so two pixels whose c - start agree on an axis have the same
            // distances on that axis, hence -- when both axes agree -- the same factors, divider and weights.
            std::vector<int32_t> cls[2];
            for (int k = 0; k < 2; ++k) {
                const int n = k == 0 ? s.dst_w : s.dst_h;
                const float hi = static_cast<float>((k == 0 ? s.src_w : s.src_h) - 1);
                std::unordered_map<uint32_t, int32_t> ids;
                cls[k].resize(n);
                for (int i = 0; i < n; ++i) {
                    float c = t->h_pos[k][i] > hi ? hi : t->h_pos[k][i];
                    c = c < 0.f ? 0.f : c;
                    const float delta = c - static_cast<float>(t->h_start[k][i]);
                    uint32_t bits;
                    memcpy(&bits, &delta, sizeof(bits));
                    cls[k][i] = ids.emplace(bits, static_cast<int32_t>(ids.size())).first->second;
                }
            }
            std::vector<int32_t> block_of(static_cast<size_t>(g.total));
            std::vector<int2> reps;
            {
                std::unordered_map<uint64_t, int32_t> blocks;
                auto visit = [&](int x, int y) {
                    const uint64_t key = (static_cast<uint64_t>(static_cast<uint32_t>(cls[1][y])) << 32) | static_cast<uint32_t>(cls[0][x]);
                    auto it = blocks.find(key);
                    if (it == blocks.end()) {
                        it = blocks.emplace(key, static_cast<int32_t>(reps.size())).first;
                        reps.push_back(make_int2(x, y));
                    }
                    block_of[static_cast<size_t>(jinc_border_slot(g, x, y))] = it->second;
                };
                for (int y = 0; y < g.H; ++y) {
                    if (y < g.by0 || y >= g.by1) {
                        for (int x = 0; x < g.W; ++x)
                            visit(x, y);
                    } else {
                        for (int x = 0; x < g.bx0; ++x)
                            visit(x, y);
                        for (int x = g.bx1; x < g.W; ++x)
                            visit(x, y);
                    }
                }
            }
            const size_t taps_n = static_cast<size_t>(s.fs) * s.fs;
            const bool use_classes = reps.size() * 4 <= static_cast<size_t>(g.total) && reps.size() * taps_n * sizeof(float) <= ((size_t)256 << 20);
            size_t free_b = 0, total_b = 0;
            cudaMemGetInfo(&free_b, &total_b);
            if (!use_classes) {
                const size_t bw_bytes = (size_t)((g.total + 31) / 32 * 32) * taps_n * sizeof(float);
                if (bw_bytes <= kBorderWeightBudget && bw_bytes < free_b / 4) {
                    if (cudaMalloc(reinterpret_cast<void**>(&t->d_border_w), bw_bytes) != cudaSuccess) {
                        cudaGetLastError();
                        t->d_border_w = nullptr;
                    }
                }
            }
            BorderSumArgs ba{g, t->ax[0].pos, t->ax[1].pos, t->ax[0].start, t->ax[1].start, t->d_lut, t->d_border_sum,
                             t->d_border_w, s.fs, s.src_w, s.src_h, s.filt_step[0], s.filt_step[1], s.radius2, s.idx_scale};
            border_sum_kernel<<<(unsigned)((g.total + 255) / 256), 256, 0, st>>>(ba);
            JINC_CUDA(cudaGetLastError());
            if (use_classes) {
                int2* d_reps = nullptr;
                if (int rc = dev_alloc(&d_reps, reps.size()))
                    return rc;
                int rc = dev_alloc(&t->d_border_block, static_cast<size_t>(g.total));
                const size_t wb_floats = reps.size() * s.fs * static_cast<size_t>((s.fs + 3) & ~3);
                rc = rc ? rc : dev_alloc(&t->d_border_wb, wb_floats);
                if (rc) {
                    cudaFree(d_reps);
                    return rc;
                }
                t->n_border_blocks = static_cast<int>(reps.size());
                JINC_CUDA(cudaMemsetAsync(t->d_border_wb, 0, wb_floats * sizeof(float), st));
                JINC_CUDA(cudaMemcpyAsync(d_reps, reps.data(), reps.size() * sizeof(int2), cudaMemcpyHostToDevice, st));
                JINC_CUDA(cudaMemcpyAsync(t->d_border_block, block_of.data(), block_of.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
                border_class_kernel<<<(unsigned)reps.size(), 128, 0, st>>>(ba, d_reps, t->d_border_wb);
                JINC_CUDA(cudaGetLastError());
                JINC_CUDA(cudaStreamSynchronize(st)); // reps is a host temporary
                cudaFree(d_reps);
                t->h_border_block = std::move(block_of);
            }
        }
    }
    plan_fast_paths(t);
    if (t->cells.ok) {
        if (int rc = upload_cells_axis(t->cells.ax[0], st))
            return rc;
        if (int rc = upload_cells_axis(t->cells.ax[1], st))
            return rc;
    }
    // the fast paths take their (few) phase blocks as kernel parameters: keep a host copy of those
    if (n_blocks > 0 && n_blocks <= 16) {
        t->h_weights.resize(n_blocks * taps);
        JINC_CUDA(cudaMemcpyAsync(t->h_weights.data(), t->d_weights, n_blocks * taps * sizeof(float),
                                  cudaMemcpyDeviceToHost, st));
    }
    JINC_CUDA(cudaStreamSynchronize(st));
    plan_up2x_taps(t);
    if (n_blocks > 0 && (s.fs & 3) != 0) {
        // the strip role and the general kernel read weight rows as 16-byte vectors: a second copy with padded rows,
        // [block][fs][fsp], while it fits the budget (many-phase tables reach 65536 blocks)
        const int fsp = (s.fs + 3) & ~3;
        const size_t padded_floats = n_blocks * s.fs * fsp;
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        if (padded_floats * sizeof(float) <= kPaddedWeightBudget && padded_floats * sizeof(float) < free_b / 4) {
            if (int rc = dev_alloc(&t->d_weights_p, padded_floats))
                return rc;
            const size_t rows = n_blocks * s.fs;
            pad_rows_kernel<<<(unsigned)((rows * fsp + 255) / 256), 256, 0, st>>>(t->d_weights_p, t->d_weights, rows, s.fs, fsp);
            JINC_CUDA(cudaGetLastError());
            JINC_CUDA(cudaStreamSynchronize(st));
        }
    }
    if (t->bgeom.total >= (1ll << 31))
        return jinc_fail(JINC_E_UNSUPPORTED, "jinc_table: %lld border pixels exceed the 32-bit slot index", t->bgeom.total);
    return jinc_build_strip_plan(t);
}

cudaError_t jinc_gather_blocks(float* out, const uint32_t* list, unsigned n, const float* phase_blocks, const float* border_blocks,
                               int block_floats, cudaStream_t st)
{
    gather_blocks_kernel<<<n, 128, 0, st>>>(out, list, phase_blocks, border_blocks, block_floats);
    return cudaGetLastError();
}

// ================================================================ C ABI: tables

extern "C" int jinc_table_create(jinc_ctx* ctx, const jinc_table_params* p, jinc_table** out)
{
    if (!ctx || !p || !out)
        return jinc_fail(JINC_E_INVALID, "jinc_table_create: null argument");
    *out = nullptr;
    if (p->quant_x < 1 || p->quant_x > 256 || p->quant_y < 1 || p->quant_y > 256)
        return jinc_fail(JINC_E_INVALID, "jinc_table_create: quant must be between 1..256");
    if (p->src_w < 1 || p->src_h < 1 || p->dst_w < 1 || p->dst_h < 1)
        return jinc_fail(JINC_E_INVALID, "jinc_table_create: plane dimensions must be positive");
    if (!(p->radius > 0.0) || !(p->crop_w > 0.0) || !(p->crop_h > 0.0))
        return jinc_fail(JINC_E_INVALID, "jinc_table_create: radius and crop size must be positive");

    const auto t_begin = std::chrono::steady_clock::now();
    auto* t = new jinc_table();
    t->ctx = ctx;
    t->params = *p;
    derive_scalars(*p, t->sc);
    if (t->sc.fs > p->src_w || t->sc.fs > p->src_h) {
        // The reference reads outside the plane here (clamped window still fs wide, :395-418).
        const int fs = t->sc.fs;
        delete t;
        return jinc_fail(JINC_E_UNSUPPORTED, "JincResize: the %dx%d filter window is larger than the %dx%d source plane",
                         fs, fs, p->src_w, p->src_h);
    }
    double lut[JINC_LUT_SAMPLES];
    jinc_lut_build_host(p->radius, p->blur, lut);
    const int rc = jinc_table_build_device(t, lut);
    if (rc != JINC_OK) {
        jinc_table_destroy(t);
        return rc;
    }
    t->build_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    *out = t;
    return JINC_OK;
}

extern "C" void jinc_table_destroy(jinc_table* t)
{
    if (!t)
        return;
    cudaSetDevice(t->ctx->device);
    for (AxisArrays& a : t->ax) {
        cudaFree(a.pos);
        cudaFree(a.start);
        cudaFree(a.qint);
        cudaFree(a.phase);
        cudaFree(a.rank);
        cudaFree(a.border);
        cudaFree(a.rep);
        cudaFree(a.rank_of);
        cudaFree(a.rep_d2);
    }
    for (CellsAxis& c : t->cells.ax) {
        cudaFree(c.d_cell);
        cudaFree(c.d_i0);
        cudaFree(c.d_n);
        cudaFree(c.d_org);
        cudaFree(c.d_rank);
    }
    cudaFree(t->d_lut);
    cudaFree(t->d_weights);
    cudaFree(t->d_weights_p);
    cudaFree(t->d_border_sum);
    cudaFree(t->d_border_w);
    cudaFree(t->d_border_block);
    cudaFree(t->d_border_wb);
    jinc_free_strip_plan(t);
    delete t;
}

extern "C" int jinc_table_get_info(const jinc_table* t, jinc_table_info* info)
{
    if (!t || !info)
        return jinc_fail(JINC_E_INVALID, "jinc_table_get_info: null argument");
    memset(info, 0, sizeof(*info));
    info->filter_size = t->sc.fs;
    info->n_phase_x = t->ax[0].n_rank;
    info->n_phase_y = t->ax[1].n_rank;
    for (uint8_t b : t->h_border[0])
        info->n_border_cols += b;
    for (uint8_t b : t->h_border[1])
        info->n_border_rows += b;
    info->fast_path = t->fast_path;
    info->interior_x0 = t->ix0;
    info->interior_x1 = t->ix1;
    info->interior_y0 = t->iy0;
    info->interior_y1 = t->iy1;
    info->filter_support = t->sc.support;
    info->build_ms = t->build_ms;
    info->up2x_taps = t->fast_path == JINC_PATH_UP2X ? t->up2x.live_taps : 0;
    return JINC_OK;
}

extern "C" int jinc_table_axis(const jinc_table* t, int axis, int32_t* start, int32_t* phase, uint8_t* border, float* pos)
{
    if (!t || axis < 0 || axis > 1)
        return jinc_fail(JINC_E_INVALID, "jinc_table_axis: bad argument");
    const size_t n = t->h_start[axis].size();
    if (start)
        memcpy(start, t->h_start[axis].data(), n * sizeof(int32_t));
    if (phase)
        memcpy(phase, t->h_phase[axis].data(), n * sizeof(int32_t));
    if (border)
        memcpy(border, t->h_border[axis].data(), n);
    if (pos)
        memcpy(pos, t->h_pos[axis].data(), n * sizeof(float));
    return JINC_OK;
}

extern "C" int jinc_table_pixel_block(const jinc_table* t, int x, int y, int64_t* block_id)
{
    if (!t || !block_id || x < 0 || y < 0 || x >= t->sc.dst_w || y >= t->sc.dst_h)
        return jinc_fail(JINC_E_INVALID, "jinc_table_pixel_block: bad argument");
    if (t->h_border[0][x] || t->h_border[1][y])
        *block_id = -1 - (static_cast<int64_t>(y) * t->sc.dst_w + x);
    else
        *block_id = static_cast<int64_t>(t->h_rank[1][y]) * t->ax[0].n_rank + t->h_rank[0][x];
    return JINC_OK;
}

extern "C" int jinc_table_pixel_weights(const jinc_table* t, int x, int y, float* weights)
{
    if (!t || !weights || x < 0 || y < 0 || x >= t->sc.dst_w || y >= t->sc.dst_h)
        return jinc_fail(JINC_E_INVALID, "jinc_table_pixel_weights: bad argument");
    return jinc_debug_pixel_weights(t, x, y, weights);
}
