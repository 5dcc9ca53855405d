// jinc_filter.cpp -- device contexts, filter instances and the host<->device frame pipeline.
//
// Replaces the per-plane geometry derivation of Create_JincResize (src/JincResize.cpp:762-866), the
// process_frame step of JincResize_GetFrame (:615) and free_JincResize (:632-647).
//
// Frame pipeline: every GPU of the filter owns `slots_per_device` in-flight slots, each with its own CUDA
// stream, device source/destination buffers and pinned staging buffers laid out identically to the device
// buffers (so one cudaMemcpyAsync moves all planes).  A frame takes a slot (GPUs round-robin), is copied H2D,
// resampled and copied D2H on that slot's stream; concurrent callers (AviSynth Prefetch threads, or
// jinc_filter_submit) therefore overlap PCIe transfers in both directions and kernels across slots and GPUs.
// Caller memory that is page-locked (by the caller, or registered here once a pageable frame buffer comes back:
// jinc_hostmem.h) is moved by DMA directly; only first-seen pageable buffers are staged through the slot's pinned
// mirror, with the copy split over helper threads.  Frames are independent, and so are row bands of one frame
// (jinc_filter_process_bands): there is no inter-GPU traffic and no collective.
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstring>
#include <memory>
#include <mutex>

#include <random>

#include "jinc_hostmem.h"
#include "jinc_internal.h"

// ================================================================ contexts

extern "C" int jinc_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" int jinc_ctx_create(int device, jinc_ctx** out)
{
    if (!out)
        return jinc_fail(JINC_E_INVALID, "jinc_ctx_create: null output");
    *out = nullptr;
    const int n = jinc_device_count();
    if (n == 0)
        return jinc_fail(JINC_E_CUDA, "JincResize: no CUDA device available (this build has no CPU fallback)");
    if (device < 0 || device >= n)
        return jinc_fail(JINC_E_INVALID, "jinc_ctx_create: device %d out of range (0..%d)", device, n - 1);
    JINC_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    JINC_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return jinc_fail(JINC_E_UNSUPPORTED, "JincResize: device %d is sm_%d%d; this library is built for sm_100a only",
                         device, prop.major, prop.minor);
    auto* c = new jinc_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->smem_optin = prop.sharedMemPerBlockOptin;
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete c;
        return jinc_fail(JINC_E_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
    }
    *out = c;
    return JINC_OK;
}

int jinc_ring_launch(jinc_ctx* ctx, const void* host, size_t bytes, cudaStream_t st, const std::function<int(const void*)>& launch)
{
    RecordRing& r = ctx->ring;
    std::lock_guard<std::mutex> lk(r.mu);
    const int slot = r.next;
    r.next = (r.next + 1) % RecordRing::kRing;
    if (!r.done[slot])
        JINC_CUDA(cudaEventCreateWithFlags(&r.done[slot], cudaEventDisableTiming));
    else
        JINC_CUDA(cudaStreamWaitEvent(st, r.done[slot], 0)); // the launch that last read this entry
    if (r.cap[slot] < bytes) {
        JINC_CUDA(cudaEventSynchronize(r.done[slot])); // no-op for a fresh event
        cudaFree(r.ptrs[slot]);
        r.ptrs[slot] = nullptr;
        r.cap[slot] = 0;
        if (cudaMalloc(reinterpret_cast<void**>(&r.ptrs[slot]), bytes) != cudaSuccess)
            return jinc_fail(JINC_E_NOMEM, "plane records: cudaMalloc(%zu) failed", bytes);
        r.cap[slot] = bytes;
    }
    // pageable source: staged by the runtime before the call returns, ordered before the kernel on `st`
    JINC_CUDA(cudaMemcpyAsync(r.ptrs[slot], host, bytes, cudaMemcpyHostToDevice, st));
    const int rc = launch(r.ptrs[slot]);
    JINC_CUDA(cudaEventRecord(r.done[slot], st));
    return rc;
}

void jinc_ring_free(jinc_ctx* ctx)
{
    RecordRing& r = ctx->ring;
    for (int k = 0; k < RecordRing::kRing; ++k) {
        if (r.done[k]) {
            cudaEventSynchronize(r.done[k]);
            cudaEventDestroy(r.done[k]);
            r.done[k] = nullptr;
        }
        cudaFree(r.ptrs[k]);
        r.ptrs[k] = nullptr;
        r.cap[k] = 0;
    }
}

extern "C" void jinc_ctx_destroy(jinc_ctx* ctx)
{
    if (!ctx)
        return;
    cudaSetDevice(ctx->device);
    jinc_ring_free(ctx);
    if (ctx->stream)
        cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" int jinc_ctx_device(const jinc_ctx* ctx) { return ctx ? ctx->device : -1; }

// ================================================================ filter

namespace {

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct PlaneLayout {
    int table = 0;          // which table (0 luma / shared, 1 subsampled chroma)
    int src_w = 0, src_h = 0, dst_w = 0, dst_h = 0;
    size_t src_off = 0, dst_off = 0; // byte offsets inside the slot buffers
    size_t src_pitch = 0, dst_pitch = 0;
};

// bytes written into a directly addressed destination plane before the transfers are enqueued; still there afterwards
// means the transfer went elsewhere (stale registration of a buffer the host has freed and re-mapped)
struct Sentinel {
    unsigned char* at = nullptr;
    uint64_t value = 0;
};
constexpr int kSentinelsPerPlane = 2;

struct Slot {
    enum State { FREE, BUSY, WAITING };
    int dev_index = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    unsigned char* d_src = nullptr;
    unsigned char* d_dst = nullptr;
    unsigned char* h_src = nullptr; // pinned
    unsigned char* h_dst = nullptr; // pinned
    State state = FREE;
    int64_t ticket = -1;
    jinc_frame pending{}; // the frame of an outstanding enqueue
    bool dst_direct = false;
    jinc_hostmem::Pin src_pin, dst_pin;
    Sentinel sentinel[JINC_MAX_PLANES * kSentinelsPerPlane];
    int n_sentinels = 0;
    // the unlocked head and tail of a registered destination buffer arrive in the pinned mirror and are copied out by the CPU
    struct Fixup {
        unsigned char* dst;
        const unsigned char* src;
        size_t n;
    } fixup[2 * JINC_MAX_PLANES + 2];
    int n_fixups = 0;
    // probe words of the uploaded source, read back when the source moved through a registration made here
    uint32_t* d_probe = nullptr;
    uint32_t* h_probe = nullptr; // pinned
    uint32_t probe_seed = 0;
    bool probe_active = false;
    int src_row0[JINC_MAX_PLANES] = {}, src_row1[JINC_MAX_PLANES] = {}; // source rows uploaded per plane
    float antiring = 0.f; // anti-ringing strength of the pending frame (captured when it was submitted)
};

constexpr int kRedoStaged = 1; // finish_frame: a registration turned out stale -- run the frame again through the mirrors

struct DeviceState {
    jinc_ctx* ctx = nullptr;
    jinc_table* tables[2] = {nullptr, nullptr};
};

// rows of one plane between host and device.  `linear`: both sides have the same pitch and the bytes between rows may be
// carried along, so ONE extent moves (the DMA engine takes a single descriptor instead of one per row); else a 2-D copy.
cudaError_t copy_plane_async(void* dst, size_t dst_pitch, const void* src, size_t src_pitch, size_t row_bytes, int rows, bool linear,
                             cudaMemcpyKind kind, cudaStream_t st)
{
    if (linear && dst_pitch == src_pitch)
        return cudaMemcpyAsync(dst, src, dst_pitch * static_cast<size_t>(rows - 1) + row_bytes, kind, st);
    return cudaMemcpy2DAsync(dst, dst_pitch, src, src_pitch, row_bytes, static_cast<size_t>(rows), kind, st);
}

std::atomic<int64_t> g_direct_src{0}, g_direct_dst{0}, g_staged{0};
std::atomic<int> g_live_filters{0};

uint64_t fresh_nonce()
{
    static std::atomic<uint64_t> ctr{[] {
        std::random_device rd;
        return (static_cast<uint64_t>(rd()) << 32) ^ rd();
    }()};
    uint64_t z = ctr.fetch_add(0x9E3779B97F4A7C15ull) + 0x9E3779B97F4A7C15ull; // splitmix64
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

} // namespace

struct jinc_filter {
    jinc_filter_params p{};
    float peak = 0.f;
    int n_tables = 1;
    jinc_table_params tparams[2]{};
    PlaneLayout planes[JINC_MAX_PLANES];
    size_t src_bytes = 0, dst_bytes = 0;
    std::vector<DeviceState> devs;
    std::vector<std::unique_ptr<Slot>> slots;
    std::mutex mu;
    std::condition_variable cv;
    int64_t next_ticket = 0; // under mu
    std::atomic<int64_t> rr{0};
    std::atomic<int64_t> launches{0};
    std::atomic<float> antiring{0.f}; // jinc_filter_set_antiring; each frame reads it once, when it is submitted
    bool registers = false; // counted as a client of the host-buffer registry
};

namespace {

// Create_JincResize geometry (:762-770 crop, :833-862 chroma shift).  cplace only matters for subsampled chroma.
void derive_table_params(const jinc_filter_params& p, jinc_table_params out[2], int* n_tables)
{
    double crop_w = p.src_width, crop_h = p.src_height;
    if (crop_w <= 0.0)
        crop_w = p.src_w - p.src_left + crop_w;
    if (crop_h <= 0.0)
        crop_h = p.src_h - p.src_top + crop_h;
    const double radius = jinc_radius_for_tap(p.tap);

    jinc_table_params& y = out[0];
    y.quant_x = p.quant_x;
    y.quant_y = p.quant_y;
    y.src_w = p.src_w;
    y.src_h = p.src_h;
    y.dst_w = p.target_w;
    y.dst_h = p.target_h;
    y.radius = radius;
    y.blur = p.blur;
    y.crop_left = p.src_left;
    y.crop_top = p.src_top;
    y.crop_w = crop_w;
    y.crop_h = crop_h;
    *n_tables = 1;
    if (p.n_planes < 2 || (p.sub_w == 0 && p.sub_h == 0))
        return;

    // The half-sample shift of co-sited chroma uses the FULL source/target widths, not the crop window (:838-841).
    const double div_w = static_cast<double>(1 << p.sub_w), div_h = static_cast<double>(1 << p.sub_h);
    const bool left_sited = p.cplace == JINC_CPLACE_MPEG2 || p.cplace == JINC_CPLACE_TOPLEFT;
    const bool top_sited = p.cplace == JINC_CPLACE_TOPLEFT;
    jinc_table_params& c = out[1];
    c = y;
    c.src_w = p.src_w >> p.sub_w;
    c.src_h = p.src_h >> p.sub_h;
    c.dst_w = p.target_w >> p.sub_w;
    c.dst_h = p.target_h >> p.sub_h;
    c.crop_left = left_sited ? (0.5 * (1.0 - static_cast<double>(p.src_w) / p.target_w) + p.src_left) / div_w
                             : p.src_left / div_w;
    c.crop_top = top_sited ? (0.5 * (1.0 - static_cast<double>(p.src_h) / p.target_h) + p.src_top) / div_h
                           : p.src_top / div_h;
    c.crop_w = crop_w / div_w;
    c.crop_h = crop_h / div_h;
    *n_tables = 2;
}

void release_slot(jinc_filter* f, Slot* s)
{
    jinc_hostmem::release(&s->src_pin);
    jinc_hostmem::release(&s->dst_pin);
    {
        std::lock_guard<std::mutex> lk(f->mu);
        s->state = Slot::FREE;
        s->ticket = -1;
    }
    f->cv.notify_all();
}

// f->mu held: a free slot, on GPU `want` if it has one (`only`: on no other GPU)
Slot* find_free_slot(jinc_filter* f, int want, bool only)
{
    Slot* any = nullptr;
    for (auto& s : f->slots) {
        if (s->state != Slot::FREE)
            continue;
        if (s->dev_index == want)
            return s.get();
        if (!any)
            any = s.get();
    }
    return only ? nullptr : any;
}

// Take a free slot, preferring GPU (n mod G) so consecutive frames spread over all GPUs; the slot's ticket is assigned
// under the lock.  block = false: nullptr when every slot is taken.
Slot* acquire_slot(jinc_filter* f, bool block)
{
    const int nd = static_cast<int>(f->devs.size());
    const int want = static_cast<int>(f->rr.fetch_add(1) % nd);
    std::unique_lock<std::mutex> lk(f->mu);
    for (;;) {
        if (Slot* s = find_free_slot(f, want, false)) {
            s->state = Slot::BUSY;
            s->ticket = f->next_ticket++;
            return s;
        }
        if (!block)
            return nullptr;
        f->cv.wait(lk);
    }
}

// the whole plane as the caller describes it (registration keys must not depend on the band being processed)
bool plane_range(const void* base, ptrdiff_t pitch, size_t row_bytes, int rows, jinc_hostmem::Range* r)
{
    if (pitch < static_cast<ptrdiff_t>(row_bytes) || rows < 1)
        return false; // bottom-up or overlapping rows: staged
    r->lo = static_cast<const unsigned char*>(base);
    r->hi = r->lo + static_cast<size_t>(pitch) * (rows - 1) + row_bytes;
    return true;
}

// Enqueue H2D + kernels + D2H for output rows [y0,y1) (luma rows) of `frame` on slot s, with anti-ringing strength
// `antiring` (0: off).  staged_only: do not address the caller's memory by DMA at all (the retry after a stale registration
// was found).
int enqueue_frame(jinc_filter* f, Slot* s, const jinc_frame* frame, int y0_luma, int y1_luma, bool whole, float antiring,
                  bool staged_only = false)
{
    DeviceState& d = f->devs[s->dev_index];
    JINC_CUDA(cudaSetDevice(d.ctx->device));
    const int sb = jinc_sample_size(f->p.sample_bytes); // bytes per sample
    const int np = f->p.n_planes;
    const bool may_register = (f->p.flags & JINC_FILTER_HOST_REGISTER) != 0;
    s->probe_active = false;
    const bool padding_ok = (f->p.flags & JINC_FILTER_DST_PADDING_WRITABLE) != 0;
    s->pending = *frame;
    s->antiring = antiring;
    s->n_sentinels = 0;

    // per plane: the output rows of this band and the source rows its windows reach
    int sy0[JINC_MAX_PLANES], sy1[JINC_MAX_PLANES], oy0[JINC_MAX_PLANES], oy1[JINC_MAX_PLANES];
    for (int i = 0; i < np; ++i) {
        const PlaneLayout& pl = f->planes[i];
        const jinc_table* t = d.tables[pl.table];
        const int shift = (pl.table == 1) ? f->p.sub_h : 0;
        oy0[i] = whole ? 0 : (y0_luma >> shift);
        oy1[i] = whole ? pl.dst_h : std::min(pl.dst_h, (y1_luma + (1 << shift) - 1) >> shift);
        if (whole) {
            sy0[i] = 0;
            sy1[i] = pl.src_h;
        } else {
            int lo = pl.src_h, hi = 0;
            for (int y = oy0[i]; y < oy1[i]; ++y) {
                lo = std::min(lo, t->h_start[1][y]);
                hi = std::max(hi, t->h_start[1][y] + t->sc.fs);
            }
            sy0[i] = std::max(lo, 0);
            sy1[i] = std::min(hi, pl.src_h);
        }
        s->src_row0[i] = sy0[i];
        s->src_row1[i] = sy1[i];
    }

    // One contiguous extent between the caller's memory and the device buffer.  Only the page-locked part of the caller's
    // buffer is addressed by DMA; the (sub-page) head and tail of a buffer registered here go through the slot's pinned
    // mirror, which has the device buffer's layout.
    auto h2d = [&](unsigned char* dev, const unsigned char* host, size_t n) -> cudaError_t {
        size_t a = 0, b = 0;
        jinc_hostmem::direct_part(s->src_pin, host, n, &a, &b);
        unsigned char* mir = s->h_src + (dev - s->d_src);
        cudaError_t e = cudaSuccess;
        if (b <= a) {
            memcpy(mir, host, n);
            return cudaMemcpyAsync(dev, mir, n, cudaMemcpyHostToDevice, s->stream);
        }
        if (a > 0) {
            memcpy(mir, host, a);
            e = cudaMemcpyAsync(dev, mir, a, cudaMemcpyHostToDevice, s->stream);
        }
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(dev + a, host + a, b - a, cudaMemcpyHostToDevice, s->stream);
        if (e == cudaSuccess && b < n) {
            memcpy(mir + b, host + b, n - b);
            e = cudaMemcpyAsync(dev + b, mir + b, n - b, cudaMemcpyHostToDevice, s->stream);
        }
        return e;
    };
    auto d2h = [&](unsigned char* host, const unsigned char* dev, size_t n, bool check_arrival) -> cudaError_t {
        size_t a = 0, b = 0;
        jinc_hostmem::direct_part(s->dst_pin, host, n, &a, &b);
        unsigned char* mir = s->h_dst + (dev - s->d_dst);
        cudaError_t e = cudaSuccess;
        if (b <= a) {
            s->fixup[s->n_fixups++] = Slot::Fixup{host, mir, n};
            return cudaMemcpyAsync(mir, dev, n, cudaMemcpyDeviceToHost, s->stream);
        }
        if (check_arrival && b - a >= 2 * sizeof(uint64_t)) {
            // arrival check: sentinels at both ends of the directly addressed part must be overwritten by the transfer
            unsigned char* at[2] = {host + a, host + b - sizeof(uint64_t)};
            for (unsigned char* q : at) {
                Sentinel& sn = s->sentinel[s->n_sentinels++];
                sn.at = q;
                sn.value = fresh_nonce();
                memcpy(sn.at, &sn.value, sizeof(sn.value));
            }
        }
        if (a > 0) {
            s->fixup[s->n_fixups++] = Slot::Fixup{host, mir, a};
            e = cudaMemcpyAsync(mir, dev, a, cudaMemcpyDeviceToHost, s->stream);
        }
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(host + a, dev + a, b - a, cudaMemcpyDeviceToHost, s->stream);
        if (e == cudaSuccess && b < n) {
            s->fixup[s->n_fixups++] = Slot::Fixup{host + b, mir + b, n - b};
            e = cudaMemcpyAsync(mir + b, dev + b, n - b, cudaMemcpyDeviceToHost, s->stream);
        }
        return e;
    };

    // ---- source planes -> device
    jinc_hostmem::Range rs[JINC_MAX_PLANES];
    bool src_direct = !staged_only, src_packed = whole, src_same_pitch = true;
    for (int i = 0; i < np; ++i) {
        const PlaneLayout& pl = f->planes[i];
        src_direct = src_direct && plane_range(frame->src[i], frame->src_pitch[i], static_cast<size_t>(pl.src_w) * sb, pl.src_h, &rs[i]);
        const bool same = frame->src_pitch[i] == static_cast<ptrdiff_t>(pl.src_pitch);
        src_same_pitch = src_same_pitch && same;
        src_packed = src_packed && same &&
                     static_cast<const unsigned char*>(frame->src[i]) - static_cast<const unsigned char*>(frame->src[0]) ==
                         static_cast<ptrdiff_t>(pl.src_off);
    }
    // memory registered here is moved as whole extents (its unlocked ends are split off), which needs the pipeline's pitch;
    // memory the caller allocated page-locked may have any pitch (2-D copies)
    src_direct = src_direct && jinc_hostmem::acquire(rs, np, may_register && src_same_pitch, d.ctx->device, &s->src_pin);
    if (src_direct && !src_same_pitch && jinc_hostmem::registered_here(&s->src_pin)) {
        jinc_hostmem::release(&s->src_pin);
        src_direct = false;
    }
    if (src_direct) {
        g_direct_src.fetch_add(1, std::memory_order_relaxed);
        s->probe_active = jinc_hostmem::registered_here(&s->src_pin);
        if (src_packed) {
            // the caller's planes are packed exactly like the slot (AviSynth+ frame buffers are): one extent per frame
            const PlaneLayout& last = f->planes[np - 1];
            const size_t bytes = last.src_off + last.src_pitch * (last.src_h - 1) + static_cast<size_t>(last.src_w) * sb;
            JINC_CUDA(h2d(s->d_src, static_cast<const unsigned char*>(frame->src[0]), bytes));
        } else {
            for (int i = 0; i < np; ++i) {
                const PlaneLayout& pl = f->planes[i];
                const int rows = sy1[i] - sy0[i];
                if (rows <= 0)
                    continue;
                unsigned char* dev = s->d_src + pl.src_off + static_cast<size_t>(sy0[i]) * pl.src_pitch;
                const unsigned char* host = static_cast<const unsigned char*>(frame->src[i]) + static_cast<ptrdiff_t>(sy0[i]) * frame->src_pitch[i];
                if (src_same_pitch)
                    JINC_CUDA(h2d(dev, host, pl.src_pitch * static_cast<size_t>(rows - 1) + static_cast<size_t>(pl.src_w) * sb));
                else
                    JINC_CUDA(copy_plane_async(dev, pl.src_pitch, host, static_cast<size_t>(frame->src_pitch[i]), static_cast<size_t>(pl.src_w) * sb,
                                               rows, false, cudaMemcpyHostToDevice, s->stream));
            }
        }
    } else {
        // pageable caller memory seen for the first time (or not registrable): stage into the slot's pinned mirror
        g_staged.fetch_add(1, std::memory_order_relaxed);
        for (int i = 0; i < np; ++i) {
            const PlaneLayout& pl = f->planes[i];
            const int rows = sy1[i] - sy0[i];
            if (rows <= 0)
                continue;
            jinc_hostmem::copy_rows(s->h_src + pl.src_off + static_cast<size_t>(sy0[i]) * pl.src_pitch, pl.src_pitch,
                                    static_cast<const unsigned char*>(frame->src[i]) + static_cast<ptrdiff_t>(sy0[i]) * frame->src_pitch[i],
                                    frame->src_pitch[i], static_cast<size_t>(pl.src_w) * sb, rows);
            if (!whole)
                JINC_CUDA(copy_plane_async(s->d_src + pl.src_off + static_cast<size_t>(sy0[i]) * pl.src_pitch, pl.src_pitch,
                                           s->h_src + pl.src_off + static_cast<size_t>(sy0[i]) * pl.src_pitch, pl.src_pitch,
                                           static_cast<size_t>(pl.src_w) * sb, rows, true, cudaMemcpyHostToDevice, s->stream));
        }
        if (whole)
            JINC_CUDA(cudaMemcpyAsync(s->d_src, s->h_src, f->src_bytes, cudaMemcpyHostToDevice, s->stream));
    }

    if (s->probe_active) {
        s->probe_seed = static_cast<uint32_t>(fresh_nonce());
        if (int rc = jinc_launch_probe(s->d_src, static_cast<uint32_t>(f->src_bytes / 4), s->probe_seed, s->d_probe, s->stream))
            return rc;
        f->launches.fetch_add(1);
        JINC_CUDA(cudaMemcpyAsync(s->h_probe, s->d_probe, JINC_PROBE_WORDS * sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
    }

    // ---- kernels: planes that share a table go out in one launch
    for (int k = 0; k < f->n_tables; ++k) {
        const void* src[JINC_MAX_PLANES];
        void* dst[JINC_MAX_PLANES];
        ptrdiff_t sp[JINC_MAX_PLANES], dp[JINC_MAX_PLANES];
        int n = 0, yb = 0, ye = 0;
        for (int i = 0; i < np; ++i) {
            const PlaneLayout& pl = f->planes[i];
            if (pl.table != k)
                continue;
            src[n] = s->d_src + pl.src_off;
            dst[n] = s->d_dst + pl.dst_off;
            sp[n] = static_cast<ptrdiff_t>(pl.src_pitch);
            dp[n] = static_cast<ptrdiff_t>(pl.dst_pitch);
            yb = oy0[i];
            ye = oy1[i];
            ++n;
        }
        if (n == 0)
            continue;
        int launched = 0;
        int rc = jinc_launch_resize_planes(d.ctx, d.tables[k], f->p.sample_bytes, f->peak, n, src, sp, dst, dp, yb, ye, s->stream,
                                            &launched);
        if (rc == JINC_OK && antiring > 0.f)
            rc = jinc_launch_antiring_planes(d.tables[k], f->p.sample_bytes, antiring, n, src, sp, dst, dp, yb, ye, s->stream, &launched);
        f->launches.fetch_add(launched);
        if (rc != JINC_OK)
            return rc;
    }

    // ---- destination planes -> host
    jinc_hostmem::Range rd[JINC_MAX_PLANES];
    bool dst_direct = !staged_only, dst_packed = whole, dst_tight = true, dst_same_pitch = true;
    for (int i = 0; i < np; ++i) {
        const PlaneLayout& pl = f->planes[i];
        const size_t row_bytes = static_cast<size_t>(pl.dst_w) * sb;
        dst_direct = dst_direct && plane_range(frame->dst[i], frame->dst_pitch[i], row_bytes, pl.dst_h, &rd[i]);
        dst_tight = dst_tight && frame->dst_pitch[i] == static_cast<ptrdiff_t>(row_bytes);
        const bool same = frame->dst_pitch[i] == static_cast<ptrdiff_t>(pl.dst_pitch);
        dst_same_pitch = dst_same_pitch && same;
        dst_packed = dst_packed && same &&
                     static_cast<unsigned char*>(frame->dst[i]) - static_cast<unsigned char*>(frame->dst[0]) == static_cast<ptrdiff_t>(pl.dst_off);
    }
    // whole extents may be written only where the bytes between rows (and planes) belong to the frame
    const bool dst_extents = dst_same_pitch && (dst_tight || padding_ok);
    dst_direct = dst_direct && jinc_hostmem::acquire(rd, np, may_register && dst_extents, d.ctx->device, &s->dst_pin);
    const bool dst_ours = dst_direct && jinc_hostmem::registered_here(&s->dst_pin);
    if (dst_ours && !dst_extents) {
        jinc_hostmem::release(&s->dst_pin);
        dst_direct = false;
    }
    s->dst_direct = dst_direct;
    s->n_fixups = 0;
    if (dst_direct) {
        g_direct_dst.fetch_add(1, std::memory_order_relaxed);
        if (dst_packed && dst_extents) {
            const PlaneLayout& last = f->planes[np - 1];
            const size_t bytes = last.dst_off + last.dst_pitch * (last.dst_h - 1) + static_cast<size_t>(last.dst_w) * sb;
            JINC_CUDA(d2h(static_cast<unsigned char*>(frame->dst[0]), s->d_dst, bytes, dst_ours));
        } else {
            for (int i = 0; i < np; ++i) {
                const PlaneLayout& pl = f->planes[i];
                const int rows = oy1[i] - oy0[i];
                if (rows <= 0)
                    continue;
                unsigned char* host = static_cast<unsigned char*>(frame->dst[i]) + static_cast<ptrdiff_t>(oy0[i]) * frame->dst_pitch[i];
                const unsigned char* dev = s->d_dst + pl.dst_off + static_cast<size_t>(oy0[i]) * pl.dst_pitch;
                if (dst_extents)
                    JINC_CUDA(d2h(host, dev, pl.dst_pitch * static_cast<size_t>(rows - 1) + static_cast<size_t>(pl.dst_w) * sb, dst_ours));
                else
                    JINC_CUDA(copy_plane_async(host, static_cast<size_t>(frame->dst_pitch[i]), dev, pl.dst_pitch, static_cast<size_t>(pl.dst_w) * sb,
                                               rows, false, cudaMemcpyDeviceToHost, s->stream));
            }
        }
    } else if (whole) {
        JINC_CUDA(cudaMemcpyAsync(s->h_dst, s->d_dst, f->dst_bytes, cudaMemcpyDeviceToHost, s->stream));
    } else {
        for (int i = 0; i < np; ++i) {
            const PlaneLayout& pl = f->planes[i];
            const int rows = oy1[i] - oy0[i];
            if (rows <= 0)
                continue;
            const size_t off = pl.dst_off + static_cast<size_t>(oy0[i]) * pl.dst_pitch;
            JINC_CUDA(copy_plane_async(s->h_dst + off, pl.dst_pitch, s->d_dst + off, pl.dst_pitch, static_cast<size_t>(pl.dst_w) * sb, rows,
                                       true, cudaMemcpyDeviceToHost, s->stream));
        }
    }
    JINC_CUDA(cudaEventRecord(s->done, s->stream));
    return JINC_OK;
}

// Wait for the slot's work and move staged output rows [y0,y1) (luma) to the caller's planes.
int finish_frame(jinc_filter* f, Slot* s, int y0_luma, int y1_luma, bool whole)
{
    DeviceState& d = f->devs[s->dev_index];
    JINC_CUDA(cudaSetDevice(d.ctx->device));
    JINC_CUDA(cudaEventSynchronize(s->done));
    const int sb = jinc_sample_size(f->p.sample_bytes); // bytes per sample
    if (s->probe_active) {
        // what the GPU received through the registration against what the caller's memory holds now
        const uint32_t n_words = static_cast<uint32_t>(f->src_bytes / 4);
        bool same = true;
        for (int k = 0; k < JINC_PROBE_WORDS && same; ++k) {
            const size_t off = static_cast<size_t>(jinc_probe_index(s->probe_seed, static_cast<uint32_t>(k), n_words)) * 4;
            for (int i = 0; i < f->p.n_planes; ++i) {
                const PlaneLayout& pl = f->planes[i];
                if (off < pl.src_off || off >= pl.src_off + pl.src_pitch * pl.src_h)
                    continue;
                const size_t row = (off - pl.src_off) / pl.src_pitch, col = (off - pl.src_off) % pl.src_pitch;
                if (col + 4 <= static_cast<size_t>(pl.src_w) * sb && static_cast<int>(row) >= s->src_row0[i] && static_cast<int>(row) < s->src_row1[i])
                    same = memcmp(static_cast<const unsigned char*>(s->pending.src[i]) + static_cast<ptrdiff_t>(row) * s->pending.src_pitch[i] + col,
                                  &s->h_probe[k], 4) == 0;
                break;
            }
        }
        s->probe_active = false;
        if (!same) {
            jinc_hostmem::distrust(&s->src_pin);
            if (s->dst_direct && s->n_sentinels > 0)
                jinc_hostmem::distrust(&s->dst_pin); // same host, same habits: take no chances with this frame
            return kRedoStaged;
        }
    }
    bool from_mirror = !s->dst_direct;
    if (s->dst_direct && s->n_sentinels > 0) {
        bool arrived = true;
        for (int k = 0; k < s->n_sentinels; ++k) {
            uint64_t now;
            memcpy(&now, s->sentinel[k].at, sizeof(now));
            arrived = arrived && now != s->sentinel[k].value;
        }
        if (!arrived) {
            // the registration behind this buffer is stale: drop it for good and deliver through the pinned mirror
            jinc_hostmem::distrust(&s->dst_pin);
            JINC_CUDA(cudaMemcpyAsync(s->h_dst, s->d_dst, f->dst_bytes, cudaMemcpyDeviceToHost, s->stream));
            JINC_CUDA(cudaStreamSynchronize(s->stream));
            from_mirror = true;
        }
    }
    if (!from_mirror) {
        for (int k = 0; k < s->n_fixups; ++k)
            memcpy(s->fixup[k].dst, s->fixup[k].src, s->fixup[k].n);
        return JINC_OK;
    }
    for (int i = 0; i < f->p.n_planes; ++i) {
        const PlaneLayout& pl = f->planes[i];
        const int shift = (pl.table == 1) ? f->p.sub_h : 0;
        const int a = whole ? 0 : (y0_luma >> shift);
        const int b = whole ? pl.dst_h : std::min(pl.dst_h, (y1_luma + (1 << shift) - 1) >> shift);
        if (b <= a)
            continue;
        jinc_hostmem::copy_rows(static_cast<unsigned char*>(s->pending.dst[i]) + static_cast<ptrdiff_t>(a) * s->pending.dst_pitch[i],
                                static_cast<size_t>(s->pending.dst_pitch[i]), s->h_dst + pl.dst_off + static_cast<size_t>(a) * pl.dst_pitch,
                                static_cast<ptrdiff_t>(pl.dst_pitch), static_cast<size_t>(pl.dst_w) * sb, b - a);
    }
    return JINC_OK;
}

// finish_frame, and when a stale registration was found, the frame again through the pinned mirrors
int complete_frame(jinc_filter* f, Slot* s, int y0_luma, int y1_luma, bool whole)
{
    int rc = finish_frame(f, s, y0_luma, y1_luma, whole);
    if (rc != kRedoStaged)
        return rc;
    const jinc_frame frame = s->pending;
    jinc_hostmem::release(&s->src_pin);
    jinc_hostmem::release(&s->dst_pin);
    rc = enqueue_frame(f, s, &frame, y0_luma, y1_luma, whole, s->antiring, true);
    if (rc != JINC_OK) {
        cudaStreamSynchronize(s->stream);
        return rc;
    }
    return finish_frame(f, s, y0_luma, y1_luma, whole);
}

int check_frame(const jinc_filter* f, const jinc_frame* frame)
{
    if (!f || !frame)
        return jinc_fail(JINC_E_INVALID, "jinc_filter: null argument");
    for (int i = 0; i < f->p.n_planes; ++i)
        if (!frame->src[i] || !frame->dst[i])
            return jinc_fail(JINC_E_INVALID, "jinc_filter: plane %d has a null pointer", i);
    return JINC_OK;
}

int submit_impl(jinc_filter* f, const jinc_frame* frame, int64_t* ticket, bool block)
{
    if (int rc = check_frame(f, frame))
        return rc;
    if (!ticket)
        return jinc_fail(JINC_E_INVALID, "jinc_filter_submit: null ticket");
    const float antiring = f->antiring.load();
    Slot* s = acquire_slot(f, block);
    if (!s)
        return jinc_fail(JINC_E_BUSY, "jinc_filter_try_submit: all %zu in-flight slots are taken", f->slots.size());
    const int64_t tk = s->ticket;
    const int rc = enqueue_frame(f, s, frame, 0, f->p.target_h, true, antiring);
    if (rc != JINC_OK) {
        cudaStreamSynchronize(s->stream);
        release_slot(f, s);
        return rc;
    }
    *ticket = tk;
    return JINC_OK;
}

} // namespace

extern "C" void jinc_filter_destroy(jinc_filter* f)
{
    if (!f)
        return;
    for (auto& s : f->slots) {
        cudaSetDevice(f->devs[s->dev_index].ctx->device);
        if (s->stream)
            cudaStreamSynchronize(s->stream);
        jinc_hostmem::release(&s->src_pin);
        jinc_hostmem::release(&s->dst_pin);
        cudaFree(s->d_src);
        cudaFree(s->d_dst);
        cudaFreeHost(s->h_src);
        cudaFreeHost(s->h_dst);
        cudaFree(s->d_probe);
        cudaFreeHost(s->h_probe);
        if (s->done)
            cudaEventDestroy(s->done);
        if (s->stream)
            cudaStreamDestroy(s->stream);
    }
    for (DeviceState& d : f->devs) {
        if (d.ctx) {
            cudaSetDevice(d.ctx->device);
            jinc_ring_free(d.ctx); // batched launches still reading the tables finish first
        }
        jinc_table_destroy(d.tables[0]);
        jinc_table_destroy(d.tables[1]);
        jinc_ctx_destroy(d.ctx);
    }
    if (f->registers)
        jinc_hostmem::client_remove();
    delete f;
    g_live_filters.fetch_sub(1);
}

extern "C" int jinc_filter_live_count(void) { return g_live_filters.load(); }

extern "C" int jinc_filter_create(const jinc_filter_params* p, jinc_filter** out)
{
    if (!p || !out)
        return jinc_fail(JINC_E_INVALID, "jinc_filter_create: null argument");
    *out = nullptr;
    if (p->n_planes < 1 || p->n_planes > JINC_MAX_PLANES)
        return jinc_fail(JINC_E_INVALID, "jinc_filter_create: n_planes must be 1..4");
    if (!jinc_sample_valid(p->sample_bytes))
        return jinc_fail(JINC_E_INVALID, "jinc_filter_create: sample_bytes must be 1, 2, 4 or JINC_SAMPLE_F16");
    // bits feed peak = (1 << bits) - 1 (:793): 8 for one-byte samples, 10..16 for two-byte samples; float ignores it
    if ((p->sample_bytes == 1 && p->bits != 8) || (p->sample_bytes == 2 && (p->bits < 9 || p->bits > 16)))
        return jinc_fail(JINC_E_INVALID, "jinc_filter_create: %d bits per component do not fit %d-byte samples", p->bits, p->sample_bytes);
    if (p->sample_bytes == JINC_SAMPLE_F16 && p->bits != 16)
        return jinc_fail(JINC_E_INVALID, "jinc_filter_create: %d bits per component do not fit half (16-bit float) samples", p->bits);
    if (p->tap < 1 || p->tap > 16)
        return jinc_fail(JINC_E_INVALID, "JincResize: tap must be between 1..16.");
    if (p->src_w < 1 || p->src_h < 1 || p->target_w < 1 || p->target_h < 1)
        return jinc_fail(JINC_E_INVALID, "jinc_filter_create: clip dimensions must be positive");
    if (p->sub_w < 0 || p->sub_w > 2 || p->sub_h < 0 || p->sub_h > 2)
        return jinc_fail(JINC_E_INVALID, "jinc_filter_create: bad chroma subsampling");
    if (p->n_devices > JINC_MAX_DEVICES)
        return jinc_fail(JINC_E_INVALID, "jinc_filter_create: at most %d devices", JINC_MAX_DEVICES);
    if (p->slots_per_device < 0 || p->slots_per_device > 64)
        return jinc_fail(JINC_E_INVALID, "jinc_filter_create: slots_per_device must be 0..64");

    int visible = jinc_device_count();
    if (visible == 0)
        return jinc_fail(JINC_E_CUDA, "JincResize: no CUDA device available (this build has no CPU fallback)");
    std::vector<int> dev_ids;
    if (p->n_devices <= 0) {
        for (int i = 0; i < visible && i < JINC_MAX_DEVICES; ++i)
            dev_ids.push_back(i);
    } else {
        for (int i = 0; i < p->n_devices; ++i)
            dev_ids.push_back(p->devices[i]);
    }

    std::unique_ptr<jinc_filter, void (*)(jinc_filter*)> f(new jinc_filter(), jinc_filter_destroy);
    g_live_filters.fetch_add(1);
    f->p = *p;
    if (p->flags & JINC_FILTER_HOST_REGISTER) {
        jinc_hostmem::client_add();
        f->registers = true;
    }
    f->peak = jinc_sample_is_float(p->sample_bytes) ? 0.f : static_cast<float>((1 << p->bits) - 1); // :793
    derive_table_params(*p, f->tparams, &f->n_tables);

    // Plane layout shared by device and pinned buffers: 64-byte pitches and 64-byte plane offsets.  Vector loads/stores
    // stay aligned, a plane whose host rows have the same pitch moves as ONE linear transfer instead of a row-by-row 2-D
    // copy, and a frame buffer packed by the same rule (AviSynth+ frame buffers are) moves as one transfer per frame.
    size_t so = 0, dof = 0;
    for (int i = 0; i < p->n_planes; ++i) {
        PlaneLayout& pl = f->planes[i];
        pl.table = (f->n_tables == 2 && (i == 1 || i == 2)) ? 1 : 0; // :552-558: alpha (3) uses the luma table
        const jinc_table_params& tp = f->tparams[pl.table];
        pl.src_w = tp.src_w;
        pl.src_h = tp.src_h;
        pl.dst_w = tp.dst_w;
        pl.dst_h = tp.dst_h;
        pl.src_pitch = align_up(static_cast<size_t>(pl.src_w) * jinc_sample_size(p->sample_bytes), 64);
        pl.dst_pitch = align_up(static_cast<size_t>(pl.dst_w) * jinc_sample_size(p->sample_bytes), 64);
        pl.src_off = so;
        pl.dst_off = dof;
        so += pl.src_pitch * pl.src_h;
        dof += pl.dst_pitch * pl.dst_h;
    }
    so = align_up(so, 256);
    dof = align_up(dof, 256);
    f->src_bytes = so;
    f->dst_bytes = dof;

    // frames in flight per GPU: a slot is held from the first copy of the source until the output has arrived, so small
    // frames get more slots (3..8, about 512 MB per GPU)
    int spd = p->slots_per_device;
    if (spd <= 0) {
        const size_t per_slot = std::max<size_t>(so + dof, 1);
        spd = static_cast<int>(std::min<size_t>(8, std::max<size_t>(3, (static_cast<size_t>(512) << 20) / per_slot)));
    }
    for (size_t di = 0; di < dev_ids.size(); ++di) {
        f->devs.emplace_back(); // owned by the filter from here on: an early return frees whatever has been created
        DeviceState& d = f->devs.back();
        int rc = jinc_ctx_create(dev_ids[di], &d.ctx);
        if (rc != JINC_OK)
            return rc;
        for (int k = 0; k < f->n_tables; ++k) {
            rc = jinc_table_create(d.ctx, &f->tparams[k], &d.tables[k]);
            if (rc != JINC_OK)
                return rc;
        }
        for (int sidx = 0; sidx < spd; ++sidx) {
            f->slots.push_back(std::make_unique<Slot>());
            Slot* s = f->slots.back().get();
            s->dev_index = static_cast<int>(di);
            JINC_CUDA(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
            JINC_CUDA(cudaEventCreateWithFlags(&s->done, cudaEventDisableTiming));
            if (cudaMalloc(reinterpret_cast<void**>(&s->d_src), so) != cudaSuccess ||
                cudaMalloc(reinterpret_cast<void**>(&s->d_dst), dof) != cudaSuccess ||
                cudaHostAlloc(reinterpret_cast<void**>(&s->h_src), so, cudaHostAllocPortable) != cudaSuccess ||
                cudaHostAlloc(reinterpret_cast<void**>(&s->h_dst), dof, cudaHostAllocPortable) != cudaSuccess ||
                cudaMalloc(reinterpret_cast<void**>(&s->d_probe), JINC_PROBE_WORDS * sizeof(uint32_t)) != cudaSuccess ||
                cudaHostAlloc(reinterpret_cast<void**>(&s->h_probe), JINC_PROBE_WORDS * sizeof(uint32_t), cudaHostAllocPortable) != cudaSuccess) {
                const char* msg = cudaGetErrorString(cudaGetLastError());
                return jinc_fail(JINC_E_NOMEM, "JincResize: failed to allocate frame buffers (%zu + %zu bytes): %s", so, dof, msg);
            }
        }
    }
    *out = f.release();
    return JINC_OK;
}

extern "C" const jinc_table* jinc_filter_table(const jinc_filter* f, int k)
{
    if (!f || k < 0 || k >= f->n_tables || f->devs.empty())
        return nullptr;
    return f->devs[0].tables[k];
}

extern "C" int jinc_filter_num_tables(const jinc_filter* f) { return f ? f->n_tables : 0; }
extern "C" int jinc_filter_num_devices(const jinc_filter* f) { return f ? static_cast<int>(f->devs.size()) : 0; }
extern "C" int jinc_filter_num_slots(const jinc_filter* f) { return f ? static_cast<int>(f->slots.size()) : 0; }
extern "C" int64_t jinc_filter_kernel_launches(const jinc_filter* f) { return f ? f->launches.load() : 0; }

extern "C" int jinc_filter_set_antiring(jinc_filter* f, float strength)
{
    if (!f)
        return jinc_fail(JINC_E_INVALID, "jinc_filter_set_antiring: null filter");
    if (!(strength >= 0.f && strength <= 1.f))
        return jinc_fail(JINC_E_INVALID, "jinc_filter_set_antiring: strength must be between 0.0 and 1.0");
    f->antiring.store(strength);
    return JINC_OK;
}

extern "C" void jinc_host_buffer_stats(int64_t* registered_bytes, int64_t* registrations, int64_t* direct_src_frames,
                                       int64_t* direct_dst_frames, int64_t* staged_frames)
{
    if (registered_bytes)
        *registered_bytes = static_cast<int64_t>(jinc_hostmem::registered_bytes());
    if (registrations)
        *registrations = jinc_hostmem::registrations();
    if (direct_src_frames)
        *direct_src_frames = g_direct_src.load();
    if (direct_dst_frames)
        *direct_dst_frames = g_direct_dst.load();
    if (staged_frames)
        *staged_frames = g_staged.load();
}

extern "C" int jinc_filter_process(jinc_filter* f, const jinc_frame* frame)
{
    if (int rc = check_frame(f, frame))
        return rc;
    const float antiring = f->antiring.load();
    Slot* s = acquire_slot(f, true);
    int rc = enqueue_frame(f, s, frame, 0, f->p.target_h, true, antiring);
    if (rc == JINC_OK)
        rc = complete_frame(f, s, 0, f->p.target_h, true);
    else
        cudaStreamSynchronize(s->stream);
    release_slot(f, s);
    return rc;
}

extern "C" int jinc_filter_process_device(jinc_filter* f, int device_index, const jinc_frame* frame, int table_mask, int parts,
                                          void* stream)
{
    if (int rc = check_frame(f, frame))
        return rc;
    if (device_index < 0 || device_index >= static_cast<int>(f->devs.size()))
        return jinc_fail(JINC_E_INVALID, "jinc_filter_process_device: bad device index %d", device_index);
    DeviceState& d = f->devs[device_index];
    JINC_CUDA(cudaSetDevice(d.ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : d.ctx->stream;
    const float antiring = f->antiring.load();
    for (int k = 0; k < f->n_tables; ++k) {
        if (!(table_mask & (1 << k)))
            continue;
        const void* src[JINC_MAX_PLANES];
        void* dst[JINC_MAX_PLANES];
        ptrdiff_t sp[JINC_MAX_PLANES], dp[JINC_MAX_PLANES];
        int n = 0;
        for (int i = 0; i < f->p.n_planes; ++i) {
            if (f->planes[i].table != k)
                continue;
            src[n] = frame->src[i];
            dst[n] = frame->dst[i];
            sp[n] = frame->src_pitch[i];
            dp[n] = frame->dst_pitch[i];
            ++n;
        }
        if (n == 0)
            continue;
        int launched = 0;
        int rc = jinc_launch_resize_planes(d.ctx, d.tables[k], f->p.sample_bytes, f->peak, n, src, sp, dst, dp, 0,
                                           d.tables[k]->sc.dst_h, st, &launched, parts);
        if (rc == JINC_OK && antiring > 0.f && parts == JINC_PART_ALL)
            rc = jinc_launch_antiring_planes(d.tables[k], f->p.sample_bytes, antiring, n, src, sp, dst, dp, 0, d.tables[k]->sc.dst_h, st,
                                             &launched);
        f->launches.fetch_add(launched);
        if (rc != JINC_OK)
            return rc;
    }
    return JINC_OK;
}

extern "C" int jinc_filter_process_device_batch(jinc_filter* f, int device_index, const jinc_frame* frames, int n_frames,
                                                int table_mask, int parts, void* stream)
{
    if (!f || !frames || n_frames < 1)
        return jinc_fail(JINC_E_INVALID, "jinc_filter_process_device_batch: bad argument");
    if (device_index < 0 || device_index >= static_cast<int>(f->devs.size()))
        return jinc_fail(JINC_E_INVALID, "jinc_filter_process_device_batch: bad device index %d", device_index);
    DeviceState& d = f->devs[device_index];
    JINC_CUDA(cudaSetDevice(d.ctx->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : d.ctx->stream;
    const float antiring = f->antiring.load();
    const size_t rec = jinc_plane_ptrs_size();
    for (int k = 0; k < f->n_tables; ++k) {
        if (!(table_mask & (1 << k)))
            continue;
        std::vector<unsigned char> host(rec * n_frames);
        int n = 0;
        for (int fi = 0; fi < n_frames; ++fi) {
            const void* src[JINC_MAX_PLANES];
            void* dst[JINC_MAX_PLANES];
            ptrdiff_t sp[JINC_MAX_PLANES], dp[JINC_MAX_PLANES];
            n = 0;
            for (int i = 0; i < f->p.n_planes; ++i) {
                if (f->planes[i].table != k)
                    continue;
                if (!frames[fi].src[i] || !frames[fi].dst[i])
                    return jinc_fail(JINC_E_INVALID, "jinc_filter_process_device_batch: frame %d plane %d has a null pointer", fi, i);
                src[n] = frames[fi].src[i];
                dst[n] = frames[fi].dst[i];
                sp[n] = frames[fi].src_pitch[i];
                dp[n] = frames[fi].dst_pitch[i];
                ++n;
            }
            if (n == 0)
                break;
            if (int rc = jinc_pack_plane_ptrs(host.data() + rec * fi, f->p.sample_bytes, n, src, sp, dst, dp))
                return rc;
        }
        if (n == 0)
            continue;
        int launched = 0;
        const int rc = jinc_ring_launch(d.ctx, host.data(), host.size(), st, [&](const void* dbuf) {
            int r = jinc_launch_resize_batch(d.ctx, d.tables[k], f->p.sample_bytes, f->peak, n, dbuf, n_frames, st, &launched, parts);
            if (r == JINC_OK && antiring > 0.f && parts == JINC_PART_ALL) // before the record: the pass reads the same plane-pointer records
                r = jinc_launch_antiring_batch(d.tables[k], f->p.sample_bytes, antiring, n, dbuf, n_frames, st, &launched);
            return r;
        });
        f->launches.fetch_add(launched);
        if (rc != JINC_OK)
            return rc;
    }
    return JINC_OK;
}

extern "C" int jinc_filter_submit(jinc_filter* f, const jinc_frame* frame, int64_t* ticket)
{
    return submit_impl(f, frame, ticket, true);
}

extern "C" int jinc_filter_try_submit(jinc_filter* f, const jinc_frame* frame, int64_t* ticket)
{
    return submit_impl(f, frame, ticket, false);
}

extern "C" int jinc_filter_wait(jinc_filter* f, int64_t ticket)
{
    if (!f)
        return jinc_fail(JINC_E_INVALID, "jinc_filter_wait: null filter");
    Slot* s = nullptr;
    {
        std::lock_guard<std::mutex> lk(f->mu);
        for (auto& c : f->slots)
            if (c->state == Slot::BUSY && c->ticket == ticket) {
                s = c.get();
                s->state = Slot::WAITING; // a second waiter on the same ticket finds nothing
            }
    }
    if (!s)
        return jinc_fail(JINC_E_INVALID, "jinc_filter_wait: unknown ticket %lld (never issued, or already waited on)",
                         static_cast<long long>(ticket));
    const int rc = complete_frame(f, s, 0, f->p.target_h, true);
    release_slot(f, s);
    return rc;
}

extern "C" int jinc_plan_frame_owner(int64_t frame, int n_parts)
{
    if (n_parts < 1 || frame < 0)
        return jinc_fail(JINC_E_INVALID, "jinc_plan_frame_owner: bad argument");
    return static_cast<int>(frame % n_parts);
}

extern "C" int jinc_plan_row_bands(int target_h, int n_parts, int32_t* y_begin, int32_t* y_end)
{
    if (target_h < 1 || n_parts < 1 || !y_begin || !y_end)
        return jinc_fail(JINC_E_INVALID, "jinc_plan_row_bands: bad argument");
    const int band = static_cast<int>(align_up(static_cast<size_t>((target_h + n_parts - 1) / n_parts), 16));
    for (int i = 0; i < n_parts; ++i) {
        y_begin[i] = std::min(target_h, i * band);
        y_end[i] = std::min(target_h, (i + 1) * band);
    }
    return JINC_OK;
}

extern "C" int jinc_filter_process_bands(jinc_filter* f, const jinc_frame* frame, int n_bands)
{
    if (int rc = check_frame(f, frame))
        return rc;
    if (n_bands < 1 || n_bands > 4096)
        return jinc_fail(JINC_E_INVALID, "jinc_filter_process_bands: n_bands must be 1..4096");
    const int nd = static_cast<int>(f->devs.size());
    std::vector<int32_t> yb(n_bands), ye(n_bands);
    if (int rc = jinc_plan_row_bands(f->p.target_h, n_bands, yb.data(), ye.data()))
        return rc;
    const float antiring = f->antiring.load(); // one strength for every band of the frame

    // Band i runs on GPU i % G through a slot of that GPU.  This caller never blocks on a slot while it holds one: when
    // its GPU has none free it first completes its own oldest band, so concurrent callers cannot deadlock each other.
    struct InFlight {
        Slot* s;
        int y0, y1;
    };
    std::vector<InFlight> fifo;
    size_t head = 0;
    int rc = JINC_OK;
    auto finish_oldest = [&]() {
        InFlight& b = fifo[head++];
        if (rc == JINC_OK)
            rc = complete_frame(f, b.s, b.y0, b.y1, false);
        else
            cudaStreamSynchronize(b.s->stream);
        release_slot(f, b.s);
    };
    for (int i = 0; i < n_bands && rc == JINC_OK; ++i) {
        if (ye[i] <= yb[i])
            continue;
        Slot* s = nullptr;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(f->mu);
                s = find_free_slot(f, i % nd, true);
                if (!s && head == fifo.size()) {
                    f->cv.wait(lk); // holding nothing: waiting is safe
                    continue;
                }
                if (s) {
                    s->state = Slot::BUSY;
                    s->ticket = f->next_ticket++;
                }
            }
            if (s)
                break;
            finish_oldest();
            if (rc != JINC_OK)
                break;
        }
        if (!s)
            break;
        rc = enqueue_frame(f, s, frame, yb[i], ye[i], false, antiring);
        if (rc != JINC_OK) {
            cudaStreamSynchronize(s->stream);
            release_slot(f, s);
            break;
        }
        fifo.push_back(InFlight{s, yb[i], ye[i]});
    }
    while (head < fifo.size())
        finish_oldest();
    return rc;
}

extern "C" int jinc_filter_process_split(jinc_filter* f, const jinc_frame* frame)
{
    if (int rc = check_frame(f, frame))
        return rc;
    const int nd = static_cast<int>(f->devs.size());
    if (nd == 1)
        return jinc_filter_process(f, frame);
    return jinc_filter_process_bands(f, frame, nd);
}
