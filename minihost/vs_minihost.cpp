/*
 * vs_minihost.cpp -- in-process stand-in for a VapourSynth (API 4) core, just large enough to load a video filter
 * plugin (VapourSynthPluginInit2), call its functions with an argument map, and pull frames through the two-phase
 * getFrame protocol (arInitial -> requestFrameFilter, arAllFramesReady -> getFrameFilter).  Frames are planar, one
 * 64-byte aligned allocation per plane, recycled through a pool like the real core's memory pool.
 *
 * TEST/BENCH INFRASTRUCTURE for avisynth-jincresize_b200/vapoursynth/; compiled against the clean-room
 * minihost/include/VapourSynth4.h (see the caveat there).  Exports the vsmh_* driver surface used from Python (ctypes).
 */
#include <dlfcn.h>

#include <atomic>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "VapourSynth4.h"

#define VSMH_API extern "C" __attribute__((visibility("default")))

namespace {
std::atomic<long> g_live_frames{0}, g_live_nodes{0};

struct Value {
    int type = ptUnset;
    std::vector<int64_t> i;
    std::vector<double> f;
    std::vector<std::string> d;
    std::vector<VSNode*> n;
};
} // namespace

struct VSMap {
    std::vector<std::pair<std::string, Value>> kv;
    bool has_error = false;
    std::string error;
    Value* find(const char* key)
    {
        for (auto& e : kv)
            if (e.first == key)
                return &e.second;
        return nullptr;
    }
    const Value* find(const char* key) const { return const_cast<VSMap*>(this)->find(key); }
    Value& get(const char* key)
    {
        if (Value* v = find(key))
            return *v;
        kv.emplace_back(key, Value());
        return kv.back().second;
    }
};

namespace {
std::mutex g_pool_mu;
std::unordered_map<size_t, std::vector<void*>> g_pool;

void* pool_get(size_t bytes)
{
    {
        std::lock_guard<std::mutex> lk(g_pool_mu);
        auto it = g_pool.find(bytes);
        if (it != g_pool.end() && !it->second.empty()) {
            void* p = it->second.back();
            it->second.pop_back();
            return p;
        }
    }
    void* mem = nullptr;
    if (posix_memalign(&mem, 64, bytes) != 0)
        return nullptr;
    memset(mem, 0, bytes);
    return mem;
}

void pool_put(void* p, size_t bytes)
{
    {
        std::lock_guard<std::mutex> lk(g_pool_mu);
        auto& v = g_pool[bytes];
        if (v.size() < 64) {
            v.push_back(p);
            return;
        }
    }
    free(p);
}
} // namespace

struct VSFrame {
    std::atomic<int> refs{1};
    VSVideoFormat fmt{};
    int w = 0, h = 0;
    uint8_t* plane[3] = {nullptr, nullptr, nullptr};
    ptrdiff_t stride[3] = {0, 0, 0};
    size_t bytes[3] = {0, 0, 0};
    int pw[3] = {0, 0, 0}, ph[3] = {0, 0, 0};
    VSMap props;
};

struct VSNode {
    std::atomic<int> refs{1};
    VSVideoInfo vi{};
    std::vector<VSFrame*> stored; // source node: frame n is stored[n % size]
    VSFilterGetFrame get_frame = nullptr;
    VSFilterFree free_fn = nullptr;
    void* instance = nullptr;
    VSCore* core = nullptr;
};

struct VSFrameContext {
    std::vector<std::pair<VSNode*, int>> requests;
    std::vector<std::pair<std::pair<VSNode*, int>, const VSFrame*>> ready;
    std::string error;
};

struct VSCore {
    int dummy = 0;
};

struct VSPlugin {
    std::string id, ns, name;
    void* dl = nullptr;
    VSCore* core = nullptr;
    struct Fn {
        std::string args, ret;
        VSPublicFunction fn;
        void* data;
    };
    std::map<std::string, Fn> fns;
};

namespace {

extern const VSAPI g_api;

VSFrame* new_frame(const VSVideoFormat* f, int w, int h, const VSFrame* prop_src)
{
    auto* fr = new VSFrame();
    fr->fmt = *f;
    fr->w = w;
    fr->h = h;
    for (int p = 0; p < f->numPlanes; ++p) {
        fr->pw[p] = p ? w >> f->subSamplingW : w;
        fr->ph[p] = p ? h >> f->subSamplingH : h;
        fr->stride[p] = (static_cast<ptrdiff_t>(fr->pw[p]) * f->bytesPerSample + 63) / 64 * 64;
        fr->bytes[p] = static_cast<size_t>(fr->stride[p]) * fr->ph[p] + 64;
        fr->plane[p] = static_cast<uint8_t*>(pool_get(fr->bytes[p]));
    }
    if (prop_src)
        fr->props.kv = prop_src->props.kv;
    g_live_frames.fetch_add(1);
    return fr;
}

void VS_CC api_free_frame(const VSFrame* cf) noexcept
{
    auto* f = const_cast<VSFrame*>(cf);
    if (!f)
        return;
    if (f->refs.fetch_sub(1) == 1) {
        for (int p = 0; p < 3; ++p)
            if (f->plane[p])
                pool_put(f->plane[p], f->bytes[p]);
        delete f;
        g_live_frames.fetch_sub(1);
    }
}

const VSFrame* VS_CC api_add_frame_ref(const VSFrame* f) noexcept
{
    const_cast<VSFrame*>(f)->refs.fetch_add(1);
    return f;
}

void VS_CC api_free_node(VSNode* n) noexcept
{
    if (!n)
        return;
    if (n->refs.fetch_sub(1) == 1) {
        if (n->free_fn)
            n->free_fn(n->instance, n->core, &g_api);
        for (VSFrame* f : n->stored)
            api_free_frame(f);
        delete n;
        g_live_nodes.fetch_sub(1);
    }
}

VSNode* VS_CC api_add_node_ref(VSNode* n) noexcept
{
    n->refs.fetch_add(1);
    return n;
}

// pull frame n of a node: stored frame, or the filter's two-phase protocol
const VSFrame* node_get_frame(VSNode* node, int n, std::string& err)
{
    if (n < 0 || n >= node->vi.numFrames) {
        err = "frame index out of range";
        return nullptr;
    }
    if (!node->get_frame)
        return api_add_frame_ref(node->stored[static_cast<size_t>(n) % node->stored.size()]);
    VSFrameContext ctx;
    void* frame_data = nullptr;
    const VSFrame* out = node->get_frame(n, arInitial, node->instance, &frame_data, &ctx, node->core, &g_api);
    if (!out && ctx.error.empty()) {
        for (auto& rq : ctx.requests) {
            const VSFrame* f = node_get_frame(rq.first, rq.second, err);
            if (!f)
                break;
            ctx.ready.push_back({rq, f});
        }
        if (err.empty())
            out = node->get_frame(n, arAllFramesReady, node->instance, &frame_data, &ctx, node->core, &g_api);
    }
    for (auto& r : ctx.ready)
        api_free_frame(r.second);
    if (!out && err.empty())
        err = ctx.error.empty() ? "filter returned no frame" : ctx.error;
    return out;
}

// ---- VSAPI entries the filter plugin uses (the rest stay null)
void VS_CC api_create_video_filter(VSMap* out, const char*, const VSVideoInfo* vi, VSFilterGetFrame gf, VSFilterFree fr, int,
                                   const VSFilterDependency*, int, void* instance, VSCore* core) noexcept
{
    auto* n = new VSNode();
    n->vi = *vi;
    n->get_frame = gf;
    n->free_fn = fr;
    n->instance = instance;
    n->core = core;
    g_live_nodes.fetch_add(1);
    Value& v = out->get("clip");
    v.type = ptVideoNode;
    v.n.push_back(n); // the map owns this reference
}
const VSVideoInfo* VS_CC api_get_video_info(VSNode* n) noexcept { return &n->vi; }
VSFrame* VS_CC api_new_video_frame(const VSVideoFormat* f, int w, int h, const VSFrame* ps, VSCore*) noexcept { return new_frame(f, w, h, ps); }
const VSMap* VS_CC api_props_ro(const VSFrame* f) noexcept { return &f->props; }
VSMap* VS_CC api_props_rw(VSFrame* f) noexcept { return &f->props; }
ptrdiff_t VS_CC api_stride(const VSFrame* f, int p) noexcept { return f->stride[p]; }
const uint8_t* VS_CC api_read_ptr(const VSFrame* f, int p) noexcept { return f->plane[p]; }
uint8_t* VS_CC api_write_ptr(VSFrame* f, int p) noexcept { return f->plane[p]; }
const VSVideoFormat* VS_CC api_frame_format(const VSFrame* f) noexcept { return &f->fmt; }
int VS_CC api_frame_w(const VSFrame* f, int p) noexcept { return f->pw[p]; }
int VS_CC api_frame_h(const VSFrame* f, int p) noexcept { return f->ph[p]; }
const VSFrame* VS_CC api_get_frame(int n, VSNode* node, char* msg, int size) noexcept
{
    std::string err;
    const VSFrame* f = node_get_frame(node, n, err);
    if (!f && msg && size > 0) {
        strncpy(msg, err.c_str(), static_cast<size_t>(size) - 1);
        msg[size - 1] = 0;
    }
    return f;
}
const VSFrame* VS_CC api_get_frame_filter(int n, VSNode* node, VSFrameContext* ctx) noexcept
{
    for (auto& r : ctx->ready)
        if (r.first.first == node && r.first.second == n)
            return api_add_frame_ref(r.second);
    return nullptr;
}
void VS_CC api_request_frame_filter(int n, VSNode* node, VSFrameContext* ctx) noexcept { ctx->requests.push_back({node, n}); }
void VS_CC api_set_filter_error(const char* msg, VSFrameContext* ctx) noexcept { ctx->error = msg ? msg : "error"; }
VSMap* VS_CC api_create_map() noexcept { return new VSMap(); }
void VS_CC api_free_map(VSMap* m) noexcept
{
    if (!m)
        return;
    for (auto& e : m->kv)
        for (VSNode* n : e.second.n)
            api_free_node(n);
    delete m;
}
void VS_CC api_map_set_error(VSMap* m, const char* msg) noexcept
{
    m->has_error = true;
    m->error = msg ? msg : "";
}
const char* VS_CC api_map_get_error(const VSMap* m) noexcept { return m->has_error ? m->error.c_str() : nullptr; }
int VS_CC api_map_num_elements(const VSMap* m, const char* key) noexcept
{
    const Value* v = m->find(key);
    if (!v)
        return -1;
    return static_cast<int>(v->i.size() + v->f.size() + v->d.size() + v->n.size());
}
template <typename T>
T get_elem(const VSMap* m, const char* key, int index, int* error, int type, const std::vector<T> Value::*member, T def)
{
    const Value* v = m->find(key);
    int e = peSuccess;
    T out = def;
    if (!v)
        e = peUnset;
    else if (v->type != type)
        e = peType;
    else if (index < 0 || index >= static_cast<int>((v->*member).size()))
        e = peIndex;
    else
        out = (v->*member)[index];
    if (error)
        *error = e;
    return out;
}
int64_t VS_CC api_map_get_int(const VSMap* m, const char* key, int index, int* error) noexcept
{
    return get_elem<int64_t>(m, key, index, error, ptInt, &Value::i, 0);
}
double VS_CC api_map_get_float(const VSMap* m, const char* key, int index, int* error) noexcept
{
    return get_elem<double>(m, key, index, error, ptFloat, &Value::f, 0.0);
}
const char* VS_CC api_map_get_data(const VSMap* m, const char* key, int index, int* error) noexcept
{
    const Value* v = m->find(key);
    int e = peSuccess;
    const char* out = nullptr;
    if (!v)
        e = peUnset;
    else if (v->type != ptData)
        e = peType;
    else if (index < 0 || index >= static_cast<int>(v->d.size()))
        e = peIndex;
    else
        out = v->d[index].c_str();
    if (error)
        *error = e;
    return out;
}
VSNode* VS_CC api_map_get_node(const VSMap* m, const char* key, int index, int* error) noexcept
{
    VSNode* n = get_elem<VSNode*>(m, key, index, error, ptVideoNode, &Value::n, nullptr);
    return n ? api_add_node_ref(n) : nullptr;
}
int VS_CC api_map_set_int(VSMap* m, const char* key, int64_t i, int append) noexcept
{
    Value& v = m->get(key);
    if (append == maReplace || v.type != ptInt) {
        v = Value();
        v.type = ptInt;
    }
    v.i.push_back(i);
    return 0;
}
int VS_CC api_map_set_float(VSMap* m, const char* key, double d, int append) noexcept
{
    Value& v = m->get(key);
    if (append == maReplace || v.type != ptFloat) {
        v = Value();
        v.type = ptFloat;
    }
    v.f.push_back(d);
    return 0;
}
int VS_CC api_map_set_data(VSMap* m, const char* key, const char* data, int size, int, int append) noexcept
{
    Value& v = m->get(key);
    if (append == maReplace || v.type != ptData) {
        v = Value();
        v.type = ptData;
    }
    v.d.emplace_back(data, size < 0 ? strlen(data) : static_cast<size_t>(size));
    return 0;
}
int VS_CC api_map_set_node(VSMap* m, const char* key, VSNode* n, int append) noexcept
{
    Value& v = m->get(key);
    if (append == maReplace || v.type != ptVideoNode) {
        for (VSNode* o : v.n)
            api_free_node(o);
        v = Value();
        v.type = ptVideoNode;
    }
    v.n.push_back(api_add_node_ref(n));
    return 0;
}

VSAPI make_api()
{
    VSAPI a;
    memset(&a, 0, sizeof(a));
    a.createVideoFilter = api_create_video_filter;
    a.freeNode = api_free_node;
    a.addNodeRef = api_add_node_ref;
    a.getVideoInfo = api_get_video_info;
    a.newVideoFrame = api_new_video_frame;
    a.freeFrame = api_free_frame;
    a.addFrameRef = api_add_frame_ref;
    a.getFramePropertiesRO = api_props_ro;
    a.getFramePropertiesRW = api_props_rw;
    a.getStride = api_stride;
    a.getReadPtr = api_read_ptr;
    a.getWritePtr = api_write_ptr;
    a.getVideoFrameFormat = api_frame_format;
    a.getFrameWidth = api_frame_w;
    a.getFrameHeight = api_frame_h;
    a.getFrame = api_get_frame;
    a.getFrameFilter = api_get_frame_filter;
    a.requestFrameFilter = api_request_frame_filter;
    a.setFilterError = api_set_filter_error;
    a.createMap = api_create_map;
    a.freeMap = api_free_map;
    a.mapSetError = api_map_set_error;
    a.mapGetError = api_map_get_error;
    a.mapNumElements = api_map_num_elements;
    a.mapGetInt = api_map_get_int;
    a.mapGetFloat = api_map_get_float;
    a.mapGetData = api_map_get_data;
    a.mapGetNode = api_map_get_node;
    a.mapSetInt = api_map_set_int;
    a.mapSetFloat = api_map_set_float;
    a.mapSetData = api_map_set_data;
    a.mapSetNode = api_map_set_node;
    return a;
}
const VSAPI g_api = make_api();

int VS_CC papi_version() noexcept { return VAPOURSYNTH_API_VERSION; }
int VS_CC papi_config(const char* id, const char* ns, const char* name, int, int api_version, int, VSPlugin* p) noexcept
{
    if ((api_version >> 16) != VAPOURSYNTH_API_MAJOR)
        return 0;
    p->id = id;
    p->ns = ns;
    p->name = name;
    return 1;
}
int VS_CC papi_register(const char* name, const char* args, const char* ret, VSPublicFunction fn, void* data, VSPlugin* p) noexcept
{
    p->fns[name] = VSPlugin::Fn{args, ret, fn, data};
    return 1;
}
const VSPLUGINAPI g_papi = {papi_version, papi_config, papi_register};

} // namespace

// ------------------------------------------------------------------------------------------ driver surface
VSMH_API VSCore* vsmh_core_create(void) { return new VSCore(); }
VSMH_API void vsmh_core_destroy(VSCore* c) { delete c; }

VSMH_API VSPlugin* vsmh_load_plugin(VSCore* core, const char* path, char* err, int err_size)
{
    void* dl = dlopen(path, RTLD_NOW | RTLD_LOCAL);
    auto fail = [&](const char* msg) -> VSPlugin* {
        if (err && err_size > 0) {
            strncpy(err, msg, static_cast<size_t>(err_size) - 1);
            err[err_size - 1] = 0;
        }
        return nullptr;
    };
    if (!dl)
        return fail(dlerror());
    auto init = reinterpret_cast<VSInitPlugin>(dlsym(dl, "VapourSynthPluginInit2"));
    if (!init)
        return fail("VapourSynthPluginInit2 not exported");
    auto* p = new VSPlugin();
    p->dl = dl;
    p->core = core;
    init(p, &g_papi);
    return p;
}
VSMH_API const char* vsmh_plugin_namespace(VSPlugin* p) { return p->ns.c_str(); }
VSMH_API const char* vsmh_plugin_id(VSPlugin* p) { return p->id.c_str(); }
VSMH_API const char* vsmh_function_args(VSPlugin* p, const char* name)
{
    auto it = p->fns.find(name);
    return it == p->fns.end() ? nullptr : it->second.args.c_str();
}

VSMH_API VSNode* vsmh_source_create(VSCore* core, int color_family, int sample_type, int bits, int ssw, int ssh, int width, int height,
                                    int num_frames, int distinct)
{
    auto* n = new VSNode();
    n->core = core;
    VSVideoFormat& f = n->vi.format;
    f.colorFamily = color_family;
    f.sampleType = sample_type;
    f.bitsPerSample = bits;
    f.bytesPerSample = bits <= 8 ? 1 : (bits <= 16 ? 2 : 4);
    f.subSamplingW = ssw;
    f.subSamplingH = ssh;
    f.numPlanes = color_family == cfGray ? 1 : 3;
    n->vi.fpsNum = 24;
    n->vi.fpsDen = 1;
    n->vi.width = width;
    n->vi.height = height;
    n->vi.numFrames = num_frames;
    for (int k = 0; k < distinct; ++k)
        n->stored.push_back(new_frame(&f, width, height, nullptr));
    g_live_nodes.fetch_add(1);
    return n;
}
VSMH_API int vsmh_source_fill_plane(VSNode* n, int k, int plane, const void* src, ptrdiff_t pitch)
{
    if (k < 0 || k >= static_cast<int>(n->stored.size()) || plane < 0 || plane >= n->vi.format.numPlanes)
        return -1;
    VSFrame* f = n->stored[k];
    const size_t row = static_cast<size_t>(f->pw[plane]) * f->fmt.bytesPerSample;
    for (int y = 0; y < f->ph[plane]; ++y)
        memcpy(f->plane[plane] + y * f->stride[plane], static_cast<const uint8_t*>(src) + y * pitch, row);
    return 0;
}
VSMH_API void vsmh_source_set_prop_int(VSNode* n, const char* key, int64_t v)
{
    for (VSFrame* f : n->stored)
        api_map_set_int(&f->props, key, v, maReplace);
}

VSMH_API VSMap* vsmh_map_create(void) { return new VSMap(); }
VSMH_API void vsmh_map_free(VSMap* m) { api_free_map(m); }
VSMH_API void vsmh_map_set_node(VSMap* m, const char* k, VSNode* n) { api_map_set_node(m, k, n, maReplace); }
VSMH_API void vsmh_map_set_int(VSMap* m, const char* k, int64_t v) { api_map_set_int(m, k, v, maReplace); }
VSMH_API void vsmh_map_set_float(VSMap* m, const char* k, double v) { api_map_set_float(m, k, v, maReplace); }
VSMH_API void vsmh_map_set_data(VSMap* m, const char* k, const char* v) { api_map_set_data(m, k, v, -1, dtUtf8, maReplace); }

// calls plugin function `name`; returns the "clip" of the result (caller frees with vsmh_free_node) or NULL with the error text
VSMH_API VSNode* vsmh_invoke(VSPlugin* p, const char* name, VSMap* args, char* err, int err_size)
{
    auto put = [&](const std::string& s) {
        if (err && err_size > 0) {
            strncpy(err, s.c_str(), static_cast<size_t>(err_size) - 1);
            err[err_size - 1] = 0;
        }
    };
    auto it = p->fns.find(name);
    if (it == p->fns.end()) {
        put(std::string("no function named ") + name);
        return nullptr;
    }
    // the argument string is "name:type[:opt];...": unknown names and missing mandatory arguments are the host's errors
    std::vector<std::string> known;
    const std::string& spec = it->second.args;
    for (size_t pos = 0; pos < spec.size();) {
        const size_t end = spec.find(';', pos);
        const std::string item = spec.substr(pos, end - pos);
        const size_t c1 = item.find(':');
        const std::string an = item.substr(0, c1);
        known.push_back(an);
        if (item.find(":opt") == std::string::npos && !args->find(an.c_str())) {
            put(std::string(name) + ": argument " + an + " is required");
            return nullptr;
        }
        pos = end == std::string::npos ? spec.size() : end + 1;
    }
    for (auto& e : args->kv) {
        bool ok = false;
        for (auto& k : known)
            ok = ok || k == e.first;
        if (!ok) {
            put(std::string(name) + ": Function does not take argument(s) named " + e.first);
            return nullptr;
        }
    }
    VSMap out;
    it->second.fn(args, &out, it->second.data, p->core, &g_api);
    VSNode* node = nullptr;
    if (out.has_error) {
        put(out.error);
    } else if (Value* v = out.find("clip")) {
        if (!v->n.empty())
            node = api_add_node_ref(v->n[0]);
    }
    for (auto& e : out.kv)
        for (VSNode* n : e.second.n)
            api_free_node(n);
    return node;
}

VSMH_API void vsmh_node_info(VSNode* n, int* width, int* height, int* num_frames, int* num_planes, int* bytes_per_sample)
{
    *width = n->vi.width;
    *height = n->vi.height;
    *num_frames = n->vi.numFrames;
    *num_planes = n->vi.format.numPlanes;
    *bytes_per_sample = n->vi.format.bytesPerSample;
}
VSMH_API void vsmh_node_format(VSNode* n, int* sample_type, int* bits_per_sample)
{
    *sample_type = n->vi.format.sampleType;
    *bits_per_sample = n->vi.format.bitsPerSample;
}
VSMH_API const VSFrame* vsmh_get_frame(VSNode* n, int k, char* err, int err_size) { return api_get_frame(k, n, err, err_size); }
VSMH_API void vsmh_frame_plane(const VSFrame* f, int plane, const uint8_t** ptr, ptrdiff_t* stride, int* w, int* h)
{
    *ptr = f->plane[plane];
    *stride = f->stride[plane];
    *w = f->pw[plane];
    *h = f->ph[plane];
}
VSMH_API int vsmh_frame_prop_int(const VSFrame* f, const char* key, int64_t* out)
{
    int err = 0;
    const int64_t v = api_map_get_int(&f->props, key, 0, &err);
    if (err)
        return 0;
    *out = v;
    return 1;
}
VSMH_API void vsmh_free_frame(const VSFrame* f) { api_free_frame(f); }
VSMH_API void vsmh_free_node(VSNode* n) { api_free_node(n); }
VSMH_API long vsmh_live_frames(void) { return g_live_frames.load(); }
VSMH_API long vsmh_live_nodes(void) { return g_live_nodes.load(); }

// frame-parallel pull with `threads` host threads (fmParallel filters are called concurrently); seconds, or < 0 on error
VSMH_API double vsmh_pull_frames(VSNode* n, int first, int count, int threads)
{
    std::atomic<int> next{0}, failed{0};
    auto worker = [&]() {
        for (;;) {
            const int i = next.fetch_add(1);
            if (i >= count)
                return;
            std::string err;
            const VSFrame* f = node_get_frame(n, first + i, err);
            if (!f)
                failed.fetch_add(1);
            else
                api_free_frame(f);
        }
    };
    const auto t0 = std::chrono::steady_clock::now();
    if (threads <= 1) {
        worker();
    } else {
        std::vector<std::thread> pool;
        for (int t = 0; t < threads; ++t)
            pool.emplace_back(worker);
        for (auto& t : pool)
            t.join();
    }
    const auto t1 = std::chrono::steady_clock::now();
    return failed.load() ? -1.0 : std::chrono::duration<double>(t1 - t0).count();
}
