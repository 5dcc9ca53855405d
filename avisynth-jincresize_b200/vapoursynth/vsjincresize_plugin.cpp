// vsjincresize_plugin.cpp -- VapourSynth (API 4) front-end over the same C ABI (include/jinc_b200.h) as the AviSynth+
// plugin: core.jinc.JincResize(clip, width, height[, tap, src_left, src_top, src_width, src_height, quant_x, quant_y,
// blur, cplace, antiring]).  The reference is itself a port of VapourSynth-JincResize (README.md:5); this is the way
// back, with the argument meanings, defaults, validation and error texts of src/JincResize.cpp:689-789 and every pixel
// computed on the GPU.  `antiring` (0.0..1.0, default 0 = off) has no reference counterpart: see
// jinc_filter_set_antiring.  No CUDA headers here and no CPU resampling path: without a usable GPU the filter
// constructor sets an error.
//
// Differences from the AviSynth+ front-end, all forced by the host: planes come in VapourSynth's order (R,G,B for RGB --
// immaterial, RGB planes share one coefficient table); the output _ChromaLocation of a subsampled clip is the cplace that
// was used (there is no reference behaviour to reproduce on this side); the host's frame buffers are page-locked only
// when JINCRESIZE_B200_HOSTREG=1 (see JINC_FILTER_HOST_REGISTER).
#include <algorithm>
#include <cctype>
#include <cstdlib>
#include <cstring>
#include <string>

#include "VapourSynth4.h"
#include "jinc_b200.h"

namespace {

struct Instance {
    VSNode* node = nullptr;
    VSVideoInfo vi{};
    jinc_filter* filter = nullptr;
    int n_planes = 0;
    bool writes_chromaloc = false;
    int chromaloc = 0;
};

const VSFrame* VS_CC get_frame(int n, int activationReason, void* instanceData, void**, VSFrameContext* frameCtx, VSCore* core,
                               const VSAPI* vsapi)
{
    auto* d = static_cast<Instance*>(instanceData);
    if (activationReason == arInitial) {
        vsapi->requestFrameFilter(n, d->node, frameCtx);
        return nullptr;
    }
    if (activationReason != arAllFramesReady)
        return nullptr;
    const VSFrame* src = vsapi->getFrameFilter(n, d->node, frameCtx);
    VSFrame* dst = vsapi->newVideoFrame(&d->vi.format, d->vi.width, d->vi.height, src, core); // properties copied from src
    jinc_frame fr;
    memset(&fr, 0, sizeof(fr));
    for (int i = 0; i < d->n_planes; ++i) {
        fr.src[i] = vsapi->getReadPtr(src, i);
        fr.src_pitch[i] = vsapi->getStride(src, i);
        fr.dst[i] = vsapi->getWritePtr(dst, i);
        fr.dst_pitch[i] = vsapi->getStride(dst, i);
    }
    if (jinc_filter_process(d->filter, &fr) != JINC_OK) {
        const std::string msg = std::string("JincResize: ") + jinc_last_error();
        vsapi->setFilterError(msg.c_str(), frameCtx);
        vsapi->freeFrame(src);
        vsapi->freeFrame(dst);
        return nullptr;
    }
    if (d->writes_chromaloc)
        vsapi->mapSetInt(vsapi->getFramePropertiesRW(dst), "_ChromaLocation", d->chromaloc, maReplace);
    vsapi->freeFrame(src);
    return dst;
}

void VS_CC free_filter(void* instanceData, VSCore*, const VSAPI* vsapi)
{
    auto* d = static_cast<Instance*>(instanceData);
    vsapi->freeNode(d->node);
    jinc_filter_destroy(d->filter);
    delete d;
}

void VS_CC create(const VSMap* in, VSMap* out, void*, VSCore* core, const VSAPI* vsapi)
{
    int err = 0;
    VSNode* node = vsapi->mapGetNode(in, "clip", 0, nullptr);
    const VSVideoInfo* vi = vsapi->getVideoInfo(node);
    auto fail = [&](const char* msg) {
        vsapi->mapSetError(out, msg);
        vsapi->freeNode(node);
    };
    auto opt_int = [&](const char* key, int64_t def) {
        const int64_t v = vsapi->mapGetInt(in, key, 0, &err);
        return err ? def : v;
    };
    auto opt_float = [&](const char* key, double def) {
        const double v = vsapi->mapGetFloat(in, key, 0, &err);
        return err ? def : static_cast<double>(static_cast<float>(v)); // script floats are 32-bit on the AviSynth side (:762-770)
    };

    if (vi->format.colorFamily == cfUndefined || vi->width <= 0 || vi->height <= 0)
        return fail("JincResize: only constant format input is supported.");
    const bool is_float = vi->format.sampleType == stFloat;
    const bool is_half = is_float && vi->format.bitsPerSample == 16; // GRAYH, YUV4xxPH, RGBH
    if ((is_float && vi->format.bitsPerSample != 32 && !is_half) || (!is_float && (vi->format.bitsPerSample < 8 || vi->format.bitsPerSample > 16)))
        return fail("JincResize: only 8..16 bit integer, 16 bit float and 32 bit float input is supported.");

    const int tap = static_cast<int>(opt_int("tap", 3));
    if (tap < 1 || tap > 16)
        return fail("JincResize: tap must be between 1..16.");
    const int quant_x = static_cast<int>(opt_int("quant_x", 256));
    if (quant_x < 1 || quant_x > 256)
        return fail("JincResize: quant_x must be between 1..256.");
    const int quant_y = static_cast<int>(opt_int("quant_y", 256));
    if (quant_y < 1 || quant_y > 256)
        return fail("JincResize: quant_y must be between 1..256.");
    const int target_w = static_cast<int>(vsapi->mapGetInt(in, "width", 0, nullptr));
    const int target_h = static_cast<int>(vsapi->mapGetInt(in, "height", 0, nullptr));
    if (target_w < 1 || target_h < 1)
        return fail("JincResize: width and height must be positive.");
    const double antiring = opt_float("antiring", 0.0);
    if (!(antiring >= 0.0 && antiring <= 1.0))
        return fail("JincResize: antiring must be between 0.0 and 1.0.");

    const bool subsampled = vi->format.colorFamily == cfYUV && (vi->format.subSamplingW || vi->format.subSamplingH);
    const char* cp = vsapi->mapGetData(in, "cplace", 0, &err);
    std::string cplace = err ? "" : cp;
    if (!cplace.empty()) {
        std::transform(cplace.begin(), cplace.end(), cplace.begin(), [](unsigned char c) { return (char)std::tolower(c); });
        if (cplace != "mpeg2" && cplace != "mpeg1" && cplace != "topleft")
            return fail("JincResize: cplace must be MPEG2, MPEG1 or topleft.");
    } else {
        // default from the first frame's _ChromaLocation, else MPEG2 (:725-742)
        cplace = "mpeg2";
        if (subsampled) {
            char buf[256];
            if (const VSFrame* f0 = vsapi->getFrame(0, node, buf, sizeof(buf))) {
                const int64_t loc = vsapi->mapGetInt(vsapi->getFramePropertiesRO(f0), "_ChromaLocation", 0, &err);
                vsapi->freeFrame(f0);
                if (!err) {
                    if (loc == 0)
                        cplace = "mpeg2";
                    else if (loc == 1)
                        cplace = "mpeg1";
                    else if (loc == 2)
                        cplace = "topleft";
                    else
                        return fail("JincResize: invalid _ChromaLocation");
                }
            }
        }
    }
    if (cplace == "topleft" && !(vi->format.colorFamily == cfYUV && vi->format.subSamplingW == 1 && vi->format.subSamplingH == 1))
        return fail("JincResize: topleft must be used only for 4:2:0 chroma subsampling.");

    jinc_filter_params p;
    memset(&p, 0, sizeof(p));
    p.src_w = vi->width;
    p.src_h = vi->height;
    p.target_w = target_w;
    p.target_h = target_h;
    p.src_left = opt_float("src_left", 0.0);
    p.src_top = opt_float("src_top", 0.0);
    p.src_width = opt_float("src_width", static_cast<double>(vi->width));
    p.src_height = opt_float("src_height", static_cast<double>(vi->height));
    p.quant_x = quant_x;
    p.quant_y = quant_y;
    p.tap = tap;
    p.blur = opt_float("blur", 0.0); // 0 => 1.0 inside the library (:772-774)
    p.cplace = cplace == "mpeg2" ? JINC_CPLACE_MPEG2 : (cplace == "mpeg1" ? JINC_CPLACE_MPEG1 : JINC_CPLACE_TOPLEFT);
    p.n_planes = vi->format.numPlanes;
    p.sample_bytes = is_half ? JINC_SAMPLE_F16 : vi->format.bytesPerSample; // the output format is the input format
    p.bits = vi->format.bitsPerSample;
    p.sub_w = subsampled ? vi->format.subSamplingW : 0;
    p.sub_h = subsampled ? vi->format.subSamplingH : 0;
    const char* devs = getenv("JINCRESIZE_B200_DEVICES");
    if (!devs || !*devs) {
        p.devices[p.n_devices++] = 0;
    } else if (strcmp(devs, "all") != 0) {
        const char* s = devs;
        while (*s && p.n_devices < JINC_MAX_DEVICES) {
            char* end = nullptr;
            const long v = strtol(s, &end, 10);
            if (end == s)
                break;
            p.devices[p.n_devices++] = static_cast<int>(v);
            s = (*end == ',') ? end + 1 : end;
        }
    }
    if (const char* slots = getenv("JINCRESIZE_B200_SLOTS"))
        p.slots_per_device = atoi(slots);
    p.flags = JINC_FILTER_DST_PADDING_WRITABLE; // VapourSynth frame planes own the padding inside their stride
    if (const char* hr = getenv("JINCRESIZE_B200_HOSTREG"))
        if (*hr == '1')
            p.flags |= JINC_FILTER_HOST_REGISTER;

    jinc_filter* filter = nullptr;
    if (jinc_filter_create(&p, &filter) != JINC_OK) {
        std::string msg = jinc_last_error();
        if (msg.rfind("JincResize:", 0) != 0)
            msg = "JincResize: " + msg;
        return fail(msg.c_str());
    }
    if (antiring > 0.0 && jinc_filter_set_antiring(filter, static_cast<float>(antiring)) != JINC_OK) {
        const std::string msg = std::string("JincResize: ") + jinc_last_error();
        jinc_filter_destroy(filter);
        return fail(msg.c_str());
    }

    auto* d = new Instance();
    d->node = node;
    d->vi = *vi;
    d->vi.width = target_w;
    d->vi.height = target_h;
    d->filter = filter;
    d->n_planes = p.n_planes;
    d->writes_chromaloc = subsampled;
    d->chromaloc = p.cplace;
    VSFilterDependency deps[] = {{node, rpStrictSpatial}};
    vsapi->createVideoFilter(out, "JincResize", &d->vi, get_frame, free_filter, fmParallel, deps, 1, d, core);
}

} // namespace

VS_EXTERNAL_API(void) VapourSynthPluginInit2(VSPlugin* plugin, const VSPLUGINAPI* vspapi)
{
    vspapi->configPlugin("com.b200.jincresize", "jinc", "EWA Jinc resampling on B200 GPUs", VS_MAKE_VERSION(2, 0), VAPOURSYNTH_API_VERSION, 0,
                         plugin);
    vspapi->registerFunction("JincResize",
                             "clip:vnode;width:int;height:int;tap:int:opt;src_left:float:opt;src_top:float:opt;src_width:float:opt;"
                             "src_height:float:opt;quant_x:int:opt;quant_y:int:opt;blur:float:opt;cplace:data:opt;antiring:float:opt;",
                             "clip:vnode;", create, nullptr, plugin);
}
