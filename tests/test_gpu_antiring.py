"""Anti-ringing: the antiring_pass kernels, jinc_filter_set_antiring / jinc_antiring_plane_device and the VapourSynth
`antiring` argument.

The pass is defined on the stored resized sample y (DESIGN.md §4.7): with ax0 = clamp(floor(pos_x), 0, W-1),
ax1 = clamp(floor(pos_x) + 1, 0, W-1) (ay0 / ay1 likewise) and lo / hi = fmin / fmax over src[ay0|ay1][ax0|ax1],
c = fmin(fmax(y, lo), hi) and out = c at s = 1, else fma(s, c, (1 - s) * y); NaN y stays NaN; integer planes round half
to even, half planes to the nearest half.  `antiring_ref` below restates it in NumPy, with the anchors taken from a
float32 re-accumulation of the oracle's positions.  The CPU tests at the end need no GPU."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from common import FULL_CASES, SMALL_CASES, assert_plane_close, oracle_frame, oracle_tables
from minihost import avs_host as ah

VS_BAD_ANTIRING = "JincResize: antiring must be between 0.0 and 1.0."


@pytest.fixture(scope="module")
def capi(native_built):
    from jinc_b200 import capi as c

    return c


@pytest.fixture(scope="module")
def gpu(capi):
    assert capi.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    return capi


# ------------------------------------------------------------------------------------------ the NumPy definition

def ref_positions(tp):
    """Output positions of one axis pair as the reference accumulates them (float32, one step at a time) from the
    oracle's table parameters: (pos_x[dst_w], pos_y[dst_h])."""
    def acc(first, step, n):
        a = np.full(n, np.float32(step), np.float32)
        a[0] = np.float32(first)
        return np.add.accumulate(a, dtype=np.float32)

    px = acc(tp.crop_left + (tp.crop_w / tp.dst_w - 1.0) / 2.0, tp.crop_w / tp.dst_w, tp.dst_w)
    py = acc(tp.crop_top + (tp.crop_h - tp.dst_h) / (tp.dst_h * 2.0), tp.crop_h / tp.dst_h, tp.dst_h)
    return px, py


def anchors(pos, n):
    f = np.floor(pos.astype(np.float64)).astype(np.int64)
    return np.clip(f, 0, n - 1), np.clip(f + 1, 0, n - 1)


def bounds(src, pos_x, pos_y):
    """lo, hi of every output sample's 2x2 source neighbourhood (NaN samples ignored), as float32."""
    S = src.astype(np.float32)
    ax0, ax1 = anchors(pos_x, S.shape[1])
    ay0, ay1 = anchors(pos_y, S.shape[0])
    r0, r1 = S[ay0], S[ay1]
    a, b, c, d = r0[:, ax0], r0[:, ax1], r1[:, ax0], r1[:, ax1]
    with np.errstate(invalid="ignore"):
        return np.fmin(np.fmin(a, b), np.fmin(c, d)), np.fmax(np.fmax(a, b), np.fmax(c, d))


def antiring_ref(y, src, pos_x, pos_y, s):
    """The pass on the stored plane y of src's resize (s > 0); the result has y's dtype."""
    lo, hi = bounds(src, pos_x, pos_y)
    yy = y.astype(np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        c = np.fmin(np.fmax(yy, lo), hi)
        if s == 1:
            out = c
        else:
            p = np.float32(np.float32(1) - np.float32(s)) * yy  # float32 product
            out = (np.float64(np.float32(s)) * c.astype(np.float64) + p.astype(np.float64)).astype(np.float32)
        out = np.where(np.isnan(yy), yy, out)
        if y.dtype in (np.float32, np.float16):
            return out.astype(y.dtype)
        return np.rint(out).astype(y.dtype)


def ordered(x):
    """Bit patterns of a float array in value order (+0 and -0 coincide), for ulp distances."""
    ib = {np.float16: np.int16, np.float32: np.int32}[x.dtype.type]
    bits = x.view(ib).astype(np.int64)
    mask = (1 << (8 * x.dtype.itemsize - 1)) - 1
    return np.where(bits < 0, -(bits & mask), bits)


def assert_pass_equal(got, want, exact, what):
    """exact: same values (NaN where NaN, +0 == -0); else within 1 LSB (integer) or 1 ulp (float)."""
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, want.shape, got.dtype)
    if got.dtype.kind == "f":
        nan = np.isnan(got)
        assert np.array_equal(nan, np.isnan(want)), f"{what}: NaN positions differ"
        d = np.abs(ordered(got[~nan]) - ordered(want[~nan]))
    else:
        d = np.abs(got.astype(np.int64) - want.astype(np.int64))
    if d.size == 0:
        return
    assert d.max() <= (0 if exact else 1), f"{what}: {int((d != 0).sum())} samples differ, by up to {int(d.max())}"


# ------------------------------------------------------------------------------------------ sample types

# (kind, numpy dtype, sample code, bits)
SAMPLES = [("u8", np.uint8, 1, 8), ("u10", np.uint16, 2, 10), ("u16", np.uint16, 2, 16), ("f16", np.float16, 0x102, 16),
           ("f32", np.float32, 4, 32)]


def noise(rng, shape, dtype, bits):
    if dtype in (np.float16, np.float32):
        return (rng.random(shape, dtype=np.float32)).astype(dtype)
    return rng.integers(0, (1 << bits), shape).astype(dtype)


def peak_of(dtype, bits):
    return 0.0 if dtype in (np.float16, np.float32) else float((1 << bits) - 1)


class DevPlane:
    """A plane in device memory with a 256-byte pitch (torch byte tensor), any sample type.  Every write synchronises the
    device: the library's calls run on streams that do not wait for torch's."""

    def __init__(self, a):
        import torch

        h, w = a.shape
        self.dtype, self.w, self.sb = a.dtype, w, a.dtype.itemsize
        self.pitch = (w * self.sb + 255) // 256 * 256
        self.t = torch.zeros((h, self.pitch), dtype=torch.uint8, device="cuda")
        self.set(a)

    def set(self, a):
        import torch

        h = a.shape[0]
        self.t[:, : self.w * self.sb].copy_(torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(h, self.w * self.sb)))
        torch.cuda.synchronize()

    @staticmethod
    def empty(h, w, dtype):
        return DevPlane(np.zeros((h, w), dtype))

    @property
    def ptr(self):
        return self.t.data_ptr()

    def get(self):
        import torch

        torch.cuda.synchronize()
        return np.ascontiguousarray(self.t[:, : self.w * self.sb].cpu().numpy()).view(self.dtype)


def device_table(capi, ctx, tp, tap, blur):
    return capi.Table(ctx, quant_x=tp.quant_x, quant_y=tp.quant_y, src_w=tp.src_w, src_h=tp.src_h, dst_w=tp.dst_w,
                      dst_h=tp.dst_h, radius=capi.radius_for_tap(tap), blur=float(np.float32(blur)),
                      crop_left=tp.crop_left, crop_top=tp.crop_top, crop_w=tp.crop_w, crop_h=tp.crop_h)


# ------------------------------------------------------------------------------------------ exactness, per plane

SMALL = {c[0]: c for c in SMALL_CASES}
PASS_CASES = [SMALL[n] for n in (
    "c1_yv12_2x_tap3",             # exact 2x, MPEG2 chroma
    "up2x_tap6_420p8",             # exact 2x, MPEG1 chroma
    "yuva420_14bit_2x",            # exact 2x, top-left chroma, alpha
    "c3_444p16_2x_tap4_crop",      # exact 2x with a crop
    "half_tap3_yv12",              # integer 1/2
    "third_tap3_y8",               # integer 1/3
    "quarter_tap3_y8",             # integer 1/4
    "down2to3_tap3_420p8",         # periodic 2:3, tap 3 (cells kernel)
    "down2to3_tap4_y16",           # periodic 2:3, tap 4
    "up1p5_tap3_420p8",            # cells 3:2
    "up4to3_tap3_420p8",           # 4:3
    "irregular_up_crop_mpeg1",     # general ratio with a crop
    "topleft_negative_crop",       # negative crop size
    "yv411_tap5",                  # 4:1:1
    "rgbap12_2x_tap6",             # alpha plane on the luma table
)] + [("odd_sizes_y", ah.Format("y", 8), 157, 93, 311, 187, dict(tap=3, src_left=0.4))]


@pytest.mark.gpu
@pytest.mark.parametrize("case", PASS_CASES, ids=[c[0] for c in PASS_CASES])
def test_pass_matches_definition(gpu, case):
    """jinc_antiring_plane_device on a GPU-resized plane against the NumPy pass on that same plane, for every table of the
    geometry and every sample type: identical at s = 1, within 1 LSB / 1 ulp at s = 0.25 and 0.5.  The table's positions
    are the float32 re-accumulation of the oracle's, and every anchor lies in the output pixel's own window."""
    import torch

    name, fmt, w, h, tw, th, kw = case
    ctx = gpu.Context(0)
    rng = np.random.default_rng(0x414E5449)
    for k, tp in enumerate(oracle_tables(fmt, w, h, tw, th, **kw)):
        tp = tp.params
        t = device_table(gpu, ctx, tp, kw.get("tap", 3), kw.get("blur", 0.0))
        px, py = ref_positions(tp)
        fs = t.info.filter_size
        for axis, pos, n in ((0, px, tp.src_w), (1, py, tp.src_h)):
            start, _, _, tpos = t.axis(axis)
            assert np.array_equal(tpos.view(np.uint32), pos.view(np.uint32)), f"{name}/table{k}: axis {axis} positions"
            a0, a1 = anchors(pos, n)
            assert ((a0 >= start) & (a1 <= start + fs - 1)).all(), f"{name}/table{k}: axis {axis} anchor outside the window"
        for kind, dtype, code, bits in SAMPLES:
            src = noise(rng, (tp.src_h, tp.src_w), dtype, bits)
            d_src = DevPlane(src)
            d_dst = DevPlane.empty(tp.dst_h, tp.dst_w, dtype)
            t.resize_device(code, peak_of(dtype, bits), d_src.ptr, d_src.pitch, d_dst.ptr, d_dst.pitch)
            y = d_dst.get()
            for s in (1.0, 0.5, 0.25):
                d_dst.set(y)
                t.antiring_device(code, s, d_src.ptr, d_src.pitch, d_dst.ptr, d_dst.pitch)
                assert_pass_equal(d_dst.get(), antiring_ref(y, src, px, py, s), s == 1.0, f"{name}/table{k}/{kind}/s={s}")
            d_dst.set(y)  # s = 0 is a no-op
            t.antiring_device(code, 0.0, d_src.ptr, d_src.pitch, d_dst.ptr, d_dst.pitch)
            assert np.array_equal(d_dst.get().view(np.uint8), y.view(np.uint8)), f"{name}/table{k}/{kind}: s = 0 changed the plane"
        t.close()
    torch.cuda.synchronize()
    ctx.close()


# ------------------------------------------------------------------------------------------ the filter pipeline

def make_filter(capi, fmt, w, h, tw, th, kind="int", **kw):
    """The filter of fmt's plane layout; kind "f16" makes it a half filter."""
    sw, sh = fmt.subsampling
    code, bits = (0x102, 16) if kind == "f16" else (np.dtype(fmt.dtype).itemsize, fmt.bits)
    return capi.Filter(src_w=w, src_h=h, target_w=tw, target_h=th, n_planes=len(fmt.planes), sample_bytes=code, bits=bits,
                       sub_w=sw, sub_h=sh, src_left=kw.get("src_left", 0.0), src_top=kw.get("src_top", 0.0),
                       src_width=kw.get("src_width"), src_height=kw.get("src_height"), quant_x=kw.get("quant_x", 256),
                       quant_y=kw.get("quant_y", 256), tap=kw.get("tap", 3), blur=kw.get("blur", 0.0),
                       cplace=kw.get("cplace", "mpeg2"), devices=[0], slots_per_device=kw.get("slots_per_device", 0),
                       flags=kw.get("flags", 0))


def frame_planes(fmt, w, h, seed, half=False):
    rng = np.random.default_rng(0x52494E47 ^ seed)
    out = []
    for i in range(len(fmt.planes)):
        shape = fmt.plane_shape(i, w, h)
        if half:
            out.append(rng.random(shape, dtype=np.float32).astype(np.float16))
        else:
            out.append(noise(rng, shape, fmt.dtype, fmt.bits))
    return out


def ref_frame(fmt, w, h, tw, th, planes, ys, s, **kw):
    """The NumPy pass over every plane of a frame whose resized planes are ys."""
    tables = [t.params for t in oracle_tables(fmt, w, h, tw, th, **kw)]
    out = []
    for i, (p, y) in enumerate(zip(planes, ys)):
        tp = tables[1] if (len(tables) > 1 and i in (1, 2)) else tables[0]
        px, py = ref_positions(tp)
        out.append(antiring_ref(y, p, px, py, s))
    return out


ORACLE_CASES = ["c1_yv12_2x_tap3", "c3_444p16_2x_tap4_crop", "c4_rgbps_2x_tap8", "c5_420p10_quarter_tap6_blur",
                "irregular_up_crop_mpeg1", "up1p5_tap3_420p8", "down2to3_tap4_y16", "yv411_tap5", "yuva420_14bit_2x"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ORACLE_CASES)
def test_filter_against_oracle(gpu, name):
    """jinc_filter_process with antiring 1 and 0.5 against the NumPy pass over the oracle's frame, within the parity bars
    (+-1 LSB; float 1e-5 relative to max(1, |ref|))."""
    _, fmt, w, h, tw, th, kw = SMALL[name]
    planes = frame_planes(fmt, w, h, seed=1)
    ys, _ = oracle_frame(fmt, w, h, tw, th, planes, **kw)
    flt = make_filter(gpu, fmt, w, h, tw, th, **kw)
    for s in (1.0, 0.5):
        flt.set_antiring(s)
        got = flt.process(planes)
        for i, (g, r) in enumerate(zip(got, ref_frame(fmt, w, h, tw, th, planes, ys, s, **kw))):
            assert_plane_close(g, r, fmt.bits == 32, f"{name}/s={s}/plane{i}")
    flt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c1_yv12_2x_tap3", "yuva420_14bit_2x", "irregular_up_crop_mpeg1", "half_tap4_f32_444"])
def test_off_means_off(gpu, name):
    """Strength 0, and 1 set back to 0, give the untouched filter's bytes with the same launches; at s > 0 every frame
    launches one more kernel per table (per table and band for row bands)."""
    _, fmt, w, h, tw, th, kw = SMALL[name]
    planes = frame_planes(fmt, w, h, seed=2)

    def run(setup, bands=0):
        flt = make_filter(gpu, fmt, w, h, tw, th, **kw)
        setup(flt)
        l0 = flt.kernel_launches
        out = flt.process(planes, bands=bands)
        n = flt.kernel_launches - l0
        tables = flt.num_tables
        flt.close()
        return out, n, tables

    base, n0, tables = run(lambda f: None)
    for setup in (lambda f: f.set_antiring(0.0), lambda f: (f.set_antiring(1.0), f.set_antiring(0.0))):
        out, n, _ = run(setup)
        assert n == n0
        for a, b in zip(out, base):
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    _, n1, _ = run(lambda f: f.set_antiring(0.5))
    assert n1 == n0 + tables
    for bands in (2, 3):
        _, nb0, _ = run(lambda f: None, bands)
        _, nb1, _ = run(lambda f: f.set_antiring(1.0), bands)
        assert nb1 - nb0 == tables * len([b for b in gpu.row_bands(th, bands) if b[1] > b[0]])


def _pinned_like(arrays):
    import torch

    out = []
    for a in arrays:
        t = torch.empty(a.shape, dtype={np.uint8: torch.uint8, np.float32: torch.float32, np.float16: torch.float16,
                                        np.uint16: torch.int16}[a.dtype.type], pin_memory=True)
        v = t.numpy().view(a.dtype)
        v[...] = a
        out.append(v)
    return out


def device_frames(capi, flt, frames):
    """Frames (lists of numpy planes) in device memory: (ctypes Frame array, keep-alive)."""
    arr = (capi.Frame * len(frames))()
    keep = []
    for fi, planes in enumerate(frames):
        for i, ((_, dshape), p) in enumerate(zip(flt.plane_shapes(), planes)):
            s, d = DevPlane(p), DevPlane.empty(dshape[0], dshape[1], p.dtype)
            arr[fi].src[i], arr[fi].src_pitch[i] = s.ptr, s.pitch
            arr[fi].dst[i], arr[fi].dst_pitch[i] = d.ptr, d.pitch
            keep.append((s, d))
    return arr, keep


PATH_CASES = ["c1_yv12_2x_tap3", "c5_420p10_quarter_tap6_blur", "up1p5_tap3_420p8", "rgbap12_2x_tap6", "f32_444_3x_tap16"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", PATH_CASES)
def test_paths_agree(gpu, name):
    """At s = 1 and 0.5: whole frames, submit/wait, 2, 3 and 7 row bands from pageable and pinned memory, and a device
    batch give the same bytes; a frame submitted before a strength change keeps the old strength."""
    import torch

    _, fmt, w, h, tw, th, kw = SMALL[name]
    frames = [frame_planes(fmt, w, h, seed=10 + f) for f in range(3)]
    flt = make_filter(gpu, fmt, w, h, tw, th, **kw)
    want = {}
    for s in (1.0, 0.5):
        flt.set_antiring(s)
        whole = [flt.process(p) for p in frames]
        want[s] = whole
        dst = flt.alloc_dst()
        flt.wait(flt.submit(frames[0], dst))
        for a, b in zip(dst, whole[0]):
            assert np.array_equal(a, b), f"{name}/s={s}: submit/wait"
        for bands in (2, 3, 7):
            for pinned in (False, True):
                src = _pinned_like(frames[1]) if pinned else frames[1]
                out = _pinned_like(flt.alloc_dst()) if pinned else None
                out = flt.process(src, out, bands=bands)
                for a, b in zip(out, whole[1]):
                    assert np.array_equal(a, b), f"{name}/s={s}: {bands} bands, pinned={pinned}"
        arr, keep = device_frames(gpu, flt, frames)
        stream = torch.cuda.Stream()
        flt.process_device_batch(arr, 0, 3, 3, stream.cuda_stream)
        stream.synchronize()
        per = len(keep) // len(frames)
        for f in range(len(frames)):
            for i in range(per):
                assert np.array_equal(keep[f * per + i][1].get(), whole[f][i]), f"{name}/s={s}: batch frame {f} plane {i}"
    # strength changes between submissions
    flt.set_antiring(1.0)
    d0, d1 = flt.alloc_dst(), flt.alloc_dst()
    t0 = flt.submit(frames[0], d0)
    flt.set_antiring(0.5)
    t1 = flt.submit(frames[1], d1)
    flt.wait(t0)
    flt.wait(t1)
    for a, b in zip(d0, want[1.0][0]):
        assert np.array_equal(a, b), f"{name}: frame submitted at s = 1"
    for a, b in zip(d1, want[0.5][1]):
        assert np.array_equal(a, b), f"{name}: frame submitted at s = 0.5"
    # the single-frame device call: the pass at s = 1 with every part, and no pass with the interior part alone
    flt.set_antiring(1.0)
    arr, keep = device_frames(gpu, flt, frames[:1])
    l0 = flt.kernel_launches
    flt.process_device(arr[0], 0, 3, 3, stream.cuda_stream)
    stream.synchronize()
    assert flt.kernel_launches - l0 == 2 * flt.num_tables, f"{name}: process_device launches"
    for i, (_, d) in enumerate(keep):
        assert np.array_equal(d.get(), want[1.0][0][i]), f"{name}: process_device plane {i}"
    n = {}
    for s in (0.0, 1.0):
        flt.set_antiring(s)
        l0 = flt.kernel_launches
        flt.process_device(arr[0], 0, 3, 1, stream.cuda_stream)
        flt.process_device_batch(arr, 0, 3, 1, stream.cuda_stream)
        stream.synchronize()
        n[s] = flt.kernel_launches - l0
    assert n[1.0] == n[0.0], f"{name}: the interior part alone ran the pass ({n})"
    flt.close()


FULL = {c[0]: c for c in FULL_CASES}


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["config1", "config2", "config3", "config4", "config5"])
def test_full_size_bounds(gpu, name):
    """The five BASELINE configs at full size: at s = 1 every sample of every plane lies in [lo, hi] of its 2x2 source
    neighbourhood; at s = 0.5 it lies between the unclamped output and that bound."""
    _, fmt, w, h, tw, th, kw = FULL[name]
    kw = dict(kw, slots_per_device=1)
    planes = frame_planes(fmt, w, h, seed=4)
    flt = make_filter(gpu, fmt, w, h, tw, th, **kw)
    raw = flt.process(planes)
    flt.set_antiring(1.0)
    full = flt.process(planes)
    flt.set_antiring(0.5)
    half = flt.process(planes)
    flt.close()
    tables = [t.params for t in oracle_tables(fmt, w, h, tw, th, **kw)]
    for i, p in enumerate(planes):
        tp = tables[1] if (len(tables) > 1 and i in (1, 2)) else tables[0]
        lo, hi = bounds(p, *ref_positions(tp))
        y, c, m = (a.astype(np.float32) for a in (raw[i], full[i], half[i]))
        assert ((c >= lo) & (c <= hi)).all(), f"{name}/plane{i}: s = 1 outside [lo, hi]"
        assert (c != y).any(), f"{name}/plane{i}: nothing was clamped"
        tol = 0.5 if fmt.bits < 32 else 0.0  # the blend rounds to the nearest code value
        assert ((m >= np.minimum(y, c) - tol) & (m <= np.maximum(y, c) + tol)).all(), f"{name}/plane{i}: s = 0.5"


@pytest.mark.gpu
@pytest.mark.parametrize("tap", [3, 8])
@pytest.mark.parametrize("bits", [8, 32])
def test_step_edge_overshoot_removed(gpu, tap, bits):
    """A hard step (and a thin line) upscaled 2x overshoots at s = 0 and not at s = 1: the maximum is at most the
    input's, the minimum at least the input's.  A constant plane is unchanged by the pass."""
    fmt = ah.Format("y", bits)
    lo, hi = (16, 235) if bits == 8 else (0.0, 1.0)
    src = np.full((48, 64), lo, fmt.dtype)
    src[:, 32:] = hi
    src[24:, 16:19] = hi
    flt = make_filter(gpu, fmt, 64, 48, 128, 96, tap=tap)
    raw = flt.process([src])[0]
    flt.set_antiring(1.0)
    out = flt.process([src])[0]
    const = np.full_like(src, 37 if bits == 8 else 0.3)
    cout = flt.process([const])[0]
    flt.set_antiring(0.0)
    craw = flt.process([const])[0]
    flt.close()
    assert raw.max() > src.max() and raw.min() < src.min(), f"tap{tap}: no ringing to remove"
    assert out.max() <= src.max() and out.min() >= src.min(), f"tap{tap}: ringing left at s = 1"
    assert (cout == const[0, 0]).all(), f"tap{tap}: a constant plane does not stay constant"
    if bits == 8:
        assert np.array_equal(cout, craw), f"tap{tap}: the pass changed the resized constant plane"


# ------------------------------------------------------------------------------------------ special values

@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float16, np.float32], ids=["f16", "f32"])
def test_special_values(gpu, dtype):
    """NaN outputs stay NaN; NaN neighbours do not change a finite output; +-Inf stays +-Inf at s = 0.5 and becomes the
    bound at s = 1; +-65504 survives on half planes.  The pass is a pure function of (plane, source, table), so the
    planes here are written directly."""
    code = 0x102 if dtype == np.float16 else 4
    ctx = gpu.Context(0)
    W, H, TW, TH = 96, 64, 192, 128
    tp = oracle_tables(ah.Format("y", 32), W, H, TW, TH, tap=3)[0].params
    t = device_table(gpu, ctx, tp, 3, 0.0)
    px, py = ref_positions(tp)
    rng = np.random.default_rng(7)
    src = rng.random((H, W), dtype=np.float32).astype(dtype)
    src[10:12, 10:12] = np.nan                       # a whole 2x2 neighbourhood of NaN
    src[30, 40] = np.nan                             # one NaN neighbour
    src[50:52, 70:72] = dtype(65504.0) if dtype == np.float16 else dtype(3e38)
    y = (rng.random((TH, TW), dtype=np.float32) * 2 - 0.5).astype(dtype)
    y[5, 5], y[60, 100], y[61, 101] = np.nan, np.inf, -np.inf
    y[21, 21] = 0.25                                 # under the all-NaN neighbourhood
    y[60, 80] = 0.5                                  # next to the single NaN
    y[101:103, 141:143] = dtype(65504.0) if dtype == np.float16 else dtype(3e38)
    y[0, 0] = -dtype(65504.0) if dtype == np.float16 else -dtype(3e38)
    d_src = DevPlane(src)
    res = {}
    for s in (1.0, 0.5):
        d = DevPlane(y)
        t.antiring_device(code, s, d_src.ptr, d_src.pitch, d.ptr, d.pitch)
        res[s] = d.get()
        assert_pass_equal(res[s], antiring_ref(y, src, px, py, s), s == 1.0, f"{dtype.__name__}/s={s}")
    lo, hi = bounds(src, px, py)
    for s, out in res.items():
        assert np.array_equal(np.isnan(out), np.isnan(y)), s
    assert np.isnan(lo[21, 21]) and res[1.0][21, 21] == y[21, 21]
    assert np.isposinf(res[0.5][60, 100]) and np.isneginf(res[0.5][61, 101])
    assert res[1.0][60, 100] == hi[60, 100].astype(dtype) and res[1.0][61, 101] == lo[61, 101].astype(dtype)
    ax0, ax1 = anchors(px, W)
    ay0, ay1 = anchors(py, H)
    nb = src[np.ix_([ay0[60], ay1[60]], [ax0[80], ax1[80]])]
    assert np.isnan(nb).sum() == 1, "src[30, 40] must be one of the four anchors of output (60, 80)"
    fin = nb[~np.isnan(nb)].astype(np.float32)  # the finite neighbours alone decide
    assert res[1.0][60, 80] == np.clip(np.float32(0.5), fin.min(), fin.max()).astype(dtype)
    big = dtype(65504.0) if dtype == np.float16 else dtype(3e38)
    for out in res.values():
        assert (out[101:103, 141:143] == big).all() and np.isfinite(out[0, 0])
    t.close()
    ctx.close()


# ------------------------------------------------------------------------------------------ VapourSynth

VS_CASES = [
    ("gray8", "y", 8, 0, 0, 160, 96, 320, 192, dict(tap=3)),
    ("yuv420p8", "420", 8, 1, 1, 160, 90, 320, 180, dict(tap=3)),
    ("rgbh", "rgbp", 16, 0, 0, 128, 72, 256, 144, dict(tap=6)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", VS_CASES, ids=[c[0] for c in VS_CASES])
def test_vs_antiring_equals_c_abi(gpu, case):
    from jinc_b200 import paths
    from minihost import vs_host

    name, fam, bits, ssw, ssh, w, h, tw, th, kw = case
    half = fam == "rgbp"
    fmt = ah.Format(fam, bits if not half else 16)
    frames = [frame_planes(fmt, w, h, seed=30 + k, half=half) for k in range(2)]
    core = vs_host.Core()
    plugin = core.load_plugin(paths.vs_plugin())
    cf = {"y": vs_host.CF_GRAY, "rgbp": vs_host.CF_RGB}.get(fam, vs_host.CF_YUV)
    src = core.source(cf, np.float16 if half else fmt.dtype, bits, ssw, ssh, w, h, frames)
    clip = plugin.invoke("JincResize", src, width=tw, height=th, antiring=1.0, **kw)
    flt = make_filter(gpu, fmt, w, h, tw, th, "f16" if half else "int", **kw)
    flt.set_antiring(1.0)
    plain = make_filter(gpu, fmt, w, h, tw, th, "f16" if half else "int", **kw)
    try:
        for k, planes in enumerate(frames):
            got, _ = clip.get_frame(k)
            want = flt.process(planes)
            raw = plain.process(planes)
            assert any(not np.array_equal(a, b) for a, b in zip(want, raw)), f"{name}: antiring changed nothing"
            for i, (g, a) in enumerate(zip(got, want)):
                assert np.array_equal(g.view(np.uint8), a.view(np.uint8)), f"{name}: frame {k} plane {i}"
    finally:
        flt.close()
        plain.close()
        clip.release()
        src.release()


# ------------------------------------------------------------------------------------------ CPU suite

def test_vs_registers_antiring(native_built):
    from jinc_b200 import paths
    from minihost import vs_host

    plugin = vs_host.Core().load_plugin(paths.vs_plugin())
    assert plugin.function_args("JincResize").endswith("cplace:data:opt;antiring:float:opt;")


@pytest.mark.parametrize("value", [-0.1, 1.5, float("nan")], ids=["negative", "above_one", "nan"])
def test_vs_rejects_bad_antiring(native_built, value):
    """Checked with the other arguments, before any GPU work."""
    from jinc_b200 import paths
    from minihost import vs_host

    core = vs_host.Core()
    plugin = core.load_plugin(paths.vs_plugin())
    src = core.source(vs_host.CF_GRAY, np.uint8, 8, 0, 0, 64, 64, [[np.zeros((64, 64), np.uint8)]])
    try:
        with pytest.raises(vs_host.VsError) as e:
            plugin.invoke("JincResize", src, width=96, height=96, antiring=value)
        assert str(e.value) == VS_BAD_ANTIRING
    finally:
        src.release()


def test_c_abi_rejects_bad_arguments(capi):
    L = capi.lib()
    assert "jinc_filter_set_antiring" in capi.EXPORTS and "jinc_antiring_plane_device" in capi.EXPORTS
    assert L.jinc_abi_version() == 2
    assert C.sizeof(capi.FilterParams) == 176
    for s in (1.0, 0.0, -1.0, float("nan")):
        assert L.jinc_filter_set_antiring(None, s) == -1
        assert "null filter" in L.jinc_last_error().decode()
    for sb, s in ((1, 1.0), (1, 0.0), (3, 1.0), (0x104, 1.0), (1, float("nan"))):  # no table without a device
        assert L.jinc_antiring_plane_device(None, None, sb, s, None, 64, None, 64, None) == -1
        assert "null argument" in L.jinc_last_error().decode()


@pytest.mark.gpu
def test_plane_device_rejects_bad_arguments(gpu):
    """With a real table: a bad sample_bytes, or a strength that is NaN or outside [0, 1], fails with JINC_E_INVALID
    before anything is launched; strength 0 is a valid call."""
    L = gpu.lib()
    ctx = gpu.Context(0)
    tp = oracle_tables(ah.Format("y", 8), 64, 48, 128, 96, tap=3)[0].params
    t = device_table(gpu, ctx, tp, 3, 0.0)
    src, dst = DevPlane.empty(48, 64, np.uint8), DevPlane.empty(96, 128, np.uint8)
    for sb in (0, 3, 8, 0x101, 0x104):
        assert L.jinc_antiring_plane_device(ctx.handle, t.handle, sb, 1.0, src.ptr, src.pitch, dst.ptr, dst.pitch, None) == -1
        assert "sample_bytes" in L.jinc_last_error().decode()
    for s in (-0.5, 1.01, float("nan"), float("inf")):
        assert L.jinc_antiring_plane_device(ctx.handle, t.handle, 1, s, src.ptr, src.pitch, dst.ptr, dst.pitch, None) == -1
        assert "strength" in L.jinc_last_error().decode()
    assert L.jinc_antiring_plane_device(ctx.handle, t.handle, 1, 0.0, src.ptr, src.pitch, dst.ptr, dst.pitch, None) == 0
    t.close()
    ctx.close()


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not installed")
def test_antiring_kernels_are_built_without_spills():
    """antiring_pass for uint8, uint16, half and float, none with a stack frame (no spills)."""
    from jinc_b200 import paths

    if not os.path.exists(paths.cuda_lib()):
        pytest.fail("libjinc_b200.so missing: run __graft_entry__.build()")
    out = subprocess.run(["cuobjdump", "-res-usage", paths.cuda_lib()], capture_output=True, text=True, check=True).stdout
    found = {}
    lines = out.splitlines()
    for i, line in enumerate(lines):
        m = re.search(r"Function (_ZN7jinc_rs13antiring_passI(h|t|6__half|f)E\S*):", line)
        if m:
            found[m.group(2)] = lines[i + 1]
    assert set(found) == {"h", "t", "6__half", "f"}, found
    for k, usage in found.items():
        assert re.search(r"STACK:0\b", usage), (k, usage)
        assert int(re.search(r"REG:(\d+)", usage).group(1)) <= 64, (k, usage)
