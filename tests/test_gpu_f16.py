"""Half-precision (IEEE binary16) planes: JINC_SAMPLE_F16 through the C ABI and the VapourSynth formats GRAYH, YUV4xxPH
and RGBH.

A half sample is widened to float exactly when it is staged, the float kernels accumulate it in the same order as a float
plane, and the sum is rounded to the nearest half with no clamp.  So a half frame must be byte-identical to the float32
frame of the widened input, rounded to half (NumPy's float32 -> float16 cast rounds to nearest even as __float2half_rn
does); NaN and Inf propagate as they do on float planes.  The CPU tests at the end need no GPU."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from common import FULL_CASES, SMALL_CASES, oracle_frame
from minihost import avs_host as ah

PATH_GENERAL, PATH_UP2X, PATH_DOWN_INT, PATH_CELLS = 0, 1, 2, 4


@pytest.fixture(scope="module")
def capi(native_built):
    from jinc_b200 import capi as c

    return c


@pytest.fixture(scope="module")
def gpu(capi):
    assert capi.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    return capi


def _filter(capi, fmt, w, h, tw, th, half, **kw):
    """The filter of `fmt`'s plane layout with half (JINC_SAMPLE_F16) or float32 samples."""
    sw, sh = fmt.subsampling
    return capi.Filter(src_w=w, src_h=h, target_w=tw, target_h=th, n_planes=len(fmt.planes),
                       sample_bytes=capi.SAMPLE_F16 if half else 4, bits=16 if half else 32, sub_w=sw, sub_h=sh,
                       src_left=kw.get("src_left", 0.0), src_top=kw.get("src_top", 0.0), src_width=kw.get("src_width"),
                       src_height=kw.get("src_height"), quant_x=kw.get("quant_x", 256), quant_y=kw.get("quant_y", 256),
                       tap=kw.get("tap", 3), blur=kw.get("blur", 0.0), cplace=kw.get("cplace", "mpeg2"), devices=[0],
                       slots_per_device=kw.get("slots_per_device", 0))


def half_planes(fmt, w, h, seed=0):
    """Seeded float16 noise: [0, 1) for luma, RGB and alpha, [-0.5, 0.5) for chroma."""
    rng = np.random.default_rng(0x46313620 ^ seed)
    planes = []
    for i in range(len(fmt.planes)):
        ph, pw = fmt.plane_shape(i, w, h)
        chroma = i in (1, 2) and fmt.family not in ("rgbp", "rgbap")
        planes.append(np.ascontiguousarray((rng.random((ph, pw), dtype=np.float32) - (0.5 if chroma else 0.0)).astype(np.float16)))
    return planes


def to_half(a):
    with np.errstate(over="ignore"):  # sums of magnitude >= 65520 round to +-Inf, as on the GPU
        return a.astype(np.float16)


def assert_rounded_identical(out16, out32, what):
    """out16 is out32 rounded to half, bit for bit; NaN positions are compared as a set (their payloads are not)."""
    assert out16.dtype == np.float16 and out16.shape == out32.shape, (what, out16.dtype, out16.shape, out32.shape)
    want = to_half(out32)
    nan = np.isnan(out16)
    assert np.array_equal(nan, np.isnan(want)), f"{what}: NaN positions differ"
    a, b = out16.view(np.uint16)[~nan], want.view(np.uint16)[~nan]
    bad = a != b
    assert not bad.any(), f"{what}: {int(bad.sum())} samples differ from the rounded float32 output"


def half_ulps(a, b):
    """Distance in half ulps (ordered bit patterns; +0 and -0 coincide)."""
    def ordered(x):
        bits = x.view(np.uint16).astype(np.int32)
        mag = bits & 0x7FFF
        return np.where(bits & 0x8000, -mag, mag)
    return np.abs(ordered(a) - ordered(b))


def _run(capi, case, half, planes, bands=0):
    _, fmt, w, h, tw, th, kw = case
    flt = _filter(capi, fmt, w, h, tw, th, half, **kw)
    out = flt.process([p.copy() for p in planes], bands=bands)
    paths = [flt.table(k).info.fast_path for k in range(flt.num_tables)]
    flt.close()
    return out, paths


# ------------------------------------------------------------------------------------------ byte identity with float32

def device_frames(capi, flt, frames, dtype):
    """Uploads `frames` (lists of numpy planes) into pitched torch tensors of `dtype`; returns (ctypes Frame array,
    keep-alive, dst tensors)."""
    import torch

    tdt = {np.float16: torch.float16, np.float32: torch.float32}[dtype]
    sb = np.dtype(dtype).itemsize
    arr = (capi.Frame * len(frames))()
    keep, dsts = [], []
    for fi, planes in enumerate(frames):
        dd = []
        for i, ((sshape, dshape), p) in enumerate(zip(flt.plane_shapes(), planes)):
            sp = (sshape[1] * sb + 255) // 256 * 256 // sb
            dp = (dshape[1] * sb + 255) // 256 * 256 // sb
            s = torch.zeros((sshape[0], sp), dtype=tdt, device="cuda")
            s[:, : sshape[1]].copy_(torch.from_numpy(p.astype(dtype)))
            d = torch.full((dshape[0], dp), 7, dtype=tdt, device="cuda")
            arr[fi].src[i], arr[fi].src_pitch[i] = s.data_ptr(), sp * sb
            arr[fi].dst[i], arr[fi].dst_pitch[i] = d.data_ptr(), dp * sb
            keep.append(s)
            dd.append(d)
        dsts.append(dd)
    torch.cuda.synchronize()
    return arr, keep, dsts


@pytest.mark.gpu
@pytest.mark.parametrize("case", SMALL_CASES, ids=[c[0] for c in SMALL_CASES])
def test_half_equals_rounded_float32(gpu, case):
    """Every small geometry (every kernel family, crops, chroma sitings, quant != 256, blur, 4:1:1, four planes, odd
    sizes) in its plane layout as half and as float32: whole frames, 2 and 7 row bands, and a device-resident batch."""
    name = case[0]
    _, fmt, w, h, tw, th, kw = case
    planes = half_planes(fmt, w, h, seed=3)
    wide = [p.astype(np.float32) for p in planes]
    out32, paths32 = _run(gpu, case, False, wide)
    out16, paths16 = _run(gpu, case, True, planes)
    assert paths16 == paths32, f"{name}: half took kernel families {paths16}, float32 {paths32}"
    for i, (a, b) in enumerate(zip(out16, out32)):
        assert np.array_equal(a.view(np.uint16), to_half(b).view(np.uint16)), f"{name}: plane {i} is not float32 rounded to half"
    for bands in (2, 7):
        banded, _ = _run(gpu, case, True, planes, bands=bands)
        for i, (a, b) in enumerate(zip(banded, out32)):
            assert np.array_equal(a.view(np.uint16), to_half(b).view(np.uint16)), f"{name}: plane {i}, {bands} row bands"

    import torch

    F = 3
    frames = [half_planes(fmt, w, h, seed=40 + f) for f in range(F)]
    flt16 = _filter(gpu, fmt, w, h, tw, th, True, **kw)
    flt32 = _filter(gpu, fmt, w, h, tw, th, False, **kw)
    arr, keep, dsts = device_frames(gpu, flt16, frames, np.float16)
    stream = torch.cuda.Stream()
    flt16.process_device_batch(arr, 0, 3, 3, stream.cuda_stream)
    stream.synchronize()
    shapes = flt16.plane_shapes()
    for f in range(F):
        want = flt32.process([p.astype(np.float32) for p in frames[f]])
        for i, b in enumerate(want):
            a = dsts[f][i][:, : shapes[i][1][1]].cpu().numpy()
            assert np.array_equal(a.view(np.uint16), to_half(b).view(np.uint16)), f"{name}: batch frame {f} plane {i}"
    flt16.close()
    flt32.close()


FULL = {c[0]: c for c in FULL_CASES}


@pytest.mark.gpu
@pytest.mark.parametrize("name,fmt", [("config2", ah.YUV420P8), ("config4", ah.RGBPS)])
def test_full_size_half_equals_rounded_float32(gpu, name, fmt):
    """Configs 2 (YUV420PH 1080p -> 2160p, tap 3) and 4 (RGBH 2160p -> 4320p, tap 8) as half: rows at the top, at the
    tile seams and at the bottom, and the left and right border columns over the full height."""
    _, cfmt, w, h, tw, th, kw = FULL[name]
    assert cfmt.family == fmt.family
    kw = dict(kw, slots_per_device=1)
    planes = half_planes(fmt, w, h, seed=11)
    out32, _ = _run(gpu, (name, fmt, w, h, tw, th, kw), False, [p.astype(np.float32) for p in planes])
    flt = _filter(gpu, fmt, w, h, tw, th, True, **kw)
    out16 = flt.process(planes)
    for i, (a, b) in enumerate(zip(out16, out32)):
        info = flt.table(1 if (flt.num_tables > 1 and i in (1, 2)) else 0).info
        assert info.fast_path == PATH_UP2X
        H = a.shape[0]
        rows = [(0, 5), (H // 2 - 3, H // 2 + 3), (H - 5, H)]
        rows += [(y, y + 2) for y in (31, 32, 63, 64, 255, 256, H // 3, 2 * H // 3) if y + 2 <= H]
        rows += [(max(0, info.interior_y0 - 2), info.interior_y0 + 2), (info.interior_y1 - 2, min(H, info.interior_y1 + 2))]
        for y0, y1 in rows:
            assert_rounded_identical(a[y0:y1], b[y0:y1], f"{name}/plane{i}/rows{y0}-{y1}")
        xl, xr = info.interior_x0 + 8, max(info.interior_x1 - 8, 0)
        assert_rounded_identical(np.ascontiguousarray(a[:, :xl]), b[:, :xl], f"{name}/plane{i}/left")
        assert_rounded_identical(np.ascontiguousarray(a[:, xr:]), b[:, xr:], f"{name}/plane{i}/right")
    flt.close()


# ------------------------------------------------------------------------------------------ special values

SPECIAL_CASES = [
    ("up2x", PATH_UP2X, ("up2x_y", ah.Format("y", 8), 200, 120, 400, 240, dict(tap=3))),
    ("down_int", PATH_DOWN_INT, ("half_y", ah.Format("y", 8), 640, 360, 320, 180, dict(tap=3))),
    ("cells", PATH_CELLS, ("up1p5_y", ah.Format("y", 8), 320, 180, 480, 270, dict(tap=3))),
    ("general", PATH_GENERAL, ("irregular_y", ah.Format("y", 8), 200, 120, 290, 170, dict(tap=4))),
]


def special_plane(w, h):
    """Noise with +-Inf, NaN, values near +-65504 and subnormals, and a step from 65504 to -65504 whose ringing
    overshoots the largest finite half."""
    rng = np.random.default_rng(5)
    p = rng.random((h, w), dtype=np.float32).astype(np.float16)
    p[10, 10], p[10, 40], p[40, 10] = np.inf, -np.inf, np.nan
    p[h - 3, w // 2] = np.nan  # a NaN whose window reaches the bottom border strip
    p[20:24, 60:66] = np.float16(65504.0)
    p[26:30, 60:66] = np.float16(-65504.0)
    p[30:34, 80:84] = np.float16(65000.0)
    tiny = np.array([2.0 ** -24, -(2.0 ** -24), 2.0 ** -20, 6.0e-5, -3.0e-6], np.float32).astype(np.float16)
    p[50:82, 20:52] = rng.choice(tiny, (32, 32))  # wider than the widest window here: outputs of subnormal sums
    p[5:9, w - 12:w - 4] = tiny[0]  # subnormals in the right border strip
    p[h // 2:h // 2 + 16, w // 2 - 8:w // 2] = np.float16(65504.0)  # the step
    p[h // 2:h // 2 + 16, w // 2:w // 2 + 8] = np.float16(-65504.0)
    return p


@pytest.mark.gpu
@pytest.mark.parametrize("kind,path,case", SPECIAL_CASES, ids=[c[0] for c in SPECIAL_CASES])
def test_specials_match_rounded_float32(gpu, kind, path, case):
    _, fmt, w, h, tw, th, kw = case
    plane = special_plane(w, h)
    out32, paths32 = _run(gpu, case, False, [plane.astype(np.float32)])
    out16, paths16 = _run(gpu, case, True, [plane])
    assert paths16 == paths32 == [path], (kind, paths16, paths32)
    a, b = out16[0], out32[0]
    assert_rounded_identical(a, b, kind)
    assert np.isnan(a).any() and np.isposinf(a).any() and np.isneginf(a).any(), kind
    overflow = np.isinf(a) & np.isfinite(b)  # a finite float32 sum of finite inputs that rounds to Inf
    assert overflow.any(), f"{kind}: no finite sum overflowed to Inf"
    tiny = (a != 0) & (np.abs(a) < np.float16(6.104e-5))
    assert tiny.any(), f"{kind}: no subnormal output"


# ------------------------------------------------------------------------------------------ against the oracle

ORACLE_CASES = ["c1_yv12_2x_tap3", "c3_444p16_2x_tap4_crop", "c4_rgbps_2x_tap8", "c5_420p10_quarter_tap6_blur",
                "irregular_up_crop_mpeg1", "up1p5_tap3_420p8", "down2to3_tap4_y16", "up4x_tap3_420p8",
                "rgbap10_irregular_up"]
SMALL = {c[0]: c for c in SMALL_CASES}


@pytest.mark.gpu
@pytest.mark.parametrize("name", ORACLE_CASES)
def test_half_against_oracle(gpu, name):
    """float16(the oracle's float32 result on the widened input) within one half ulp of the half output wherever
    |result| >= 2^-6: there a half ulp (>= 2^-16) exceeds the float parity bar of 1e-5 relative to max(1, |result|).
    Closer to zero, where cancelling sums leave float32 rounding noise of many (subnormal) half ulps, the half output
    is within that float bar of the oracle plus half a half ulp of rounding."""
    case = SMALL[name]
    _, fmt, w, h, tw, th, kw = case
    planes = half_planes(fmt, w, h, seed=9)
    out16, _ = _run(gpu, case, True, planes)
    ref, _ = oracle_frame(ah.Format(fmt.family, 32), w, h, tw, th, [p.astype(np.float32) for p in planes], **kw)
    for i, (a, r) in enumerate(zip(out16, ref)):
        big = np.abs(r) >= 2.0 ** -6
        d = np.where(big, half_ulps(a, to_half(r)), 0)
        assert d.max() <= 1, f"{name}/plane{i}: {int(d.max())} half ulps at {np.unravel_index(d.argmax(), d.shape)}"
        err = np.abs(a.astype(np.float64) - r.astype(np.float64))[~big]
        assert (err <= 1e-5 + 2.0 ** -18).all(), f"{name}/plane{i}: {err.max():.3e} from the oracle near zero"


# ------------------------------------------------------------------------------------------ VapourSynth

VS_HALF = [
    ("grayh", "y", 0, 0, 160, 96, 320, 192, dict(tap=3)),
    ("yuv420ph_mpeg2", "420", 1, 1, 160, 90, 320, 180, dict(tap=3, cplace="mpeg2")),
    ("yuv420ph_topleft", "420", 1, 1, 200, 120, 300, 180, dict(tap=4, cplace="topleft")),
    ("rgbh", "rgbp", 0, 0, 128, 72, 256, 144, dict(tap=6)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", VS_HALF, ids=[c[0] for c in VS_HALF])
def test_vs_half_clips(gpu, case):
    """GRAYH, YUV420PH and RGBH through core.jinc.JincResize: 16-bit float out, frames equal to the C-ABI half path
    (and so to float32 rounded to half)."""
    from jinc_b200 import paths
    from minihost import vs_host

    name, fam, ssw, ssh, w, h, tw, th, kw = case
    fmt = ah.Format(fam, 16)
    frames = [half_planes(fmt, w, h, seed=20 + k) for k in range(2)]
    core = vs_host.Core()
    plugin = core.load_plugin(paths.vs_plugin())
    cf = {"y": vs_host.CF_GRAY, "rgbp": vs_host.CF_RGB}.get(fam, vs_host.CF_YUV)
    src = core.source(cf, np.float16, 16, ssw, ssh, w, h, frames)
    clip = plugin.invoke("JincResize", src, width=tw, height=th, **kw)
    flt16 = _filter(gpu, fmt, w, h, tw, th, True, **kw)
    flt32 = _filter(gpu, fmt, w, h, tw, th, False, **kw)
    try:  # release the clips whatever happens: the core counts live frames and nodes for every later test
        assert clip.format == (vs_host.ST_FLOAT, 16) and clip.info["bytes_per_sample"] == 2
        for k, planes in enumerate(frames):
            got, _ = clip.get_frame(k)
            want = flt16.process(planes)
            wide = flt32.process([p.astype(np.float32) for p in planes])
            for i, (g, a, b) in enumerate(zip(got, want, wide)):
                assert g.dtype == np.float16
                assert np.array_equal(g.view(np.uint16), a.view(np.uint16)), f"{name}: frame {k} plane {i} differs from the C ABI"
                assert np.array_equal(g.view(np.uint16), to_half(b).view(np.uint16)), f"{name}: frame {k} plane {i}"
    finally:
        flt16.close()
        flt32.close()
        clip.release()
        src.release()


# ------------------------------------------------------------------------------------------ CPU suite

VS_BAD_FLOAT = "JincResize: only 8..16 bit integer, 16 bit float and 32 bit float input is supported."


@pytest.mark.parametrize("bits,dtype", [(8, np.float16), (24, np.float32)])
def test_vs_rejects_other_float_depths(native_built, bits, dtype):
    from jinc_b200 import paths
    from minihost import vs_host

    core = vs_host.Core()
    plugin = core.load_plugin(paths.vs_plugin())
    src = core.source(vs_host.CF_GRAY, dtype, bits, 0, 0, 64, 64, [[np.zeros((64, 64), dtype)]])
    assert src.format == (vs_host.ST_FLOAT, bits)
    try:
        with pytest.raises(vs_host.VsError) as e:
            plugin.invoke("JincResize", src, width=96, height=96)
        assert str(e.value) == VS_BAD_FLOAT
    finally:
        src.release()


def test_half_filter_needs_16_bits(capi):
    """JINC_SAMPLE_F16 with bits != 16 fails with JINC_E_INVALID while the parameters are checked, before any device is
    touched; the other sample sizes keep their rules."""
    assert capi.SAMPLE_F16 == 0x102 and capi.DTYPES[capi.SAMPLE_F16] is np.float16
    for bits in (0, 8, 10, 15, 17, 32):
        with pytest.raises(capi.JincError, match=r"^\[-1\] .*bits per component"):
            capi.Filter(src_w=64, src_h=64, target_w=128, target_h=128, n_planes=1, sample_bytes=capi.SAMPLE_F16, bits=bits,
                        devices=[0])
    for sb in (0, 3, 8, 0x101, 0x104, 0x202):
        with pytest.raises(capi.JincError, match=r"^\[-1\] .*sample_bytes"):
            capi.Filter(src_w=64, src_h=64, target_w=128, target_h=128, n_planes=1, sample_bytes=sb, bits=16, devices=[0])
    if capi.device_count() == 0:  # valid parameters get as far as looking for a device
        with pytest.raises(capi.JincError, match=r"^\[-2\]"):
            capi.Filter(src_w=64, src_h=64, target_w=128, target_h=128, n_planes=1, sample_bytes=capi.SAMPLE_F16, bits=16,
                        devices=[0])


def _sass_per_kernel(lib_path):
    out = subprocess.run(["cuobjdump", "-sass", lib_path], capture_output=True, text=True, check=True).stdout
    counts, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            counts[cur] = 0
        elif cur is not None and re.search(r"\bFFMA2\b", line):
            counts[cur] += 1
    names = subprocess.run(["c++filt"], input="\n".join(counts), capture_output=True, text=True, check=True).stdout.split("\n")
    return {n: counts[k] for n, k in zip(names, counts)}


@pytest.mark.skipif(shutil.which("cuobjdump") is None or shutil.which("c++filt") is None, reason="cuobjdump not installed")
def test_half_kernels_are_built():
    """The library holds __half instantiations of every kernel family, and the exact-2x ones multiply every tap: their
    FFMA2 count is that of the float kernels (no tap mask of the integer planes leaked in)."""
    from jinc_b200 import paths

    if not os.path.exists(paths.cuda_lib()):
        pytest.fail("libjinc_b200.so missing: run __graft_entry__.build()")
    n = _sass_per_kernel(paths.cuda_lib())
    for fs in (7, 9, 11, 13, 15, 17):
        for ox, oy in ((0, 0), (0, 1), (1, 0), (1, 1)):
            sig = f", {fs}, {ox}, {oy}, false, 0>(jinc_rs::UpArgs, jinc_rs::UpWeights<{fs}>)"
            half, flt = n.get(f"void jinc_rs::resample_up2x<__half{sig}"), n.get(f"void jinc_rs::resample_up2x<float{sig}")
            assert half is not None and flt is not None, (fs, ox, oy)
            assert half == flt, (fs, ox, oy, half, flt)
            if fs <= 9:
                assert half == 4 * 4 * fs * fs, (fs, half)
    for k in n:  # neither a tap-mask variant nor bulk-copy staging for half planes
        m = re.match(r"void jinc_rs::resample_up2x<__half, \d+, [01], [01], (\w+), (\d+)>", k)
        assert m is None or m.groups() == ("false", "0"), k
    for kern in ("jinc_rs::resample_down<__half,", "jinc_rs::resample_cells<__half,", "resample_strips<__half,"):
        assert any(kern in k for k in n), kern
