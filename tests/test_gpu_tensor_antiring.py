"""Differentiable anti-ringing: jinc_antiring_planes_device, jinc_antiring_adjoint_planes_device and
jinc_resize(..., antiring=).

The backward of resize + clamp (DESIGN.md §4.9) is defined per output sample from the stored resized sample y, its four
anchors a0..a3 and lo / hi = fmin / fmax over them: inside (y NaN or lo <= y <= hi) g_y = g; below / above g_y = (1 - s) g
(+0 at s = 1) and s g (g at s = 1) goes to the first anchor in a0..a3 order equal to lo / hi; grad_src = A^T g_y + r, r the
routed values summed in row-major output order from the first one.  `rule_reference` restates that in float32 NumPy and
takes A^T g_y from jinc_resize_adjoint_planes_device, so the kernels are checked bit for bit.  The CPU tests at the top
need no GPU: they check the rule against finite differences of a float64 model and the monotone positions the gather's
binary search relies on."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from common import FULL_CASES, SMALL_CASES
from test_gpu_antiring import VS_BAD_ANTIRING, anchors, ref_positions
from test_gpu_tensor_adjoint import geometries, gpu_table, oracle_table, sparse_chunks

SMALL = {c[0]: c for c in SMALL_CASES}
FULL = {c[0]: c for c in FULL_CASES}


# ------------------------------------------------------------------------------------------ CPU tests

FD_CASES = ["c1_yv12_2x_tap3", "half_tap3_yv12", "irregular_up_crop_mpeg1", "up1p5_tap3_f32_y", "topleft_negative_crop"]


def dense_model(ot):
    """A as one float64 CSR matrix (outputs x source samples) from the oracle's weights."""
    import scipy.sparse as sp

    parts = [m for _, m, _ in sparse_chunks(ot)]
    return sp.vstack(parts).tocsr()


def model_forward(A, src, ax, ay, s):
    """float64 resize + clamp: (out, y, lo, hi, anchor values (4, n), anchor flat indices (4, n))."""
    H, W = src.shape
    ax0, ax1 = ax
    ay0, ay1 = ay
    idx = np.stack([(ay0[:, None] * W + ax0[None, :]), (ay0[:, None] * W + ax1[None, :]),
                    (ay1[:, None] * W + ax0[None, :]), (ay1[:, None] * W + ax1[None, :])]).reshape(4, -1)
    y = A @ src.ravel()
    a = src.ravel()[idx]
    lo, hi = a.min(0), a.max(0)
    c = np.clip(y, lo, hi)
    return s * c + (1 - s) * y, y, lo, hi, a, idx


@pytest.mark.parametrize("name", FD_CASES)
def test_rule_is_the_derivative(native_built, name):
    """Central finite differences of the float64 resize + clamp equal the rule's gradient along random directions, at
    strengths 0.3 and 1, on inputs without ties.  The step is far below every distance to a kink, where the map is linear,
    so the difference quotient is exact up to float64 rounding."""
    rng = np.random.default_rng(0x46440A)
    for label, (H, W), args, p, tap, blur in geometries(SMALL[name]):
        ot = oracle_table(p, tap, blur)
        A = dense_model(ot)
        ot.close()
        px, py = ref_positions(p)
        ax, ay = anchors(px, W), anchors(py, H)
        src = rng.random((H, W))
        src[:, : W // 3] += 2.0  # a hard step: outputs beside it overshoot and are clamped
        g = rng.standard_normal(p.dst_h * p.dst_w)
        for s in (0.3, 1.0):
            out, y, lo, hi, a, idx = model_forward(A, src, ax, ay, s)
            below, above = y < lo, y > hi
            assert below.any() and above.any() and (~(below | above)).any(), label
            gy = np.where(below | above, (1 - s) * g, g)
            r = np.zeros(H * W)
            k = np.argmax(a == np.where(below, lo, hi)[None, :], axis=0)  # first anchor equal to the bound
            sel = below | above
            np.add.at(r, idx[k, np.arange(idx.shape[1])][sel], s * g[sel])
            grad = A.T @ gy + r
            # distance to the nearest kink: y reaching lo / hi, or two anchors crossing
            srt = np.sort(a, axis=0)
            margin = min(np.abs(y - lo).min(), np.abs(y - hi).min(), np.diff(srt, axis=0)[np.diff(srt, axis=0) > 0].min())
            for _ in range(3):
                d = rng.choice([-1.0, 1.0], size=(H, W))
                reach = np.abs(A) @ np.abs(d.ravel())
                eps = 0.01 * margin / max(1.0, float(reach.max()))
                f = lambda v: float(g @ model_forward(A, v, ax, ay, s)[0])
                fd = (f(src + eps * d) - f(src - eps * d)) / (2 * eps)
                want = float(grad @ d.ravel())
                scale = float(np.abs(g).sum() * 4)
                assert abs(fd - want) <= 1e-6 * scale + 1e-16 * float(np.abs(g).sum()) * np.abs(out).max() / eps, \
                    (label, s, fd, want, eps)


@pytest.mark.parametrize("case", SMALL_CASES + FULL_CASES, ids=[c[0] for c in SMALL_CASES + FULL_CASES])
def test_floored_positions_are_non_decreasing(native_built, case):
    """The gather finds the outputs a source sample anchors by binary search on floor(pos): it must never decrease."""
    for label, _, _, p, tap, blur in geometries(case):
        for pos in ref_positions(p):
            assert (np.diff(np.floor(pos.astype(np.float64))) >= 0).all(), label


def test_host_side_validation():
    """Checked before the device: a bad strength is a ValueError with the VapourSynth filter's text; a CPU tensor with a
    valid one still has no CPU path."""
    import torch

    from jinc_b200.tensor import jinc_resize

    for bad in (float("nan"), -0.1, 1.5):
        with pytest.raises(ValueError) as e:
            jinc_resize(torch.zeros(8, 8), 16, 16, antiring=bad)
        assert str(e.value) == VS_BAD_ANTIRING.replace("JincResize", "jinc_resize")
    for ok in (0.0, 0.5, 1.0):
        with pytest.raises(ValueError, match="no CPU path"):
            jinc_resize(torch.zeros(8, 8), 16, 16, antiring=ok)


@pytest.mark.skipif(shutil.which("cuobjdump") is None and not os.path.exists("/usr/local/cuda/bin/cuobjdump"),
                    reason="cuobjdump not installed")
def test_adjoint_kernels_are_built_without_spills(native_built):
    from jinc_b200 import paths

    lib = paths.cuda_lib()
    if not os.path.exists(lib):
        pytest.fail("libjinc_b200.so missing: run __graft_entry__.build()")
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    lines = subprocess.run([tool, "-res-usage", lib], capture_output=True, text=True, check=True).stdout.splitlines()
    found = {}
    for i, line in enumerate(lines):
        m = re.search(r"Function (\S*(antiring_grad_out|antiring_route_gather)I(f|6__half)E\S*):", line)
        if m:
            found[(m.group(2), m.group(3))] = lines[i + 1]
    assert set(found) == {(k, t) for k in ("antiring_grad_out", "antiring_route_gather") for t in ("f", "6__half")}, found
    for k, usage in found.items():
        assert "LOCAL:0" in usage and re.search(r"STACK:0\b", usage), (k, usage)


# ------------------------------------------------------------------------------------------ GPU helpers

@pytest.fixture(scope="module")
def gpu(native_built):
    from jinc_b200 import capi

    assert capi.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    return capi


@pytest.fixture(scope="module")
def ctx(gpu):
    return gpu.Context(0)


def stream():
    import torch

    from jinc_b200.tensor import _stream

    return _stream(torch.device("cuda", torch.cuda.current_device()))


def sample_code(capi, dtype):
    return {np.uint8: 1, np.uint16: 2, np.float16: capi.SAMPLE_F16, np.float32: 4}[np.dtype(dtype).type]


def resize_planes(tab, capi, x, h, w):
    """jinc_resize_planes_device on the (n, H, W) CUDA tensor x -> (n, h, pitch) tensor (rows padded to 16 bytes) and
    its (n, h, w) view."""
    import torch

    n, H, W = x.shape
    isz = x.element_size()
    pitch = (w * isz + 15) // 16 * 16 // isz
    y = torch.zeros((n, h, pitch), dtype=x.dtype, device=x.device)
    tab.resize_planes_device(sample_code(capi, x.cpu().numpy().dtype), 0.0 if x.is_floating_point() else
                             float(np.iinfo(x.cpu().numpy().dtype).max), n, x.data_ptr(), W * isz, H * W * isz,
                             y.data_ptr(), pitch * isz, h * pitch * isz, stream())
    return y, y[..., :w]


def antiring_adjoint(tab, capi, s, x, y, g):
    """jinc_antiring_adjoint_planes_device: x (n, H, W), y (n, h, pitch) as resize_planes returns it, g (n, h, w) float32
    -> (g_y, grad_src) float32."""
    import torch

    n, H, W = x.shape
    h, w = g.shape[1:]
    isz = x.element_size()
    gy = torch.full((n, h, w), float("nan"), device=x.device)
    gs = torch.full((n, H, W), float("nan"), device=x.device)
    g = g.contiguous()
    tab.antiring_adjoint_planes_device(sample_code(capi, np.float16 if x.dtype.itemsize == 2 else np.float32), s, n,
                                       (x.data_ptr(), W * isz, H * W * isz),
                                       (y.data_ptr(), y.stride(1) * isz, y.stride(0) * isz),
                                       (g.data_ptr(), w * 4, h * w * 4), (gy.data_ptr(), w * 4, h * w * 4),
                                       (gs.data_ptr(), W * 4, H * W * 4), stream())
    return gy, gs


def plain_adjoint(tab, g, H, W):
    import torch

    g = g.contiguous()
    n, h, w = g.shape
    out = torch.full((n, H, W), float("nan"), device=g.device)
    tab.adjoint_planes_device(n, g.data_ptr(), w * 4, h * w * 4, out.data_ptr(), W * 4, H * W * 4, stream())
    return out


def rule_reference(src, y, g, pos_x, pos_y, s, atg_of):
    """The rule in float32 NumPy for one plane: (g_y, grad_src).  atg_of(g_y) -> A^T g_y (the library's adjoint)."""
    H, W = src.shape
    if s == 0:  # off: g_y is g itself and nothing is routed
        return g.copy(), atg_of(g.copy()).reshape(H, W)
    S = src.astype(np.float32)
    Y = y.astype(np.float32)
    ax0, ax1 = anchors(pos_x, W)
    ay0, ay1 = anchors(pos_y, H)
    a = [S[ay0][:, ax0], S[ay0][:, ax1], S[ay1][:, ax0], S[ay1][:, ax1]]
    with np.errstate(invalid="ignore", over="ignore"):
        lo = np.fmin(np.fmin(a[0], a[1]), np.fmin(a[2], a[3]))
        hi = np.fmax(np.fmax(a[0], a[1]), np.fmax(a[2], a[3]))
        below, above = Y < lo, Y > hi
        routed = below | above
        s32 = np.float32(s)
        if s == 1:
            gy = np.where(routed, np.float32(0.0), g)
            val = g
        else:
            gy = np.where(routed, (np.float32(1.0) - s32) * g, g).astype(np.float32)
            val = (s32 * g).astype(np.float32)
        b = np.where(below, lo, hi)
        k = np.where(a[0] == b, 0, np.where(a[1] == b, 1, np.where(a[2] == b, 2, 3)))
        sx = np.where(k & 1, ax1[None, :], ax0[None, :])
        sy = np.where(k & 2, ay1[:, None], ay0[:, None])
        idx = (sy * W + sx)[routed]  # row-major output order
        v = val[routed]
        r = np.zeros(H * W, np.float32)
        has = np.zeros(H * W, bool)
        first = np.unique(idx, return_index=True)[1]
        r[idx[first]] = v[first]  # the sum starts from the first routed value (a routed -0.0 keeps its sign)
        has[idx[first]] = True
        rest = np.ones(len(idx), bool)
        rest[first] = False
        np.add.at(r, idx[rest], v[rest])
        atg = atg_of(gy.astype(np.float32)).ravel()
        gs = np.where(has, (atg + r).astype(np.float32), atg)
    return gy.astype(np.float32), gs.reshape(H, W).astype(np.float32)


def assert_bits(got, want, what):
    """Bit-identical, except that every NaN equals every NaN (the GPU's arithmetic returns the canonical NaN)."""
    assert got.shape == want.shape, (what, got.shape, want.shape)
    nan = np.isnan(got)
    assert np.array_equal(nan, np.isnan(want)), f"{what}: NaN positions differ ({int((nan != np.isnan(want)).sum())})"
    diff = got.view(np.uint32)[~nan] != want.view(np.uint32)[~nan]
    assert not diff.any(), f"{what}: {int(diff.sum())} samples differ"


def planes_and_gradients(H, W, h, w, rng, dtype):
    """Four source planes (noise, hard steps, plateaus with ties, special values) and their output gradients."""
    noise = rng.random((H, W), dtype=np.float32)
    yy, xx = np.mgrid[0:H, 0:W]
    steps = (((xx // 7) + (yy // 5)) % 2).astype(np.float32) * 3.0 - 1.0
    plateau = np.round(rng.random((H, W)) * 2).astype(np.float32) / 2  # three levels: many equal anchors
    special = rng.random((H, W), dtype=np.float32)
    special[(xx % 5 == 0) & (yy % 3 == 0)] = 1.0
    special[::11, ::13] = np.nan
    special[3::17, 5::19] = np.inf
    special[7::23, 2::29] = -np.inf
    special[1::7, 4::9] = -0.0
    src = np.stack([noise, steps, plateau, special]).astype(dtype)
    g = rng.standard_normal((4, h, w)).astype(np.float32)
    g[3, ::13, ::17] = np.nan
    g[3, 5::19, 3::11] = np.inf
    g[3, 9::31, 7::13] = -np.inf
    g[2, ::3, ::2] = -0.0
    return src, g


def check_case(gpu, ctx, label, H, W, p, tap, blur, dtype, strengths, rng, planes=None):
    import torch

    tab = gpu_table(gpu, ctx, p, tap, blur)
    h, w = p.dst_h, p.dst_w
    src, g = planes_and_gradients(H, W, h, w, rng, dtype)
    if planes is not None:
        src, g = src[planes], g[planes]
    x = torch.from_numpy(src).cuda()
    y, yv = resize_planes(tab, gpu, x, h, w)
    _, _, _, px = tab.axis(0)
    _, _, _, py = tab.axis(1)
    ys = yv.cpu().numpy()
    gt = torch.from_numpy(g).cuda()
    for s in strengths:
        gy, gs = antiring_adjoint(tab, gpu, s, x, y, gt)
        gy, gs = gy.cpu().numpy(), gs.cpu().numpy()
        for i in range(src.shape[0]):
            atg_of = lambda v: plain_adjoint(tab, torch.from_numpy(v).cuda()[None], H, W).cpu().numpy()[0]
            want_gy, want_gs = rule_reference(src[i], ys[i], g[i], px, py, s, atg_of)
            assert_bits(gy[i], want_gy, f"{label}/{np.dtype(dtype).name}/s={s}/plane {i}: g_y")
            assert_bits(gs[i], want_gs, f"{label}/{np.dtype(dtype).name}/s={s}/plane {i}: grad_src")
    tab.close()


# ------------------------------------------------------------------------------------------ forward

FWD_SAMPLES = [("u8", np.uint8, 8), ("u10", np.uint16, 10), ("u16", np.uint16, 16), ("f16", np.float16, 0),
               ("f32", np.float32, 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["c1_yv12_2x_tap3", "irregular_up_crop_mpeg1", "half_tap3_yv12"])
def test_batched_clamp_equals_per_plane_calls(gpu, ctx, case):
    """jinc_antiring_planes_device equals jinc_antiring_plane_device on each plane, byte for byte."""
    import torch

    for label, (H, W), args, p, tap, blur in geometries(SMALL[case]):
        tab = gpu_table(gpu, ctx, p, tap, blur)
        h, w = p.dst_h, p.dst_w
        for kind, dt, bits in FWD_SAMPLES:
            rng = np.random.default_rng(5)
            for n in (1, 3, 4, 5, 7):
                if dt in (np.float16, np.float32):
                    a = (rng.random((n, H, W)) * 2 - 0.5).astype(dt)
                else:
                    a = rng.integers(0, 1 << bits, (n, H, W)).astype(dt)
                a[:, :, : W // 2] = a[:, :, : W // 2] // 4 if a.dtype.kind == "u" else a[:, :, : W // 2] * 0.25
                x = torch.from_numpy(a).cuda()
                isz = x.element_size()
                pitch = (w * isz + 15) // 16 * 16
                code = sample_code(gpu, dt)
                peak = float((1 << bits) - 1) if bits else 0.0
                base = torch.zeros((n, h, pitch), dtype=torch.uint8, device="cuda")
                tab.resize_planes_device(code, peak, n, x.data_ptr(), W * isz, H * W * isz, base.data_ptr(), pitch,
                                         h * pitch, stream())
                for s in (0.3, 1.0):
                    batch, single = base.clone(), base.clone()
                    tab.antiring_planes_device(code, s, n, x.data_ptr(), W * isz, H * W * isz, batch.data_ptr(), pitch,
                                               h * pitch, stream())
                    for i in range(n):
                        tab.antiring_device(code, s, x[i].data_ptr(), W * isz, single[i].data_ptr(), pitch, stream())
                    torch.cuda.synchronize()
                    assert not torch.equal(batch, base), f"{label}/{kind}/n={n}/s={s}: nothing was clamped"
                    assert torch.equal(batch[..., : w * isz], single[..., : w * isz]), f"{label}/{kind}/n={n}/s={s}"
        tab.close()


VS_CASES = ["c1_yv12_2x_tap3", "irregular_up_crop_mpeg1", "half_tap3_yv12", "up1p5_tap3_f32_y"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", VS_CASES)
def test_tensor_forward_equals_vapoursynth_filter(gpu, name):
    """jinc_resize(x, antiring=s) on one plane equals core.jinc.JincResize(antiring=s) on a GRAY clip, byte for byte."""
    from jinc_b200 import paths
    from jinc_b200.tensor import jinc_resize
    from minihost import vs_host

    import torch

    _, fmt, w, h, tw, th, kw = SMALL[name]
    script = {k: v for k, v in kw.items() if k != "cplace"}
    core = vs_host.Core()
    vsp = core.load_plugin(paths.vs_plugin())
    rng = np.random.default_rng(17)
    for dt, bits in (("uint8", 8), ("uint16", 10), ("float32", 32), ("float16", 16)):
        if dt.startswith("float"):
            plane = (rng.random((h, w)) * 2 - 0.5).astype(dt)
        else:
            plane = rng.integers(0, 1 << min(bits, 16), (h, w)).astype(dt)
        for s in (0.3, 1.0):
            src = core.source(vs_host.CF_GRAY, np.dtype(dt), bits, 0, 0, w, h, [[plane]])
            clip = vsp.invoke("JincResize", src, width=tw, height=th, antiring=s, **script)
            (want,), _ = clip.get_frame(0)
            clip.release()
            src.release()
            got = jinc_resize(torch.from_numpy(plane).cuda(), tw, th, bits=bits if dt.startswith("uint") else None,
                              antiring=s, **script).cpu().numpy()
            assert np.array_equal(got.view(np.uint8), np.ascontiguousarray(want).view(np.uint8)), f"{name}/{dt}/s={s}"


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float32", "float16", "uint8"])
def test_antiring_zero_is_the_plain_path(gpu, dtype):
    import torch

    from jinc_b200.tensor import jinc_resize

    dt = getattr(torch, dtype)
    x0 = torch.rand((2, 90, 160), device="cuda")
    x0[:, :, :80] += 2.0
    x0 = x0.to(dt) if dt.is_floating_point else (x0 * 60).to(dt)
    if not dt.is_floating_point:
        assert torch.equal(jinc_resize(x0, 320, 180, antiring=0.0), jinc_resize(x0, 320, 180))
        return
    g = torch.randn((2, 180, 320), device="cuda").to(dt)
    a, b = x0.clone().requires_grad_(), x0.clone().requires_grad_()
    ya, yb = jinc_resize(a, 320, 180, antiring=0.0), jinc_resize(b, 320, 180)
    (ya * g).sum().backward()
    (yb * g).sum().backward()
    assert torch.equal(ya, yb) and torch.equal(a.grad, b.grad)
    assert not torch.equal(jinc_resize(x0, 320, 180, antiring=1.0), yb)


# ------------------------------------------------------------------------------------------ backward, bit for bit

@pytest.mark.gpu
@pytest.mark.parametrize("case", SMALL_CASES, ids=[c[0] for c in SMALL_CASES])
def test_backward_bits_against_the_rule(gpu, ctx, case):
    """g_y and grad_src of every table of every small case, float32 and half sources, strengths 0, 0.25 and 1, on noise,
    hard steps, plateaus (ties) and NaN / +-Inf / -0.0 in the source and NaN / +-Inf / -0.0 in g."""
    rng = np.random.default_rng(0x52554C45)
    for label, (H, W), args, p, tap, blur in geometries(case):
        for dtype in (np.float32, np.float16):
            check_case(gpu, ctx, label, H, W, p, tap, blur, dtype, (0.0, 0.25, 1.0), rng)


@pytest.mark.gpu
@pytest.mark.parametrize("name,strengths", [("config2", (0.25, 1.0)), ("config4", (1.0,))])
def test_full_size_backward_bits(gpu, ctx, name, strengths):
    """The same bit-identity on the full-size config 2 luma table and the config 4 table (noise and hard steps)."""
    rng = np.random.default_rng(0x46554C4C)
    label, (H, W), args, p, tap, blur = geometries(FULL[name])[0]
    check_case(gpu, ctx, f"{name}/{label}", H, W, p, tap, blur, np.float32, strengths, rng, planes=[0, 1])


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["c1_yv12_2x_tap3", "c4_rgbps_2x_tap8", "c5_420p10_quarter_tap6_blur", "up4x_tap3_420p8"])
def test_backward_bits_do_not_depend_on_batch_position(gpu, ctx, case):
    import torch

    for label, (H, W), args, p, tap, blur in geometries(SMALL[case]):
        tab = gpu_table(gpu, ctx, p, tap, blur)
        h, w = p.dst_h, p.dst_w
        x = torch.rand((9, H, W), device="cuda")
        x[:, :, : W // 2] += 1.0
        g = torch.randn((9, h, w), device="cuda")
        y, _ = resize_planes(tab, gpu, x, h, w)
        for s in (0.25, 1.0):
            gy9, gs9 = antiring_adjoint(tab, gpu, s, x, y, g)
            gy1, gs1 = antiring_adjoint(tab, gpu, s, x[6:7].clone(), y[6:7].clone(), g[6:7].clone())
            gy5, gs5 = antiring_adjoint(tab, gpu, s, x[2:7].clone(), y[2:7].clone(), g[2:7].clone())
            torch.cuda.synchronize()
            for what, a, b in (("g_y 1", gy1[0], gy9[6]), ("grad_src 1", gs1[0], gs9[6]), ("g_y 5", gy5[4], gy9[6]),
                               ("grad_src 5", gs5[4], gs9[6])):
                assert torch.equal(a.view(torch.int32), b.view(torch.int32)), (label, s, what)
        tab.close()


# ------------------------------------------------------------------------------------------ autograd

def c1_luma(gpu, ctx):
    label, (H, W), args, p, tap, blur = geometries(SMALL["c1_yv12_2x_tap3"])[0]
    return gpu_table(gpu, ctx, p, tap, blur), (H, W), args, p


def entry_point_grad(gpu, tab, x, g, s, h, w):
    """x.grad as the entry point gives it: resize, then jinc_antiring_adjoint_planes_device on the float32 gradient."""
    import torch

    xs = x.detach().reshape(-1, *x.shape[-2:])
    y, _ = resize_planes(tab, gpu, xs, h, w)
    _, gs = antiring_adjoint(tab, gpu, s, xs, y, g.float().reshape(-1, h, w))
    return gs.to(x.dtype).view(x.shape)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float32", "float16"])
def test_autograd_backward_is_the_entry_point(gpu, ctx, dtype):
    import torch

    from jinc_b200.tensor import jinc_resize

    tab, (H, W), args, p = c1_luma(gpu, ctx)
    dt = getattr(torch, dtype)
    for s in (0.4, 1.0):
        x0 = torch.rand((2, 3, H, W), device="cuda")
        x0[..., : W // 2] += 1.0
        x = x0.to(dt).requires_grad_()
        y = jinc_resize(x, antiring=s, **args)
        g = torch.randn(y.shape, device="cuda").to(dt)
        (y * g).sum().backward()
        want = entry_point_grad(gpu, tab, x, g, s, p.dst_h, p.dst_w)
        assert x.grad.dtype == dt and torch.equal(x.grad, want), s
    tab.close()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float32", "float16"])
def test_gradient_expanded_over_a_leading_dimension(gpu, ctx, dtype):
    import torch

    from jinc_b200.tensor import jinc_resize

    tab, (H, W), args, p = c1_luma(gpu, ctx)
    dt = getattr(torch, dtype)
    x0 = torch.rand((4, H, W), device="cuda")
    x0[..., : W // 3] -= 1.0
    x = x0.to(dt).requires_grad_()
    g = torch.randn((p.dst_h, p.dst_w), device="cuda").to(dt)
    (jinc_resize(x, antiring=1.0, **args).sum(0) * g).sum().backward()
    want = entry_point_grad(gpu, tab, x, g.expand(4, p.dst_h, p.dst_w), 1.0, p.dst_h, p.dst_w)
    assert torch.equal(x.grad, want)
    tab.close()


@pytest.mark.gpu
def test_in_place_on_output_works_and_on_input_raises(gpu):
    import torch

    from jinc_b200.tensor import jinc_resize

    x = torch.rand((2, 90, 160), device="cuda", requires_grad=True)
    g = torch.randn((2, 181, 318), device="cuda")
    y = jinc_resize(x, 318, 181, antiring=0.5)
    y.mul_(2.0)
    (y * g).sum().backward()
    ref = x.detach().clone().requires_grad_()
    (jinc_resize(ref, 318, 181, antiring=0.5) * (2.0 * g)).sum().backward()
    assert torch.equal(x.grad, ref.grad)

    leaf = torch.rand((2, 90, 160), device="cuda", requires_grad=True)
    x2 = leaf * 1.0
    y2 = jinc_resize(x2, 320, 180, antiring=1.0)
    x2.add_(1.0)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        y2.sum().backward()


@pytest.mark.gpu
def test_side_stream_needs_no_extra_synchronisation(gpu):
    import torch

    from jinc_b200.tensor import jinc_resize

    x0 = torch.rand((4, 270, 480), device="cuda")
    x0[..., :240] += 1.0
    xr = x0.clone().requires_grad_()
    ref_y = jinc_resize(xr, 960, 540, antiring=0.75)
    ref_y.square().sum().backward()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        x = torch.rand((4, 270, 480), device="cuda")
        x.copy_(x0)  # ordered on s only
        x.requires_grad_()
        y = jinc_resize(x, 960, 540, antiring=0.75)
        y.square().sum().backward()
        got_y, got_g = y.detach().clone(), x.grad.clone()
    torch.cuda.current_stream().wait_stream(s)
    assert torch.equal(got_y, ref_y.detach()) and torch.equal(got_g, xr.grad)


# ------------------------------------------------------------------------------------------ bad arguments

def _call(capi, fn, args):
    rc = getattr(capi.lib(), fn)(*args)
    return rc, capi.lib().jinc_last_error().decode()


def _expect_rejections(capi, fn, good, bad):
    import torch

    assert _call(capi, fn, good)[0] == 0, _call(capi, fn, good)
    torch.cuda.synchronize()
    for what, change in bad.items():
        args = list(good)
        for i, v in change.items():
            args[i] = v
        rc, msg = _call(capi, fn, args)
        assert rc == -1 and fn in msg, (what, rc, msg)


@pytest.mark.gpu
def test_planes_clamp_rejects_bad_arguments(gpu, ctx):
    import torch

    tab = gpu.Table(ctx, src_w=64, src_h=32, dst_w=128, dst_h=64, radius=gpu.radius_for_tap(3))
    src = torch.zeros((2, 32, 64), device="cuda")
    dst = torch.zeros((2, 64, 132), device="cuda")
    s, d = src.data_ptr(), dst.data_ptr()
    good = [ctx.handle, tab.handle, 4, 1.0, 2, s, 64 * 4, 32 * 64 * 4, d, 132 * 4, 64 * 132 * 4, None]
    _expect_rejections(gpu, "jinc_antiring_planes_device", good, {
        "null ctx": {0: None}, "null table": {1: None}, "null src": {5: None}, "null dst": {8: None},
        "no planes": {4: 0}, "negative planes": {4: -3}, "sample_bytes 3": {2: 3}, "sample_bytes 8": {2: 8},
        "strength nan": {3: float("nan")}, "strength below 0": {3: -0.1}, "strength above 1": {3: 1.5},
        "dst misaligned": {8: d + 4}, "dst pitch not 16": {9: 130 * 4}, "dst plane stride not 16": {10: 64 * 132 * 4 + 4},
    })
    tab.close()


@pytest.mark.gpu
def test_adjoint_call_rejects_bad_arguments(gpu, ctx):
    import torch

    tab = gpu.Table(ctx, src_w=64, src_h=32, dst_w=128, dst_h=64, radius=gpu.radius_for_tap(3))
    x = torch.zeros((2, 32, 64), device="cuda")
    y = torch.zeros((2, 64, 128), device="cuda")
    g = torch.zeros((2, 64, 128), device="cuda")
    gy = torch.zeros((2, 64, 128), device="cuda")
    gs = torch.zeros((2, 32, 64), device="cuda")
    X, Y, G, GY, GS = x.data_ptr(), y.data_ptr(), g.data_ptr(), gy.data_ptr(), gs.data_ptr()
    sp, ss, dp, ds = 64 * 4, 32 * 64 * 4, 128 * 4, 64 * 128 * 4
    good = [ctx.handle, tab.handle, 4, 1.0, 2, X, sp, ss, Y, dp, ds, G, dp, ds, GY, dp, ds, GS, sp, ss, None]
    _expect_rejections(gpu, "jinc_antiring_adjoint_planes_device", good, {
        "null ctx": {0: None}, "null table": {1: None}, "null src": {5: None}, "null y": {8: None},
        "null grad_dst": {11: None}, "null grad_y": {14: None}, "null grad_src": {17: None},
        "no planes": {4: 0}, "negative planes": {4: -1},
        "sample_bytes 1": {2: 1}, "sample_bytes 2": {2: 2}, "sample_bytes 3": {2: 3},
        "strength nan": {3: float("nan")}, "strength below 0": {3: -0.25}, "strength above 1": {3: 1.01},
        "src misaligned": {5: X + 2}, "src pitch short": {6: 63 * 4}, "src pitch not 4": {6: 64 * 4 + 2},
        "src plane stride short": {7: 31 * 64 * 4}, "y misaligned": {8: Y + 1}, "y pitch short": {9: 127 * 4},
        "y plane stride not 4": {10: ds + 2}, "grad_dst misaligned": {11: G + 2}, "grad_dst pitch not 4": {12: dp + 1},
        "grad_dst plane stride zero": {13: 0}, "grad_y misaligned": {14: GY + 2}, "grad_y pitch short": {15: dp - 4},
        "grad_y plane stride short": {16: ds - dp}, "grad_src misaligned": {17: GS + 2}, "grad_src pitch short": {18: sp - 4},
        "grad_src plane stride not 4": {19: ss + 1},
        "grad_src overlaps grad_dst": {17: G + ds}, "grad_src overlaps grad_y": {17: GY + 4},
        "grad_y overlaps grad_dst": {14: G + 64},
    })
    # half planes: pitches in half samples
    xh = torch.zeros((2, 32, 64), dtype=torch.float16, device="cuda")
    yh = torch.zeros((2, 64, 128), dtype=torch.float16, device="cuda")
    good_h = list(good)
    good_h[2], good_h[5], good_h[6], good_h[7] = gpu.SAMPLE_F16, xh.data_ptr(), 64 * 2, 32 * 64 * 2
    good_h[8], good_h[9], good_h[10] = yh.data_ptr(), 128 * 2, 64 * 128 * 2
    _expect_rejections(gpu, "jinc_antiring_adjoint_planes_device", good_h, {
        "half src pitch short": {6: 63 * 2}, "half y misaligned": {8: yh.data_ptr() + 1}, "half y pitch odd": {9: 128 * 2 + 1},
    })
    tab.close()
