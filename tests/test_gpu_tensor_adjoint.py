"""The PyTorch front-end (jinc_b200.tensor.jinc_resize), the batched plane call and the adjoint of the resampler.

The resize is a fixed linear map out = A * src whose weights are the table's (the oracle's per-pixel blocks).  The adjoint
sums, for each source sample, w * g over the outputs whose window covers it, in one canonical order (output rows
ascending, then columns ascending, fmaf from 0), so it is checked against A^T g in float64 with a rounding bound, and the
Jacobian of a float32 call is the oracle's weights bit for bit.  The CPU tests at the top need no GPU."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from common import FULL_CASES, SMALL_CASES

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def f32(v):
    return float(np.float32(v))


def geometries(case):
    """One entry per coefficient table of a case: (label, src (H, W), jinc_resize kwargs, oracle TableParams, tap, blur).
    Chroma tables are given as explicit crops, rounded to float32 as jinc_resize rounds them."""
    from oracle import cpu as oc

    name, fmt, w, h, tw, th, kw = case
    sw, sh = fmt.subsampling
    tap, blur = kw.get("tap", 3), kw.get("blur", 0.0)
    pp = oc.plane_params(w, h, tw, th, src_left=kw.get("src_left", 0.0), src_top=kw.get("src_top", 0.0),
                         src_width=kw.get("src_width"), src_height=kw.get("src_height"), quant_x=kw.get("quant_x", 256),
                         quant_y=kw.get("quant_y", 256), tap=tap, sub_w=sw, sub_h=sh, cplace=kw.get("cplace", "mpeg2"))
    out = []
    for k, p in enumerate(pp):
        p.crop_left, p.crop_top, p.crop_w, p.crop_h = f32(p.crop_left), f32(p.crop_top), f32(p.crop_w), f32(p.crop_h)
        args = dict(width=p.dst_w, height=p.dst_h, tap=tap, src_left=p.crop_left, src_top=p.crop_top, src_width=p.crop_w,
                    src_height=p.crop_h, quant_x=p.quant_x, quant_y=p.quant_y, blur=blur)
        out.append((f"{name}/{'luma' if k == 0 else 'chroma'}", (p.src_h, p.src_w), args, p, tap, blur))
    return out


def oracle_table(p, tap, blur):
    from oracle import cpu as oc

    return oc.Table(p, oc.make_lut(tap, blur))


def axes(ot):
    return ot.meta[0, :, 0].astype(np.int64), ot.meta[:, 0, 1].astype(np.int64)


# ------------------------------------------------------------------------------------------ CPU tests

@pytest.mark.parametrize("case", SMALL_CASES + FULL_CASES, ids=[c[0] for c in SMALL_CASES + FULL_CASES])
def test_window_origins_are_non_decreasing(native_built, case):
    """The covering outputs of a source column form one contiguous range only if start_x / start_y never decrease; the
    adjoint kernels find that range by binary search."""
    for label, _, _, p, tap, blur in geometries(case):
        ot = oracle_table(p, tap, blur)
        sx, sy = axes(ot)
        assert (ot.meta[:, :, 0] == sx[None, :]).all() and (ot.meta[:, :, 1] == sy[:, None]).all(), label
        assert (np.diff(sx) >= 0).all() and (np.diff(sy) >= 0).all(), label
        ot.close()


def test_rejects_cpu_tensors_dtypes_and_bits():
    """Checked on the host before the library is loaded: the dtype (TypeError), then bits, then the device (ValueError)."""
    import torch

    from jinc_b200.tensor import jinc_resize

    with pytest.raises(ValueError, match="no CPU path"):
        jinc_resize(torch.zeros(8, 8), 16, 16)
    with pytest.raises(ValueError, match="no CPU path"):
        jinc_resize(torch.zeros(2, 8, 8, dtype=torch.uint16), 16, 16, bits=10)
    for dt in (torch.float64, torch.bfloat16, torch.int32, torch.int16, torch.int8):
        with pytest.raises(TypeError):
            jinc_resize(torch.zeros(8, 8, dtype=dt), 16, 16)
    for dt, bits in ((torch.uint8, 10), (torch.uint16, 8), (torch.uint16, 17), (torch.float32, 16), (torch.float16, 8)):
        with pytest.raises(ValueError, match="bits"):
            jinc_resize(torch.zeros(8, 8, dtype=dt), 16, 16, bits=bits)
    with pytest.raises(TypeError):
        jinc_resize(np.zeros((8, 8), np.float32), 16, 16)


@pytest.mark.skipif(shutil.which("cuobjdump") is None and not os.path.exists("/usr/local/cuda/bin/cuobjdump"),
                    reason="cuobjdump not installed")
def test_adjoint_kernels_built_without_spills(native_built):
    from jinc_b200 import paths

    lib = paths.cuda_lib()
    if not os.path.exists(lib):
        pytest.skip("library not built")
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    out = subprocess.run([tool, "-res-usage", lib], capture_output=True, text=True, check=True).stdout
    lines = out.splitlines()
    found = {}
    for i, line in enumerate(lines):
        m = re.search(r"Function (\S*adjoint_(?:up2x|general)\S*):", line)
        if m:
            usage = lines[i + 1]
            assert "LOCAL:0" in usage and "STACK:0" in usage, (m.group(1), usage)
            found[m.group(1)] = usage
    assert "sm_100a" in out or "sm_100" in out
    for fs in (7, 9, 11, 13, 15, 17):
        assert any(f"adjoint_up2xILi{fs}E" in k for k in found), f"no exact-2x adjoint for fs {fs}"
    assert any("adjoint_general" in k for k in found)


# ------------------------------------------------------------------------------------------ GPU helpers

@pytest.fixture(scope="module")
def gpu(native_built):
    from jinc_b200 import capi

    assert capi.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    return capi


@pytest.fixture(scope="module")
def ctx(gpu):
    return gpu.Context(0)


def gpu_table(capi, ctx, p, tap, blur):
    return capi.Table(ctx, quant_x=p.quant_x, quant_y=p.quant_y, src_w=p.src_w, src_h=p.src_h, dst_w=p.dst_w, dst_h=p.dst_h,
                      radius=capi.radius_for_tap(tap), blur=f32(blur), crop_left=p.crop_left, crop_top=p.crop_top,
                      crop_w=p.crop_w, crop_h=p.crop_h)


def adjoint(tab, g):
    """jinc_resize_adjoint_planes_device on a float32 CUDA tensor (N, h, w) -> (N, H, W)."""
    import torch

    g = g.contiguous()
    n, h, w = g.shape
    out = torch.full((n, tab_src(tab)[0], tab_src(tab)[1]), float("nan"), device=g.device)
    tab.adjoint_planes_device(n, g.data_ptr(), w * 4, h * w * 4, out.data_ptr(), out.shape[2] * 4, out.shape[1] * out.shape[2] * 4,
                              torch_stream(g.device))
    return out


def torch_stream(device):
    from jinc_b200.tensor import _stream

    return _stream(device)


def tab_src(tab):
    return tab.src_shape


def sparse_chunks(ot, rows=None, max_entries=1 << 24):
    """(output rows y0:y1, CSR matrix of those outputs' weights over the whole source, in float64) in chunks; `rows`:
    only outputs whose window covers one of these source rows."""
    import scipy.sparse as sp

    fs, cs = ot.filter_size, ot.coeff_stride
    sx, sy = axes(ot)
    H, W = ot.params.src_h, ot.params.src_w
    h, w = ot.dst_h, ot.dst_w
    idx = (np.arange(fs)[:, None] * cs + np.arange(fs)[None, :]).ravel()
    ly, lx = np.divmod(np.arange(fs * fs), fs)
    if rows is None:
        ys = np.arange(h)
    else:
        rows = np.asarray(rows)
        ys = np.nonzero(((sy[:, None] <= rows[None, :]) & (rows[None, :] < sy[:, None] + fs)).any(1))[0]
    step = max(1, max_entries // max(1, w * fs * fs))
    for c0 in range(0, len(ys), step):
        yy = ys[c0:c0 + step]
        off = ot.meta[yy, :, 2].astype(np.int64)  # (ny, w)
        wts = ot.factor[off[..., None] + idx[None, None, :]].astype(np.float64)  # (ny, w, fs*fs)
        col = (sy[yy][:, None, None] + ly[None, None, :]) * W + sx[None, :, None] + lx[None, None, :]
        row = (np.arange(len(yy))[:, None, None] * w + np.arange(w)[None, :, None]) + np.zeros_like(col)
        m = sp.csr_matrix((wts.ravel(), (row.ravel(), col.ravel())), shape=(len(yy) * w, H * W))
        ones = sp.csr_matrix((np.ones(wts.size), (row.ravel(), col.ravel())), shape=(len(yy) * w, H * W))
        yield yy, m, ones


def adjoint_reference(ot, g, rows=None):
    """float64 A^T g, sum |w g| and covering tap counts per source sample (rows: only the outputs covering them)."""
    H, W = ot.params.src_h, ot.params.src_w
    ref = np.zeros(H * W)
    mag = np.zeros(H * W)
    cnt = np.zeros(H * W)
    g = g.astype(np.float64)
    for yy, m, ones in sparse_chunks(ot, rows):
        gv = g[yy].ravel()
        ref += m.T @ gv
        mag += abs(m).T @ np.abs(gv)
        cnt += ones.T @ np.ones_like(gv)
    return ref.reshape(H, W), mag.reshape(H, W), cnt.reshape(H, W)


def assert_within_gamma(got, ref, mag, cnt, what, rows=None):
    u = 2.0 ** -24
    gamma = cnt * u / (1 - cnt * u)
    got = got.astype(np.float64)
    sel = slice(None) if rows is None else np.asarray(rows)
    err = np.abs(got[sel] - ref[sel])
    bad = err > gamma[sel] * mag[sel]
    assert not bad.any(), f"{what}: {int(bad.sum())} samples beyond gamma_n * sum|w g| (max err {err.max():.3e})"
    zero = cnt[sel] == 0
    assert (got[sel][zero] == 0).all(), f"{what}: uncovered samples must be written as 0"


# ------------------------------------------------------------------------------------------ forward

DTYPES = ["uint8", "uint16", "float16", "float32"]


def random_planes(shape, dtype, bits, seed):
    import torch

    rng = np.random.default_rng(seed)
    if dtype in ("float16", "float32"):
        a = rng.random(shape, dtype=np.float32).astype(dtype)
    else:
        a = rng.integers(0, 1 << bits, shape).astype(dtype)
    return torch.from_numpy(a).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("case", SMALL_CASES, ids=[c[0] for c in SMALL_CASES])
def test_batched_forward_equals_per_plane_calls(gpu, ctx, case):
    """jinc_resize on a (3, 2, H, W) batch (one jinc_resize_planes_device call) equals jinc_resize_plane_device on each
    plane, byte for byte, for every table of every small case and each dtype."""
    import torch

    from jinc_b200.tensor import jinc_resize

    fmt = case[1]
    for label, (H, W), args, p, tap, blur in geometries(case):
        tab = gpu_table(gpu, ctx, p, tap, blur)
        for dt in DTYPES:
            bits = {"uint8": 8, "uint16": fmt.bits if 9 <= fmt.bits <= 16 else 16}.get(dt)
            x = random_planes((3, 2, H, W), dt, bits or 0, 11)
            y = jinc_resize(x, bits=bits, **args)
            assert y.shape == (3, 2, p.dst_h, p.dst_w) and y.dtype == x.dtype
            sb = {"uint8": 1, "uint16": 2, "float16": gpu.SAMPLE_F16, "float32": 4}[dt]
            isz = x.element_size()
            pitch = (p.dst_w * isz + 15) // 16 * 16
            peak = float((1 << bits) - 1) if bits else 0.0
            xs = x.view(-1, H, W)
            ref = torch.empty((6, p.dst_h, pitch // isz), dtype=x.dtype, device="cuda")
            for i in range(6):
                tab.resize_device(sb, peak, xs[i].data_ptr(), W * isz, ref[i].data_ptr(), pitch, torch_stream(x.device))
            torch.cuda.synchronize()
            got = y.reshape(6, p.dst_h, p.dst_w).cpu().numpy().view(np.uint8)
            want = ref[..., :p.dst_w].cpu().numpy().view(np.uint8)
            assert np.array_equal(got, want), f"{label}/{dt}: batched call differs from per-plane calls"
        tab.close()


VS_CASES = ["c1_yv12_2x_tap3", "irregular_up_crop_mpeg1", "topleft_negative_crop", "half_tap3_yv12", "up1p5_tap3_f32_y"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", VS_CASES)
def test_equals_vapoursynth_filter_on_gray(gpu, name):
    """A call on one plane equals core.jinc.JincResize on a GRAY clip with the same script arguments, byte for byte."""
    import torch

    from jinc_b200 import paths
    from jinc_b200.tensor import jinc_resize
    from minihost import vs_host

    case = {c[0]: c for c in SMALL_CASES}[name]
    _, fmt, w, h, tw, th, kw = case
    script = {k: v for k, v in kw.items() if k != "cplace"}
    core = vs_host.Core()
    vsp = core.load_plugin(paths.vs_plugin())
    for dt, bits in (("uint8", 8), ("uint16", 10), ("float32", 32), ("float16", 16)):
        x = random_planes((h, w), dt, min(bits, 16), 5)
        plane = x.cpu().numpy()
        src = core.source(vs_host.CF_GRAY, np.dtype(dt), bits, 0, 0, w, h, [[plane]])
        clip = vsp.invoke("JincResize", src, width=tw, height=th, **script)
        (want,), _ = clip.get_frame(0)
        clip.release()
        src.release()
        got = jinc_resize(x, tw, th, bits=bits if dt.startswith("uint") else None, **script).cpu().numpy()
        assert np.array_equal(got.view(np.uint8), np.ascontiguousarray(want).view(np.uint8)), f"{name}/{dt}"


# ------------------------------------------------------------------------------------------ adjoint

@pytest.mark.gpu
@pytest.mark.parametrize("case", SMALL_CASES, ids=[c[0] for c in SMALL_CASES])
def test_adjoint_against_float64(gpu, ctx, case):
    """Every source sample of A^T g is within gamma_n * sum |w g| of the float64 value (n: the sample's covering taps);
    samples no output covers are 0."""
    import torch

    for label, (H, W), args, p, tap, blur in geometries(case):
        tab = gpu_table(gpu, ctx, p, tap, blur)
        tab.src_shape = (H, W)
        g = np.random.default_rng(3).standard_normal((p.dst_h, p.dst_w)).astype(np.float32)
        got = adjoint(tab, torch.from_numpy(g).cuda()[None]).cpu().numpy()[0]
        ot = oracle_table(p, tap, blur)
        ref, mag, cnt = adjoint_reference(ot, g)
        assert_within_gamma(got, ref, mag, cnt, label)
        ot.close()
        tab.close()


JAC_CASES = [
    ("up2x_tap3", dict(W=80, H=26, width=160, height=52, tap=3)),
    ("down_half_tap3", dict(W=48, H=30, width=24, height=15, tap=3)),
    ("irregular_crop", dict(W=37, H=23, width=51, height=19, tap=4, src_left=1.3, src_top=0.6, src_width=33.5, src_height=21.25)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,geo", JAC_CASES, ids=[c[0] for c in JAC_CASES])
def test_jacobian_is_the_oracle_weights(gpu, name, geo):
    """The Jacobian of a float32 call equals the oracle's weights bit for bit: each entry is one fmaf(w, 1, 0)."""
    import torch

    from jinc_b200.tensor import jinc_resize
    from oracle import cpu as oc

    geo = dict(geo)
    W, H = geo.pop("W"), geo.pop("H")
    w, h, tap = geo["width"], geo["height"], geo["tap"]
    pp = oc.plane_params(W, H, w, h, src_left=geo.get("src_left", 0.0), src_top=geo.get("src_top", 0.0),
                         src_width=geo.get("src_width"), src_height=geo.get("src_height"), tap=tap)
    ot = oracle_table(pp[0], tap, 0.0)
    fs = ot.filter_size
    sx, sy = axes(ot)
    want = np.zeros((h, w, H, W), np.float32)
    for y in range(h):
        for x in range(w):
            want[y, x, sy[y]:sy[y] + fs, sx[x]:sx[x] + fs] = ot.block(y, x)
    ot.close()
    # every row of the Jacobian at once: a batch of h*w copies of x, backward with one-hot output gradients
    x = torch.rand((h * w, H, W), device="cuda", requires_grad=True)
    y = jinc_resize(x, **geo)
    eye = torch.eye(h * w, device="cuda").view(h * w, h, w)
    (jac,) = torch.autograd.grad(y, x, grad_outputs=eye)
    assert np.array_equal(jac.view(h, w, H, W).cpu().numpy(), want), name
    if h * w <= 1024:
        x1 = torch.rand((H, W), device="cuda")
        jf = torch.autograd.functional.jacobian(lambda t: jinc_resize(t, **geo), x1)
        assert np.array_equal(jf.cpu().numpy(), want), name


FULL = {c[0]: c for c in FULL_CASES}


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["config1", "config2", "config3", "config4", "config5"])
def test_full_size_adjoint(gpu, ctx, name):
    """Full-size tables: the dot-product identity <A x, g> = <x, A^T g> in float64, and sampled source rows (top, middle,
    bottom, and each side of the exact-2x rectangle's edges) against the float64 reference built for those rows."""
    import torch

    from jinc_b200.tensor import jinc_resize

    for label, (H, W), args, p, tap, blur in geometries(FULL[name]):
        rng = np.random.default_rng(9)
        x = torch.from_numpy(rng.random((H, W), dtype=np.float32)).cuda()
        g = rng.standard_normal((p.dst_h, p.dst_w)).astype(np.float32)
        tab = gpu_table(gpu, ctx, p, tap, blur)
        tab.src_shape = (H, W)
        ax = jinc_resize(x, **args).double().cpu().numpy()
        atg = adjoint(tab, torch.from_numpy(g).cuda()[None]).cpu().numpy()[0]
        lhs = float((ax * g).sum())
        rhs = float((x.double().cpu().numpy() * atg).sum())
        bound = 1e-5 * 2.0 * float(np.abs(g).sum()) * float(x.abs().max())  # sum|A| per output is below 2
        assert abs(lhs - rhs) <= bound, f"{label}: <Ax,g> = {lhs} vs <x,A^T g> = {rhs}"
        info = tab.info
        ot = oracle_table(p, tap, blur)
        fs = ot.filter_size
        sx, sy = axes(ot)
        rows = {0, 1, H // 2, H - 2, H - 1}
        if info.fast_path == 1:  # rows on each side of where the 2x kernel's source rectangle starts and ends
            y0 = int(sy[info.interior_y0]) + fs - 1
            y1 = int(sy[info.interior_y1 - 1])
            rows |= {r for r in (y0 - 1, y0, y0 + 1, y0 + 2, y1 - 1, y1, y1 + 1) if 0 <= r < H}
        rows = sorted(rows)
        ref, mag, cnt = adjoint_reference(ot, g, rows)
        assert_within_gamma(atg, ref, mag, cnt, label, rows)
        ot.close()
        tab.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["c2_420p8_2x_tap3_mpeg2", "c4_rgbps_2x_tap8", "half_tap3_yv12", "irregular_up_crop_mpeg1"])
def test_inf_reaches_exactly_its_window(gpu, ctx, case):
    import torch

    for label, (H, W), args, p, tap, blur in geometries({c[0]: c for c in SMALL_CASES}[case]):
        tab = gpu_table(gpu, ctx, p, tap, blur)
        tab.src_shape = (H, W)
        ot = oracle_table(p, tap, blur)
        fs = ot.filter_size
        sx, sy = axes(ot)
        for (yy, xx) in ((p.dst_h // 2, p.dst_w // 2), (0, 0), (p.dst_h - 1, 3)):
            g = torch.rand((1, p.dst_h, p.dst_w), device="cuda")
            g[0, yy, xx] = float("inf")
            got = adjoint(tab, g).cpu().numpy()[0]
            win = np.zeros((H, W), bool)
            win[sy[yy]:sy[yy] + fs, sx[xx]:sx[xx] + fs] = True
            assert np.array_equal(~np.isfinite(got), win), f"{label}: Inf at ({yy}, {xx})"
        ot.close()
        tab.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["c2_420p8_2x_tap3_mpeg2", "c4_rgbps_2x_tap8", "c5_420p10_quarter_tap6_blur", "up1p5_tap3_420p8"])
def test_adjoint_bits_do_not_depend_on_batch_position(gpu, ctx, case):
    import torch

    for label, (H, W), args, p, tap, blur in geometries({c[0]: c for c in SMALL_CASES}[case]):
        tab = gpu_table(gpu, ctx, p, tap, blur)
        tab.src_shape = (H, W)
        g = torch.randn((64, p.dst_h, p.dst_w), device="cuda")
        one = adjoint(tab, g[37:38].clone())
        batch = adjoint(tab, g)
        again = adjoint(tab, g)
        torch.cuda.synchronize()
        assert torch.equal(one[0].view(torch.int32), batch[37].view(torch.int32)), label
        assert torch.equal(batch.view(torch.int32), again.view(torch.int32)), label
        tab.close()


# ------------------------------------------------------------------------------------------ autograd

@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float32", "float16"])
def test_autograd_backward_is_the_adjoint(gpu, ctx, dtype):
    import torch

    from jinc_b200.tensor import jinc_resize

    case = {c[0]: c for c in SMALL_CASES}["c1_yv12_2x_tap3"]
    (label, (H, W), args, p, tap, blur) = geometries(case)[0]
    tab = gpu_table(gpu, ctx, p, tap, blur)
    tab.src_shape = (H, W)
    dt = getattr(torch, dtype)
    x = torch.rand((2, 3, H, W), device="cuda").to(dt).requires_grad_()
    y = jinc_resize(x, **args)
    g = torch.randn(y.shape, device="cuda").to(dt)
    (y * g).sum().backward()
    want = adjoint(tab, g.float().reshape(6, p.dst_h, p.dst_w)).to(dt).view(x.shape)
    assert x.grad.dtype == dt and torch.equal(x.grad, want)
    x.grad = None
    jinc_resize(x, **args).sum().backward()  # zero-stride expanded gradient
    want = adjoint(tab, torch.ones((6, p.dst_h, p.dst_w), device="cuda")).to(dt).view(x.shape)
    assert torch.equal(x.grad, want)
    tab.close()


@pytest.mark.gpu
def test_side_stream_needs_no_extra_synchronisation(gpu):
    import torch

    from jinc_b200.tensor import jinc_resize

    x0 = torch.rand((4, 270, 480), device="cuda")
    ref_y = jinc_resize(x0, 960, 540)
    xr = x0.clone().requires_grad_()
    jinc_resize(xr, 960, 540).square().sum().backward()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        x = torch.rand((4, 270, 480), device="cuda")
        x.copy_(x0)  # ordered on s only
        x.requires_grad_()
        y = jinc_resize(x, 960, 540)
        y.square().sum().backward()
        got_y, got_g = y.detach().clone(), x.grad.clone()
    torch.cuda.current_stream().wait_stream(s)
    assert torch.equal(got_y, ref_y) and torch.equal(got_g, xr.grad)


@pytest.mark.gpu
def test_second_device(gpu):
    import torch

    from jinc_b200.tensor import jinc_resize

    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    x = torch.rand((2, 90, 160))
    a = jinc_resize(x.cuda(0).requires_grad_(), 320, 180)
    b = jinc_resize(x.cuda(1).requires_grad_(), 320, 180)
    assert b.device == torch.device("cuda:1") and torch.equal(a.cpu(), b.cpu())


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float32", "float16"])
def test_backward_of_a_gradient_expanded_over_a_leading_dimension(gpu, ctx, dtype):
    """y.sum(0) hands backward a gradient whose plane stride is 0: it is made contiguous, and x.grad is the adjoint of it."""
    import torch

    from jinc_b200.tensor import jinc_resize

    (label, (H, W), args, p, tap, blur) = geometries({c[0]: c for c in SMALL_CASES}["c1_yv12_2x_tap3"])[0]
    tab = gpu_table(gpu, ctx, p, tap, blur)
    tab.src_shape = (H, W)
    dt = getattr(torch, dtype)
    x = torch.rand((4, H, W), device="cuda").to(dt).requires_grad_()
    g = torch.randn((p.dst_h, p.dst_w), device="cuda").to(dt)
    (jinc_resize(x, **args).sum(0) * g).sum().backward()
    want = adjoint(tab, g.float().expand(4, p.dst_h, p.dst_w)).to(dt)
    assert torch.equal(x.grad, want), label
    tab.close()


@pytest.mark.gpu
@pytest.mark.parametrize("width,height", [(320, 180), (318, 181)], ids=["unpadded", "padded"])
def test_output_can_be_modified_in_place_before_backward(gpu, ctx, width, height):
    """The result is a tensor of its own, not a view: in-place ops on it work under autograd, with or without row padding."""
    import torch

    from jinc_b200.tensor import jinc_resize

    x = torch.rand((2, 3, 90, 160), device="cuda", requires_grad=True)
    g = torch.randn((2, 3, height, width), device="cuda")
    y = jinc_resize(x, width, height)
    assert y._base is None and y.shape == (2, 3, height, width)
    assert y.stride(-2) == (width + 3) // 4 * 4 and y.stride(-3) == height * y.stride(-2)
    y.mul_(2.0)
    (y * g).sum().backward()
    ref = torch.rand((2, 3, 90, 160), device="cuda").copy_(x.detach()).requires_grad_()
    (jinc_resize(ref, width, height) * (2.0 * g)).sum().backward()
    assert torch.equal(x.grad, ref.grad)
    z = jinc_resize(x, width, height)
    z.clamp_(0.0, 1.0)
    z.sum().backward()  # clamp_ is differentiable; the point is that autograd accepts the in-place op


def _abi_call_error(capi, fn, *args):
    rc = getattr(capi.lib(), fn)(*args)
    return rc, capi.lib().jinc_last_error().decode()


@pytest.mark.gpu
def test_planes_call_rejects_bad_arguments(gpu, ctx):
    """jinc_resize_planes_device: JINC_E_INVALID, with a message naming the function, for every bad argument."""
    import torch

    capi = gpu
    tab = capi.Table(ctx, src_w=64, src_h=32, dst_w=128, dst_h=64, radius=capi.radius_for_tap(3))
    src = torch.zeros((2, 32, 64), device="cuda")
    dst = torch.zeros((2, 64, 128 + 4), device="cuda")
    s, d = src.data_ptr(), dst.data_ptr()
    good = [ctx.handle, tab.handle, 4, 0.0, 2, s, 64 * 4, 32 * 64 * 4, d, 132 * 4, 64 * 132 * 4, None]
    assert _abi_call_error(capi, "jinc_resize_planes_device", *good)[0] == 0
    torch.cuda.synchronize()
    bad = {
        "null ctx": {0: None}, "null table": {1: None}, "null src": {5: None}, "null dst": {8: None},
        "no planes": {4: 0}, "negative planes": {4: -3}, "sample_bytes 3": {2: 3}, "sample_bytes 8": {2: 8},
        "dst misaligned": {8: d + 4}, "dst pitch not 16": {9: 130 * 4}, "dst plane stride not 16": {10: 64 * 132 * 4 + 4},
    }
    for what, change in bad.items():
        args = list(good)
        for i, v in change.items():
            args[i] = v
        rc, msg = _abi_call_error(capi, "jinc_resize_planes_device", *args)
        assert rc == -1 and "jinc_resize_planes_device" in msg, (what, rc, msg)
    tab.close()


@pytest.mark.gpu
def test_adjoint_call_rejects_bad_arguments(gpu, ctx):
    """jinc_resize_adjoint_planes_device: JINC_E_INVALID, with a message naming the function, for every bad argument."""
    import torch

    capi = gpu
    tab = capi.Table(ctx, src_w=64, src_h=32, dst_w=128, dst_h=64, radius=capi.radius_for_tap(3))
    g = torch.zeros((2, 64, 128), device="cuda")
    o = torch.zeros((2, 32, 64), device="cuda")
    gp, op = g.data_ptr(), o.data_ptr()
    good = [ctx.handle, tab.handle, 2, gp, 128 * 4, 64 * 128 * 4, op, 64 * 4, 32 * 64 * 4, None]
    assert _abi_call_error(capi, "jinc_resize_adjoint_planes_device", *good)[0] == 0
    torch.cuda.synchronize()
    bad = {
        "null ctx": {0: None}, "null table": {1: None}, "null grad_dst": {3: None}, "null grad_src": {6: None},
        "no planes": {2: 0}, "grad_dst misaligned": {3: gp + 2}, "grad_src misaligned": {6: op + 1},
        "grad_dst pitch short": {4: 127 * 4}, "grad_dst pitch not 4": {4: 128 * 4 + 2},
        "grad_src pitch short": {7: 63 * 4}, "grad_src pitch not 4": {7: 64 * 4 + 1},
        "grad_dst plane stride short": {5: 63 * 128 * 4}, "grad_dst plane stride zero": {5: 0},
        "grad_src plane stride short": {8: 31 * 64 * 4}, "grad_src plane stride not 4": {8: 32 * 64 * 4 + 2},
        "overlap": {6: gp + 64 * 128 * 4},
    }
    for what, change in bad.items():
        args = list(good)
        for i, v in change.items():
            args[i] = v
        rc, msg = _abi_call_error(capi, "jinc_resize_adjoint_planes_device", *args)
        assert rc == -1 and "jinc_resize_adjoint_planes_device" in msg, (what, rc, msg)
    tab.close()
