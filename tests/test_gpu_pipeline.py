"""GPU tests of the entry points around the kernels: the device-resident calls bench.py times
(jinc_filter_process_device / _batch), the row-band split (jinc_filter_process_bands / _split), the in-process multi-GPU
paths, the submit/wait tickets and the host-buffer registry (jinc_hostmem) of the frame pipeline.

Everything is called through the C ABI (include/jinc_b200.h) and compared with the CPU oracle, or -- for the band
split, which must not change a single bit -- with the whole-frame result of the same filter.
"""
import ctypes as C

import numpy as np
import pytest

from common import SMALL_CASES, assert_plane_close, make_filter, make_planes, oracle_frame

pytestmark = pytest.mark.gpu

CASES = {c[0]: c for c in SMALL_CASES}


@pytest.fixture(scope="module")
def capi(native_built):
    from jinc_b200 import capi as c

    assert c.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    return c


def device_frames(capi, flt, fmt, frames, pitch_align=256):
    """Uploads `frames` (lists of numpy planes) into pitched torch tensors; returns (ctypes Frame array, keep-alive, dst tensors)."""
    import torch

    sb = np.dtype(fmt.dtype).itemsize
    tdt = {1: torch.uint8, 2: torch.uint16, 4: torch.float32}[sb]
    shapes = flt.plane_shapes()
    arr = (capi.Frame * len(frames))()
    keep, dsts = [], []
    for fi, planes in enumerate(frames):
        dd = []
        for i, ((sshape, dshape), p) in enumerate(zip(shapes, planes)):
            sp = ((sshape[1] * sb + pitch_align - 1) // pitch_align * pitch_align) // sb
            dp = ((dshape[1] * sb + pitch_align - 1) // pitch_align * pitch_align) // sb
            s = torch.zeros((sshape[0], sp), dtype=tdt, device="cuda")
            s[:, : sshape[1]].copy_(torch.from_numpy(p))
            d = torch.full((dshape[0], dp), 7, dtype=tdt, device="cuda")
            arr[fi].src[i], arr[fi].src_pitch[i] = s.data_ptr(), sp * sb
            arr[fi].dst[i], arr[fi].dst_pitch[i] = d.data_ptr(), dp * sb
            keep.append(s)
            dd.append(d)
        dsts.append(dd)
    torch.cuda.synchronize()
    return arr, keep, dsts


DEVICE_CASES = ["c2_420p8_2x_tap3_mpeg2", "c3_444p16_2x_tap4_crop", "c4_rgbps_2x_tap8", "c5_420p10_quarter_tap6_blur",
                "down2to3_tap3_420p8", "up4to3_tap3_420p8", "up1p5_tap3_420p8", "rgbap10_irregular_up", "irregular_down_quant"]


@pytest.mark.parametrize("name", DEVICE_CASES)
def test_device_batch_matches_oracle(capi, name):
    """jinc_filter_process_device_batch -- the call bench.py's kernel-only figure times: one launch per table covers all
    frames (grid.y = frame).  Every frame of the batch is downloaded and compared with the oracle, so a launch that wrote
    the right samples into the wrong frame cannot pass (the frames differ)."""
    import torch

    _, fmt, w, h, tw, th, kw = CASES[name]
    flt = make_filter(fmt, w, h, tw, th, **kw)
    F = 5
    frames = [make_planes(fmt, w, h, "noise", seed=100 + f) for f in range(F)]
    arr, keep, dsts = device_frames(capi, flt, fmt, frames)
    stream = torch.cuda.Stream()
    n0 = flt.kernel_launches
    flt.process_device_batch(arr, 0, 3, 3, stream.cuda_stream)
    stream.synchronize()
    assert flt.kernel_launches - n0 == flt.num_tables  # one launch per coefficient table for the whole batch
    shapes = flt.plane_shapes()
    for f in range(F):
        ref, _ = oracle_frame(fmt, w, h, tw, th, frames[f], **kw)
        for i, r in enumerate(ref):
            got = dsts[f][i][:, : shapes[i][1][1]].cpu().numpy()
            assert_plane_close(got, r, fmt.bits == 32, f"{name}/batch/frame{f}/plane{i}")
    flt.close()


@pytest.mark.parametrize("name", DEVICE_CASES[:5])
def test_device_single_frame_matches_oracle(capi, name):
    """jinc_filter_process_device, with the table mask and part selectors: tables run separately give the same frame, and
    interior + border launched separately tile the plane exactly (no sample written twice with different values, none
    left out)."""
    import torch

    _, fmt, w, h, tw, th, kw = CASES[name]
    flt = make_filter(fmt, w, h, tw, th, **kw)
    planes = make_planes(fmt, w, h, "noise", seed=5)
    ref, _ = oracle_frame(fmt, w, h, tw, th, planes, **kw)
    shapes = flt.plane_shapes()
    for mode in ("all", "per_table", "parts"):
        arr, keep, dsts = device_frames(capi, flt, fmt, [planes], pitch_align=64)
        if mode == "all":
            flt.process_device(arr[0], 0, 3, 3)
        elif mode == "per_table":
            for k in range(flt.num_tables):
                flt.process_device(arr[0], 0, 1 << k, 3)
        else:
            flt.process_device(arr[0], 0, 3, 1)  # interior tiles only
            flt.process_device(arr[0], 0, 3, 2)  # border strips only
        torch.cuda.synchronize()
        for i, r in enumerate(ref):
            got = dsts[0][i][:, : shapes[i][1][1]].cpu().numpy()
            assert_plane_close(got, r, fmt.bits == 32, f"{name}/device/{mode}/plane{i}")
    flt.close()


def test_device_batch_on_alternating_streams(capi):
    """More batched calls than the ring of plane-pointer buffers has entries, alternating between two streams: an entry is
    only reused after the launch that read it (event), so every call's frames come out right."""
    import torch

    _, fmt, w, h, tw, th, kw = CASES["c1_yv12_2x_tap3"]
    flt = make_filter(fmt, w, h, tw, th, **kw)
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    calls = []
    for c in range(12):
        frames = [make_planes(fmt, w, h, "noise", seed=1000 + 10 * c + f) for f in range(2)]
        arr, keep, dsts = device_frames(capi, flt, fmt, frames)
        flt.process_device_batch(arr, 0, 3, 3, streams[c & 1].cuda_stream)
        calls.append((frames, arr, keep, dsts))
    torch.cuda.synchronize()
    shapes = flt.plane_shapes()
    for frames, _, _, dsts in calls:
        for f, planes in enumerate(frames):
            ref, _ = oracle_frame(fmt, w, h, tw, th, planes, **kw)
            for i, r in enumerate(ref):
                assert_plane_close(dsts[f][i][:, : shapes[i][1][1]].cpu().numpy(), r, False, "streams")
    flt.close()


BAND_CASES = ["c2_420p8_2x_tap3_mpeg2", "c3_444p16_2x_tap4_crop", "c4_rgbps_2x_tap8", "c5_420p10_quarter_tap6_blur",
              "down2to3_tap3_420p8", "up4to3_tap3_420p8", "up4x_tap3_420p8", "up1p5_tap3_420p8", "irregular_up_crop_mpeg1",
              "yuva420_14bit_2x", "third_tap3_y8", "steep_down_444p16_tap5", "down3to4_tap3_444p10", "up9to4_tap4_y16",
              "down2to3_tap4_y16"]


@pytest.mark.parametrize("n_bands", [2, 3, 7])
@pytest.mark.parametrize("name", BAND_CASES)
def test_row_bands_equal_whole_frame(capi, name, n_bands):
    """jinc_filter_process_bands: the frame cut into n row bands (each through its own slot: partial source upload from
    the per-axis origins, kernels clipped to the band, partial download) is BYTE-identical to the whole frame, for every
    kernel family, with subsampled chroma, and for pageable as well as page-locked caller buffers."""
    import torch

    _, fmt, w, h, tw, th, kw = CASES[name]
    planes = make_planes(fmt, w, h, "noise", seed=3)
    flt = make_filter(fmt, w, h, tw, th, **kw)
    whole = flt.process(planes)
    bands = capi.row_bands(th, n_bands)
    assert bands[0][0] == 0 and max(b for _, b in bands) == th
    got = flt.process([p.copy() for p in planes], bands=n_bands)
    for i, (a, b) in enumerate(zip(whole, got)):
        assert np.array_equal(a, b), f"{name}: plane {i} differs between {n_bands} bands and the whole frame"
    pin_src = [torch.from_numpy(p.copy()).pin_memory() for p in planes]
    pin_dst = [torch.from_numpy(np.zeros_like(a)).pin_memory() for a in whole]
    flt.process([t.numpy() for t in pin_src], [t.numpy() for t in pin_dst], bands=n_bands)
    for i, (a, b) in enumerate(zip(whole, pin_dst)):
        assert np.array_equal(a, b.numpy()), f"{name}: plane {i} differs (pinned buffers, {n_bands} bands)"
    ref, _ = oracle_frame(fmt, w, h, tw, th, planes, **kw)
    for i, (g, r) in enumerate(zip(got, ref)):
        assert_plane_close(g, r, fmt.bits == 32, f"{name}/bands/plane{i}")
    flt.close()


def test_split_over_repeated_device_ids(capi):
    """jinc_filter_process_split cuts one frame into one band per device of the filter; a filter built over the same GPU
    three times exercises exactly that path on a one-GPU box."""
    _, fmt, w, h, tw, th, kw = CASES["c2_420p8_2x_tap3_mpeg2"]
    planes = make_planes(fmt, w, h, "noise", seed=8)
    one = make_filter(fmt, w, h, tw, th, **kw)
    whole = one.process(planes)
    one.close()
    flt = make_filter(fmt, w, h, tw, th, devices=(0, 0, 0), **kw)
    assert flt.num_devices == 3
    got = flt.process(planes, split=True)
    for a, b in zip(whole, got):
        assert np.array_equal(a, b)
    flt.close()


def test_bands_from_concurrent_callers(capi):
    """Several threads cut different frames into bands on one filter at once: slots are shared without deadlock."""
    import threading

    _, fmt, w, h, tw, th, kw = CASES["c1_yv12_2x_tap3"]
    flt = make_filter(fmt, w, h, tw, th, **kw)
    frames = [make_planes(fmt, w, h, "noise", seed=40 + s) for s in range(8)]
    want = [flt.process(f) for f in frames]
    outs = [None] * len(frames)

    def work(i):
        outs[i] = flt.process(frames[i], bands=2 + i % 4)

    ts = [threading.Thread(target=work, args=(i,)) for i in range(len(frames))]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=120)
        assert not t.is_alive(), "band split deadlocked"
    for a, b in zip(want, outs):
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
    flt.close()


def test_tickets_and_busy(capi):
    """try_submit reports JINC_E_BUSY once every slot is taken instead of blocking; a ticket can be waited on once."""
    _, fmt, w, h, tw, th, kw = CASES["c1_yv12_2x_tap3"]
    flt = make_filter(fmt, w, h, tw, th, **kw)
    n = flt.num_slots
    assert 3 <= n <= 8
    frames = [make_planes(fmt, w, h, "noise", seed=s) for s in range(n)]
    outs = [flt.alloc_dst() for _ in frames]
    tickets = [flt.try_submit(f, o) for f, o in zip(frames, outs)]
    assert all(t is not None for t in tickets) and len(set(tickets)) == n
    assert flt.try_submit(frames[0], flt.alloc_dst()) is None  # full: BUSY, not a deadlock
    for t in tickets:
        flt.wait(t)
    with pytest.raises(capi.JincError, match="already waited"):
        flt.wait(tickets[0])
    for f, o in zip(frames, outs):
        ref, _ = oracle_frame(fmt, w, h, tw, th, f, **kw)
        for g, r in zip(o, ref):
            assert_plane_close(g, r, False, "tickets")
    assert flt.try_submit(frames[0], outs[0]) is not None  # slots are free again
    flt.close()


def test_bad_bits_are_rejected(capi):
    from minihost import avs_host as ah

    for sb, bits in ((1, 0), (1, 10), (2, 8), (2, 17), (2, 31)):
        with pytest.raises(capi.JincError, match="bits per component"):
            capi.Filter(src_w=64, src_h=64, target_w=128, target_h=128, n_planes=1, sample_bytes=sb, bits=bits, devices=[0])
    with pytest.raises(capi.JincError, match="devices"):
        capi.Filter(src_w=64, src_h=64, target_w=128, target_h=128, n_planes=1, sample_bytes=1, bits=8, devices=[0] * 17)
    n = capi.live_filters()  # failed constructions leave no filter behind
    with pytest.raises(capi.JincError):
        make_filter(ah.Format("y", 8), 8, 8, 4, 4, tap=8)
    assert capi.live_filters() == n


# ------------------------------------------------------------------------------------------ host-buffer registry

def _frame_buffer(shapes_bytes):
    """One contiguous pageable allocation holding all planes, packed the way AviSynth+ packs a frame buffer (64-byte
    pitches and plane offsets); returns (owner array, [plane views as uint8 2-D])."""
    offs, total = [], 0
    for rows, row_bytes in shapes_bytes:
        pitch = (row_bytes + 63) // 64 * 64
        offs.append((total, pitch))
        total += pitch * rows
    raw = np.zeros(total + 64 + 256, np.uint8)
    base = (-raw.ctypes.data) % 64
    views = []
    for (rows, row_bytes), (off, pitch) in zip(shapes_bytes, offs):
        v = raw[base + off: base + off + pitch * rows].reshape(rows, pitch)[:, :row_bytes]
        views.append(v)
    return raw, views


def test_recycled_pageable_buffers_get_registered(capi):
    """A pageable frame buffer that comes back is page-locked by the pipeline (on a helper thread, while that frame is
    still staged) and from then on moved without the staging copy (packed AviSynth-style buffers: one extent per frame
    and direction, the sub-page head and tail through the mirror); results do not change.  Without
    JINC_FILTER_HOST_REGISTER every frame stays staged."""
    import time

    _, fmt, w, h, tw, th, kw = CASES["c2_420p8_2x_tap3_mpeg2"]
    planes = make_planes(fmt, w, h, "noise", seed=21)
    ref, _ = oracle_frame(fmt, w, h, tw, th, planes, **kw)
    for flags, expect_direct in ((capi.FLAG_DST_PADDING_WRITABLE | capi.FLAG_HOST_REGISTER, True), (0, False)):
        flt = make_filter(fmt, w, h, tw, th, flags=flags, **kw)
        shapes = flt.plane_shapes()
        sraw, sviews = _frame_buffer([(s[0], s[1]) for s, _ in shapes])
        draw, dviews = _frame_buffer([(d[0], d[1]) for _, d in shapes])
        for v, p in zip(sviews, planes):
            v[:] = p
        st0 = capi.host_buffer_stats()
        direct_runs = 0
        for it in range(40):
            for v in dviews:
                v[:] = 0
            before = capi.host_buffer_stats()
            flt.process(sviews, dviews)
            after = capi.host_buffer_stats()
            for i, (g, r) in enumerate(zip(dviews, ref)):
                assert_plane_close(g, r, False, f"registry/flags{flags}/iter{it}/plane{i}")
            if after["direct_dst_frames"] > before["direct_dst_frames"] and after["direct_src_frames"] > before["direct_src_frames"]:
                direct_runs += 1
                if direct_runs == 3:
                    break
            elif expect_direct:
                time.sleep(0.02)  # the helper thread is still page-locking the buffers
            elif it == 3:
                break
        st1 = capi.host_buffer_stats()
        flt.close()
        if expect_direct:
            assert direct_runs == 3, "the recycled buffers never became directly addressable"
            assert st1["registrations"] - st0["registrations"] == 2  # the source and the destination frame buffer
            assert st1["staged_frames"] - st0["staged_frames"] >= 2  # first sighting, and the one during registration
        else:
            assert st1["registrations"] == st0["registrations"] and direct_runs == 0
            assert st1["staged_frames"] - st0["staged_frames"] == 4
        del sraw, draw


class _Mapping:
    """A frame buffer in its own anonymous mapping that can be torn down and re-created AT THE SAME ADDRESS with fresh
    pages -- what a host's frame cache does when it frees a buffer and the next allocation lands where it was."""

    def __init__(self, sizes):
        import mmap

        self.libc = C.CDLL(None, use_errno=True)
        self.libc.mmap.restype = C.c_void_p
        self.libc.mmap.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_long]
        self.libc.munmap.argtypes = [C.c_void_p, C.c_size_t]
        self.sizes = sizes
        total = sum(r * ((c + 63) // 64 * 64) for r, c in sizes)
        self.length = (total + 2 * mmap.PAGESIZE) // mmap.PAGESIZE * mmap.PAGESIZE
        self.prot, self.flags = mmap.PROT_READ | mmap.PROT_WRITE, mmap.MAP_PRIVATE | mmap.MAP_ANONYMOUS
        self.addr = self.libc.mmap(None, self.length, self.prot, self.flags, -1, 0)
        assert self.addr not in (None, C.c_void_p(-1).value)

    def views(self, dtype=np.uint8):
        out, off = [], 0
        for r, c in self.sizes:
            pitch = (c + 63) // 64 * 64
            buf = (C.c_uint8 * (pitch * r)).from_address(self.addr + off)
            out.append(np.frombuffer(buf, np.uint8).reshape(r, pitch)[:, :c].view(dtype))
            off += pitch * r
        return out

    def remap(self):
        assert self.libc.munmap(self.addr, self.length) == 0
        again = self.libc.mmap(self.addr, self.length, self.prot, self.flags | 0x10, -1, 0)  # MAP_FIXED
        assert again == self.addr

    def close(self):
        self.libc.munmap(self.addr, self.length)


@pytest.mark.parametrize("side", ["dst", "src"])
def test_stale_registration_is_detected(capi, side):
    """The host frees a registered frame buffer and fresh memory is mapped at the same address (what a frame cache does
    under memory pressure).  A transfer through the stale registration reaches the buffer's FORMER physical pages: a
    destination frame would never arrive, a source frame would be an old one.  The pipeline's checks (arrival
    sentinels / probe words) notice, the registration is dropped for good, and the frame is redone through the staged
    path -- the caller gets the right frame every time."""
    _, fmt, w, h, tw, th, kw = CASES["c2_420p8_2x_tap3_mpeg2"]
    planes = make_planes(fmt, w, h, "noise", seed=33)
    ref, _ = oracle_frame(fmt, w, h, tw, th, planes, **kw)
    flt = make_filter(fmt, w, h, tw, th, flags=capi.FLAG_HOST_REGISTER | capi.FLAG_DST_PADDING_WRITABLE, **kw)
    shapes = flt.plane_shapes()
    m = _Mapping([(d[0], d[1]) for _, d in shapes] if side == "dst" else [(s[0], s[1]) for s, _ in shapes])

    def run(src_planes, want, tag):
        if side == "dst":
            dv = m.views()
            flt.process(src_planes, dv)
            got = dv
        else:
            sv = m.views()
            for v, p in zip(sv, src_planes):
                v[:] = p
            got = flt.process(sv)
        for i, (g, r) in enumerate(zip(got, want)):
            assert_plane_close(g, r, False, f"stale/{side}/{tag}/plane{i}")

    import time

    st0 = capi.host_buffer_stats()
    key = "direct_dst_frames" if side == "dst" else "direct_src_frames"
    for it in range(60):  # staged, staged while a helper thread page-locks the buffer, then direct
        run(planes, ref, f"before{it}")
        if capi.host_buffer_stats()[key] - st0[key] >= 2:
            break
        time.sleep(0.02)
    st1 = capi.host_buffer_stats()
    assert st1[key] - st0[key] >= 2 and st1["registrations"] > st0["registrations"] and st1["registered_bytes"] > 0
    m.remap()
    planes2 = make_planes(fmt, w, h, "noise", seed=34)
    ref2, _ = oracle_frame(fmt, w, h, tw, th, planes2, **kw)
    for it in range(3):
        run(planes2, ref2, f"after{it}")
    flt.close()
    m.close()
    assert capi.host_buffer_stats()["registered_bytes"] == 0  # the last registering filter took every registration with it


# ------------------------------------------------------------------------------------------ more than one GPU

def _two_gpus(capi):
    if capi.device_count() < 2:
        pytest.skip("needs two GPUs")


@pytest.mark.parametrize("name", ["c2_420p8_2x_tap3_mpeg2", "c5_420p10_quarter_tap6_blur", "up1p5_tap3_420p8", "c4_rgbps_2x_tap8"])
def test_two_gpu_row_band_split(capi, name):
    """One frame cut into one band per GPU (jinc_filter_process_split over devices 0 and 1) and into five bands
    alternating between the GPUs: byte-identical to the single-GPU whole frame."""
    _two_gpus(capi)
    _, fmt, w, h, tw, th, kw = CASES[name]
    planes = make_planes(fmt, w, h, "noise", seed=13)
    one = make_filter(fmt, w, h, tw, th, devices=(0,), **kw)
    whole = one.process(planes)
    one.close()
    flt = make_filter(fmt, w, h, tw, th, devices=(0, 1), **kw)
    assert flt.num_devices == 2
    for how in (dict(split=True), dict(bands=5)):
        got = flt.process(planes, **how)
        for i, (a, b) in enumerate(zip(whole, got)):
            assert np.array_equal(a, b), f"{name}: plane {i} differs ({how})"
    flt.close()


def test_two_gpu_frame_round_robin(capi):
    """jinc_filter_submit hands consecutive frames to alternating GPUs; every frame comes back in its own buffers and
    matches the oracle whichever GPU computed it."""
    _two_gpus(capi)
    _, fmt, w, h, tw, th, kw = CASES["c2_420p8_2x_tap3_mpeg2"]
    flt = make_filter(fmt, w, h, tw, th, devices=(0, 1), **kw)
    frames = [make_planes(fmt, w, h, "noise", seed=70 + s) for s in range(10)]
    outs = [flt.alloc_dst() for _ in frames]
    tickets = []
    for f, o in zip(frames, outs):
        if len(tickets) >= flt.num_slots:
            flt.wait(tickets.pop(0))
        tickets.append(flt.submit(f, o))
    for t in tickets:
        flt.wait(t)
    for f, o in zip(frames, outs):
        ref, _ = oracle_frame(fmt, w, h, tw, th, f, **kw)
        for g, r in zip(o, ref):
            assert_plane_close(g, r, False, "round robin")
    flt.close()


PLAN_CASES = ["c1_yv12_2x_tap3", "c2_420p8_2x_tap3_mpeg2", "c3_444p16_2x_tap4_crop", "c4_rgbps_2x_tap8", "up2x_tap6_420p8",
              "yuva420_14bit_2x", "up4to3_tap3_420p8", "up4x_tap3_420p8", "c5_420p10_quarter_tap6_blur", "half_tap3_yv12",
              "quarter_tap4_422p12", "third_tap3_y8",
              # ratios whose positions never repeat exactly: every border pixel keeps its own weights (JINC_SK_PER_PIXEL)
              "up1p5_tap3_420p8", "up1p5_tap4_444p16_crop", "up5to4_tap3_420p8", "down3to4_tap3_444p10", "up1p5_tap3_f32_y"]


@pytest.mark.parametrize("name", PLAN_CASES)
def test_strip_plan_equals_prologue_path(capi, name, monkeypatch):
    """Whole-frame launches run their border strips from the table's strip plan (jinc_table_strip_plan: patches, thread
    records and packed weight blocks worked out once per table); with JINCRESIZE_B200_STRIP_PLAN=0 a table has no plan and
    every strip block derives its work in its prologue.  Both accumulate every sample in the same tap order: the frames
    must be BYTE-identical (and both within the bar of the oracle, checked by the other tests)."""
    _, fmt, w, h, tw, th, kw = CASES[name]
    planes = make_planes(fmt, w, h, "noise", seed=11)
    monkeypatch.setenv("JINCRESIZE_B200_STRIP_PLAN", "0")
    plain = make_filter(fmt, w, h, tw, th, **kw)
    assert all(plain.table(i).strip_plan == (0, 0) for i in range(plain.num_tables))
    want = plain.process(planes)
    plain.close()
    monkeypatch.delenv("JINCRESIZE_B200_STRIP_PLAN")
    flt = make_filter(fmt, w, h, tw, th, **kw)
    n, staged = flt.table(0).strip_plan
    assert n > 0 and 0 <= staged <= n, f"{name}: no strip plan was built ({n}, {staged})"
    got = flt.process(planes)
    for i, (a, b) in enumerate(zip(want, got)):
        assert np.array_equal(a, b), f"{name}: plane {i} differs between the planned and the prologue strips"
    ref, _ = oracle_frame(fmt, w, h, tw, th, planes, **kw)
    for i, (g, r) in enumerate(zip(got, ref)):
        assert_plane_close(g, r, fmt.bits == 32, f"{name}/plan/plane{i}")
    flt.close()


@pytest.mark.parametrize("name", ["c4_rgbps_2x_tap8", "up2x_tap7_f32_y"])
def test_bulk_copy_staging_equals_register_staging(capi, name, monkeypatch):
    """JINCRESIZE_B200_TMA=1: float tiles of the exact-2x kernel are landed in shared memory by the bulk-copy engine
    (cp.async.bulk + mbarrier, one copy per tile row) instead of through registers; the arithmetic is untouched, so the
    frames are byte-identical.  Pinned device planes (16-byte aligned rows) are what the frame pipeline provides."""
    _, fmt, w, h, tw, th, kw = CASES[name]
    planes = make_planes(fmt, w, h, "noise", seed=5)
    flt = make_filter(fmt, w, h, tw, th, **kw)
    want = flt.process(planes)
    monkeypatch.setenv("JINCRESIZE_B200_TMA", "1")
    got = flt.process(planes)
    monkeypatch.delenv("JINCRESIZE_B200_TMA")
    for i, (a, b) in enumerate(zip(want, got)):
        assert np.array_equal(a, b), f"{name}: plane {i} differs between bulk-copy and register staging"
    flt.close()
