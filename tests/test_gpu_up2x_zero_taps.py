"""Exactly-zero Jinc taps skipped by the exact-2x kernel of 8- and 16-bit planes (csrc/jinc_up2x_taps.h).

The disc-shaped window leaves about a third of every fs x fs phase block at weight 0.  A table takes the tightest compiled
tap mask whose skipped taps are all zero in it; fma(s, 0, acc) == acc for finite s, so the frames must be byte-identical
to the kernel that multiplies every tap (JINCRESIZE_B200_UP2X_ZERO_TAPS=0)."""
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

from common import FULL_CASES, SMALL_CASES, assert_plane_close, make_filter, make_planes, oracle_frame
from minihost import avs_host as ah

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "tools"))
import gen_up2x_taps  # noqa: E402

PATH_UP2X = 1
SWITCH = "JINCRESIZE_B200_UP2X_ZERO_TAPS"

CASES = {c[0]: c for c in SMALL_CASES}
for _n in ("c1_yv12_2x_tap3", "c2_420p8_2x_tap3_mpeg2", "c3_444p16_2x_tap4_crop", "yuva420_14bit_2x", "up2x_tap6_420p8",
           "up2x_tap7_f32_y"):
    assert _n in CASES
# every chroma siting of tap 3 and tap 4, blur, other phase quantisations, an odd plane with partial tiles, 10/16 bits
for _tap in (3, 4):
    CASES[f"t{_tap}_444p8"] = (None, ah.Format("444", 8), 200, 120, 400, 240, dict(tap=_tap))
    for _fam, _bits in (("422", 8), ("420", 8)):
        for _cp in ("mpeg2", "mpeg1", "topleft"):
            CASES[f"t{_tap}_{_fam}p{_bits}_{_cp}"] = (None, ah.Format(_fam, _bits), 200, 120, 400, 240, dict(tap=_tap, cplace=_cp))
CASES["t3_420p8_blur1.3"] = (None, ah.YUV420P8, 200, 120, 400, 240, dict(tap=3, blur=1.3))
CASES["t4_420p10_blur0.8"] = (None, ah.Format("420", 10), 200, 120, 400, 240, dict(tap=4, blur=0.8))
CASES["t3_422p8_quant64x100"] = (None, ah.Format("422", 8), 200, 120, 400, 240, dict(tap=3, quant_x=64, quant_y=100))
CASES["t4_y16_quant200x48_shift"] = (None, ah.Format("y", 16), 200, 120, 400, 240, dict(tap=4, quant_x=200, quant_y=48,
                                                                                         src_left=0.37, src_top=0.11))
CASES["t3_y8_odd"] = (None, ah.Format("y", 8), 301, 171, 602, 342, dict(tap=3))
CASES["t3_420p10_odd_crop"] = (None, ah.Format("420", 10), 287, 163, 574, 326, dict(tap=3, src_left=1.3, src_top=0.6))
CASES["t4_444p16_topleft"] = (None, ah.YUV444P16, 160, 96, 320, 192, dict(tap=4, cplace="topleft"))


def _process(fmt, w, h, tw, th, kw, planes, bands=0):
    flt = make_filter(fmt, w, h, tw, th, **kw)
    out = flt.process([p.copy() for p in planes], bands=bands)
    infos = [flt.table(i).info for i in range(flt.num_tables)]
    flt.close()
    return out, infos


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_zero_taps_byte_identical(native_built, name, monkeypatch):
    _, fmt, w, h, tw, th, kw = CASES[name]
    planes = make_planes(fmt, w, h, "noise", seed=17)
    monkeypatch.setenv(SWITCH, "0")
    want, full_infos = _process(fmt, w, h, tw, th, kw, planes)
    monkeypatch.delenv(SWITCH)
    got, infos = _process(fmt, w, h, tw, th, kw, planes)
    for i, (a, b) in enumerate(zip(want, got)):
        assert np.array_equal(a, b), f"{name}: plane {i} differs between every tap and the zero taps skipped"
    for full, info in zip(full_infos, infos):
        if info.fast_path == PATH_UP2X:
            assert full.up2x_taps == 4 * info.filter_size ** 2
            if fmt.bits < 32 and info.filter_size <= 9:
                assert info.up2x_taps < 4 * info.filter_size ** 2, f"{name}: no tap mask was selected"
    banded, _ = _process(fmt, w, h, tw, th, kw, planes, bands=3)
    for i, (a, b) in enumerate(zip(got, banded)):
        assert np.array_equal(a, b), f"{name}: plane {i} differs between 3 row bands and the whole frame"
    ref, _ = oracle_frame(fmt, w, h, tw, th, planes, **kw)
    for i, (g, r) in enumerate(zip(got, ref)):
        assert_plane_close(g, r, fmt.bits == 32, f"{name}/zero-taps/plane{i}")


def _nonzero_phase_taps(table):
    info = table.info
    return sum(int(np.count_nonzero(table.pixel_weights(info.interior_x0 + px, info.interior_y0 + py)))
               for py in range(2) for px in range(2))


@pytest.mark.gpu
def test_zero_tap_variant_selection(native_built, monkeypatch):
    """Configs 1 and 2 multiply no zero weight at all; the crop of config 3 takes the generic mask of its (ox1, oy1)."""
    full = {c[0]: c for c in FULL_CASES}
    for name in ("config1", "config2"):
        _, fmt, w, h, tw, th, kw = full[name]
        flt = make_filter(fmt, w, h, tw, th, **kw)
        for k in range(flt.num_tables):
            t = flt.table(k)
            assert t.info.fast_path == PATH_UP2X
            assert t.info.up2x_taps == _nonzero_phase_taps(t), f"{name} table {k}"
        flt.close()
    _, fmt, w, h, tw, th, kw = full["config3"]
    flt = make_filter(fmt, w, h, tw, th, **kw)
    info = flt.table(0).info
    assert info.fast_path == PATH_UP2X and _nonzero_phase_taps(flt.table(0)) <= info.up2x_taps < 4 * info.filter_size ** 2
    flt.close()
    monkeypatch.setenv(SWITCH, "0")
    for name in ("config2", "config3"):
        _, fmt, w, h, tw, th, kw = full[name]
        flt = make_filter(fmt, w, h, tw, th, **kw)
        for k in range(flt.num_tables):
            info = flt.table(k).info
            assert info.up2x_taps == 4 * info.filter_size ** 2
        flt.close()


def _ffma2_per_kernel(lib_path):
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
def test_zero_tap_kernels_drop_the_ffma2():
    """The masks reach the machine code: config 2's luma (centred) and chroma (MPEG2) variants issue one FFMA2 per live
    tap and cell of a thread (124 and 130 taps, four cells), the every-tap kernels all 4 * fs^2 * 4."""
    from jinc_b200 import paths

    n = _ffma2_per_kernel(paths.cuda_lib())
    for t in ("unsigned char", "unsigned short"):
        assert n[f"void jinc_rs::resample_up2x<{t}, 7, 1, 1, false, 1>(jinc_rs::UpArgs, jinc_rs::UpWeights<7>)"] == 496
        assert n[f"void jinc_rs::resample_up2x<{t}, 7, 0, 1, false, 2>(jinc_rs::UpArgs, jinc_rs::UpWeights<7>)"] == 520
        for ox, oy in ((0, 0), (0, 1), (1, 0), (1, 1)):
            assert n[f"void jinc_rs::resample_up2x<{t}, 7, {ox}, {oy}, false, 0>(jinc_rs::UpArgs, jinc_rs::UpWeights<7>)"] == 784
            assert n[f"void jinc_rs::resample_up2x<{t}, 9, {ox}, {oy}, false, 0>(jinc_rs::UpArgs, jinc_rs::UpWeights<9>)"] == 1296
        for fs in (7, 9):  # every variant: a row loop left rolled would show fewer
            for m, (_, ox, oy, mask) in enumerate(gen_up2x_taps.variants(fs), start=1):
                live = sum(bin(b).count("1") for ph in mask for blk in ph for b in blk)
                kern = f"void jinc_rs::resample_up2x<{t}, {fs}, {ox}, {oy}, false, {m}>(jinc_rs::UpArgs, jinc_rs::UpWeights<{fs}>)"
                assert n[kern] == 4 * live, kern


def test_tap_mask_header_is_generated():
    """csrc/jinc_up2x_taps.h is exactly what tools/gen_up2x_taps.py writes."""
    gen = subprocess.run([sys.executable, os.path.join(REPO, "tools", "gen_up2x_taps.py")], capture_output=True, text=True,
                         check=True).stdout
    with open(os.path.join(REPO, "avisynth-jincresize_b200", "csrc", "jinc_up2x_taps.h")) as f:
        assert f.read() == gen
