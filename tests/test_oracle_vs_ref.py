"""Pins the CPU oracle to the reference by EXECUTION: the unmodified reference sources, compiled into
oracle/_ref/libjincresize_ref.so and driven through its own AviSynth plugin API under the mini-host, must agree with
oracle/jinc_oracle.c bit for bit (LUT as float for all 16 taps, tables, opt=0 frames).  Skipped only where the prebuilt
reference library is absent; tests/test_oracle_golden.py covers that case with committed digests."""
import numpy as np
import pytest

from oracle import ref as oref

from common import SMALL_CASES, make_planes, oracle_frame


@pytest.fixture(scope="module")
def ref(native_built, have_ref):
    if not have_ref:
        pytest.skip("oracle/_ref not built (`make ref` needs the reference sources)")
    from minihost import avs_host as ah
    from jinc_b200 import paths

    env = ah.Env()
    env.load_plugin(oref.REF_PLUGIN)
    return env, oref.RefTables()


def test_lut_matches_reference_for_every_tap(ref):
    from minihost import avs_host as ah
    from oracle import cpu as oc

    env, rt = ref
    src = env.source(ah.Format("y", 8), 80, 80, [[np.zeros((80, 80), np.uint8)]])
    for tap in range(1, 17):
        for blur in (None, 0.9, 1.1):
            kw = dict(tap=tap, opt=0)
            if blur:
                kw["blur"] = blur
            clip = env.invoke("JincResize", src, 120, 120, **kw)
            theirs = rt.lut(clip).astype(np.float32)
            mine = oc.make_lut(tap, blur or 0.0).astype(np.float32)
            assert np.array_equal(theirs.view(np.uint32), mine.view(np.uint32)), (tap, blur)
            clip.release()
    src.release()


def test_radius_constants_match_reference_doubles(ref):
    """jinc zeros (tap -> radius): filter_size and support of a tiny clip pin every one of the 16 doubles."""
    from minihost import avs_host as ah
    from oracle import cpu as oc

    env, rt = ref
    src = env.source(ah.Format("y", 8), 80, 80, [[np.zeros((80, 80), np.uint8)]])
    for tap in range(1, 17):
        clip = env.invoke("JincResize", src, 57, 43, tap=tap, opt=0)
        fs, cs, meta, factor = rt.table(clip, 0, 57, 43)
        p = oc.plane_params(80, 80, 57, 43, tap=tap)[0]
        t = oc.Table(p, oc.make_lut(tap))
        assert t.filter_size == fs and np.array_equal(t.meta, meta)
        assert np.array_equal(t.factor.view(np.uint32), factor.view(np.uint32))
        clip.release()
    src.release()


@pytest.mark.parametrize("case", SMALL_CASES, ids=[c[0] for c in SMALL_CASES])
def test_tables_and_frames_bit_exact(ref, case):
    env, rt = ref
    name, fmt, w, h, tw, th, kw = case
    planes = make_planes(fmt, w, h, "noise")
    src = env.source(fmt, w, h, [planes])
    clip = env.invoke("JincResize", src, tw, th, opt=0, threads=1, **kw)
    theirs, _ = clip.get_frame(0)
    mine, tabs = oracle_frame(fmt, w, h, tw, th, planes, **kw)
    assert rt.count(clip) == len(tabs)
    sw, sh = fmt.subsampling
    for k, t in enumerate(tabs):
        dw, dh = (tw, th) if k == 0 else (tw >> sw, th >> sh)
        fs, cs, meta, factor = rt.table(clip, k, dw, dh)
        assert (fs, cs) == (t.filter_size, t.coeff_stride)
        assert np.array_equal(meta, t.meta)
        assert np.array_equal(factor.view(np.uint32), t.factor.view(np.uint32))
    for a, b in zip(theirs, mine):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    clip.release()
    src.release()


def test_reference_simd_paths_stay_within_one_lsb_of_opt0(ref):
    """Calibrates the +-1 LSB bar: the reference's own AVX2 path vs its opt=0 path."""
    from minihost import avs_host as ah

    env, _ = ref
    fmt, w, h = ah.YV12, 160, 90
    planes = make_planes(fmt, w, h, "noise")
    src = env.source(fmt, w, h, [planes])
    a, _ = env.invoke("JincResize", src, 320, 180, opt=0).get_frame(0)
    b, _ = env.invoke("JincResize", src, 320, 180, opt=2).get_frame(0)
    for x, y in zip(a, b):
        assert np.abs(x.astype(int) - y.astype(int)).max() <= 1
