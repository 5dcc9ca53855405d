#!/usr/bin/env python
"""tools/bench_f16.py -- half-precision planes (JINC_SAMPLE_F16) against float32 planes on bench.py's geometries.

    python tools/bench_f16.py [--configs 2 4 5] [--pairs 3] [--steps K] [--e2e-steps K] [--warmup W]

For each config the same seeded float16 frames run as half planes and, widened, as float32 planes (the sample type of
the config is replaced; geometry, tap, crop, blur and cplace are bench.py's).  Prints one JSON line per config:
  kernel   jinc_filter_process_device_batch on device-resident frames (CUDA events around `steps` launches per table),
           float32 and half alternated in `pairs` pairs; every batch is at least twice the 126 MB L2.  Gpixel/s counts
           output luma pixels; fma_frac is the algorithmic 2 * fs^2 FLOP per output sample over the FP32-FMA peak that
           bench.py measures (avisynth-jincresize_b200/fma_peak)
  e2e      jinc_filter_submit / jinc_filter_wait on caller-pinned host frames, `inflight` frames in flight: frames/s,
           float32 and half alternated in the same pairs
  check    the timed half output against the timed float32 output rounded to half (NumPy's cast rounds to nearest
           even, as the kernels do), on sampled rows of the first and last frame of the batch
A GPU is required: there is no CPU fallback."""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "avisynth-jincresize_b200"))

import bench  # noqa: E402  (the workloads and the FMA peak)
from jinc_b200 import capi  # noqa: E402

L2_BYTES = 126e6


def make_filter(cfg, half: bool, slots: int):
    fmt, kw = cfg["fmt"], cfg["kw"]
    sw, sh = fmt.subsampling
    return capi.Filter(src_w=cfg["w"], src_h=cfg["h"], target_w=cfg["tw"], target_h=cfg["th"], n_planes=len(fmt.planes),
                       sample_bytes=capi.SAMPLE_F16 if half else 4, bits=16 if half else 32, sub_w=sw, sub_h=sh,
                       src_left=kw.get("src_left", 0.0), src_top=kw.get("src_top", 0.0), quant_x=kw.get("quant_x", 256),
                       quant_y=kw.get("quant_y", 256), tap=cfg["tap"], blur=kw.get("blur", 0.0),
                       cplace=kw.get("cplace", "mpeg2"), devices=[0], slots_per_device=slots)


def half_frame(cfg, seed: int):
    """Seeded float16 noise: [0, 1) for luma and RGB, [-0.5, 0.5) for chroma."""
    fmt = cfg["fmt"]
    rng = np.random.default_rng(0x46313620 ^ seed)
    planes = []
    for i in range(len(fmt.planes)):
        ph, pw = fmt.plane_shape(i, cfg["w"], cfg["h"])
        chroma = i in (1, 2) and fmt.family not in ("rgbp", "rgbap")
        planes.append(np.ascontiguousarray((rng.random((ph, pw), dtype=np.float32) - (0.5 if chroma else 0.0)).astype(np.float16)))
    return planes


class Arm:
    """One sample type of one config: filter, device-resident batch, pinned host frames."""

    def __init__(self, cfg, half: bool, frames_np, inflight: int):
        import torch

        self.half = half
        self.dtype = np.float16 if half else np.float32
        tdt = torch.float16 if half else torch.float32
        sb = np.dtype(self.dtype).itemsize
        self.flt = make_filter(cfg, half, inflight)
        self.shapes = self.flt.plane_shapes()
        self.infos = [self.flt.table(k).info for k in range(self.flt.num_tables)]
        self.dev_dst, self.keep, self.host_src, self.host_dst = [], [], [], []
        dev = []
        for planes in frames_np:
            fr = capi.Frame()
            dd = []
            for i, ((sshape, dshape), p) in enumerate(zip(self.shapes, planes)):
                sp = (sshape[1] * sb + 255) // 256 * 256 // sb
                dp = (dshape[1] * sb + 255) // 256 * 256 // sb
                s = torch.zeros((sshape[0], sp), dtype=tdt, device="cuda")
                s[:, : sshape[1]].copy_(torch.from_numpy(p.astype(self.dtype)))
                d = torch.zeros((dshape[0], dp), dtype=tdt, device="cuda")
                fr.src[i], fr.src_pitch[i] = s.data_ptr(), sp * sb
                fr.dst[i], fr.dst_pitch[i] = d.data_ptr(), dp * sb
                self.keep.append(s)
                dd.append(d)
            dev.append(fr)
            self.dev_dst.append(dd)
            self.host_src.append([torch.from_numpy(p.astype(self.dtype)).pin_memory() for p in planes])
            self.host_dst.append([torch.zeros(dshape, dtype=tdt).pin_memory() for _, dshape in self.shapes])
        self.frames = (capi.Frame * len(dev))(*dev)
        self.raw = [self.flt._frame([t.numpy() for t in s], [t.numpy() for t in d]) for s, d in zip(self.host_src, self.host_dst)]
        self.stream = torch.cuda.Stream()
        torch.cuda.synchronize()

    def kernel_step(self):
        st = self.stream.cuda_stream
        self.flt.process_device_batch(self.frames, 0, 1, 3, st)
        if self.flt.num_tables > 1:
            self.flt.process_device_batch(self.frames, 0, 2, 3, st)

    def kernel_ms(self, steps: int, warmup: int) -> float:
        import torch

        for _ in range(warmup):
            self.kernel_step()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for _ in range(steps):
            self.kernel_step()
        e1.record(self.stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / steps

    def e2e_fps(self, steps: int, inflight: int) -> float:
        def run(k):
            tickets = []
            for _ in range(k):
                for fr in self.raw:
                    if len(tickets) >= inflight:
                        self.flt.wait(tickets.pop(0))
                    tickets.append(self.flt.submit_raw(fr))
            for t in tickets:
                self.flt.wait(t)

        run(1)
        t0 = time.perf_counter()
        run(steps)
        return steps * len(self.raw) / (time.perf_counter() - t0)

    def rows(self, f: int, i: int, ys):
        return self.dev_dst[f][i][ys, : self.shapes[i][1][1]].cpu().numpy()

    def close(self):
        self.flt.close()


def measure(cid: int, args) -> dict:
    import torch

    cfg = bench.CONFIGS[cid]
    fmt = cfg["fmt"]
    half_bytes = sum((fmt.plane_shape(i, cfg["w"], cfg["h"])[0] * fmt.plane_shape(i, cfg["w"], cfg["h"])[1] +
                      fmt.plane_shape(i, cfg["tw"], cfg["th"])[0] * fmt.plane_shape(i, cfg["tw"], cfg["th"])[1]) * 2
                     for i in range(len(fmt.planes)))
    F = max(cfg["frames"], math.ceil(2 * L2_BYTES / half_bytes))
    frames = [half_frame(cfg, seed=f) for f in range(F)]
    arms = {False: Arm(cfg, False, frames, args.inflight), True: Arm(cfg, True, frames, args.inflight)}
    infos = arms[True].infos
    assert [i.fast_path for i in infos] == [i.fast_path for i in arms[False].infos]
    flop = bench.algorithmic_work(cfg, infos[0].filter_size, infos[-1].filter_size)[0] * F
    peak_tf, peak_how = bench.fma_peak_tflops()
    gpix = cfg["tw"] * cfg["th"] * F / 1e9
    kern = {False: [], True: []}
    e2e = {False: [], True: []}
    for _ in range(args.pairs):
        for half in (False, True):
            kern[half].append(arms[half].kernel_ms(args.steps, args.warmup))
    for _ in range(args.pairs):
        for half in (False, True):
            e2e[half].append(arms[half].e2e_fps(args.e2e_steps, args.inflight))

    # the timed outputs: half against float32 rounded to half on sampled rows of the first and last frame
    checked = bad = 0
    for f in (0, F - 1):
        for i, (_, dshape) in enumerate(arms[True].shapes):
            H = dshape[0]
            ys = sorted(set([0, 1, H // 2, H - 2, H - 1] + list(range(0, H, 37))))
            a, b = arms[True].rows(f, i, ys), arms[False].rows(f, i, ys)
            with np.errstate(over="ignore"):
                want = b.astype(np.float16)
            bad += int((a.view(np.uint16) != want.view(np.uint16)).sum())
            checked += a.size
    for a in arms.values():
        a.close()
    arms.clear()
    torch.cuda.empty_cache()

    def kern_obj(ms_list):
        return {"ms_per_step": [round(m, 4) for m in ms_list], "gpixel_s": [round(gpix / (m * 1e-3), 2) for m in ms_list],
                "fma_frac": [round(flop / (m * 1e-3) / 1e12 / peak_tf, 4) for m in ms_list]}

    k32, k16 = statistics.median(kern[False]), statistics.median(kern[True])
    f32, f16 = statistics.median(e2e[False]), statistics.median(e2e[True])
    return {"config": cid, "workload": cfg["name"], "sample_types": "float32 vs half (same geometry, widened input)",
            "kernel_paths": [bench.KERNEL_NAMES.get(i.fast_path, "resample_strips") for i in infos],
            "frames_per_batch": F, "batch_mb": {"f16": round(F * half_bytes / 1e6, 1), "f32": round(2 * F * half_bytes / 1e6, 1)},
            "steps": args.steps, "pairs": args.pairs,
            "kernel": {"f32": kern_obj(kern[False]), "f16": kern_obj(kern[True]), "median_time_ratio_f16_over_f32": round(k16 / k32, 4)},
            "fma_peak_tflops": round(peak_tf, 2), "fma_peak_source": peak_how,
            "e2e": {"api": "jinc_filter_submit/jinc_filter_wait, caller-pinned host frames, %d in flight" % args.inflight,
                    "steps": args.e2e_steps, "f32_fps": [round(v, 2) for v in e2e[False]], "f16_fps": [round(v, 2) for v in e2e[True]],
                    "median_fps_ratio_f16_over_f32": round(f16 / f32, 4)},
            "check": {"samples": checked, "differ": bad, "ok": bad == 0,
                      "what": "half output == float32 output rounded to half, sampled rows of frames 0 and F-1"}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[2, 4, 5])
    ap.add_argument("--pairs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--inflight", type=int, default=3)
    args = ap.parse_args()
    import torch

    if capi.device_count() < 1 or not torch.cuda.is_available():
        sys.exit("bench_f16: no CUDA device (there is no CPU fallback)")
    name = torch.cuda.get_device_name(0)
    for cid in args.configs:
        line = measure(cid, args)
        line["device"] = name
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
