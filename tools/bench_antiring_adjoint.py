#!/usr/bin/env python
"""tools/bench_antiring_adjoint.py -- the backward of resize + anti-ringing (jinc_antiring_adjoint_planes_device) against the
plain adjoint (jinc_resize_adjoint_planes_device), kernel-only.

    python tools/bench_antiring_adjoint.py [--configs 2 4 5] [--pairs 3] [--seconds 1.0]
    python tools/bench_antiring_adjoint.py --profile          (a torch.profiler run of its own: time per launch)

For the luma table of bench.py's configs 2 (1080p -> 2160p, tap 3), 4 (tap 8, float RGB) and 5 (the 1/4 downscale), float32
and half source planes: a batch larger than twice the 126 MB L2 (source, resized planes and the three gradients) goes
through the backward at strength 1 and through the plain adjoint, each timed with CUDA events over a window of at least
`seconds`, the two alternated in `pairs` pairs.  The same is done for the forward through the tensor API, jinc_resize with
antiring=1 against without.  --profile times each of the backward's three launches (antiring_grad_out, the adjoint
kernels, antiring_route_gather) and reports, for the two new passes, the bytes they need over their time against the
7.7 TB/s HBM bandwidth of the data sheet.  The bytes a pass needs, at the least:
  antiring_grad_out      y (sample) + g (4 B) in, g_y (4 B) out per output sample, and the anchors: every source sample
                         once, or four per output sample when that is fewer (downscales);
  antiring_route_gather  y per output sample, the anchors as above, and per clamped output sample its g (4 B) and the
                         grad_src sample it reaches read and written (8 B).
One JSON line per measurement, the card's name, power limit and SM clock before and after.  A GPU is required: there is
no CPU fallback."""
from __future__ import annotations

import argparse
import json
import os
import re
import statistics
import subprocess
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "avisynth-jincresize_b200"))

import bench  # noqa: E402  (the workloads)
from jinc_b200 import capi  # noqa: E402
from jinc_b200.tensor import jinc_resize  # noqa: E402
from oracle import cpu as oc  # noqa: E402  (the per-table geometry)

L2_BYTES = 126e6
HBM_BYTES_S = 7.7e12
SAMPLES = {"float32": (4, 4), "float16": (capi.SAMPLE_F16, 2)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def luma_table(ctx, cfg):
    fmt, kw = cfg["fmt"], cfg["kw"]
    sw, sh = fmt.subsampling
    p = oc.plane_params(cfg["w"], cfg["h"], cfg["tw"], cfg["th"], src_left=kw.get("src_left", 0.0),
                        src_top=kw.get("src_top", 0.0), quant_x=kw.get("quant_x", 256), quant_y=kw.get("quant_y", 256),
                        tap=cfg["tap"], sub_w=sw, sub_h=sh, cplace=kw.get("cplace", "mpeg2"))[0]
    return capi.Table(ctx, quant_x=p.quant_x, quant_y=p.quant_y, src_w=p.src_w, src_h=p.src_h, dst_w=p.dst_w,
                      dst_h=p.dst_h, radius=capi.radius_for_tap(cfg["tap"]), blur=float(np.float32(kw.get("blur", 0.0))),
                      crop_left=p.crop_left, crop_top=p.crop_top, crop_w=p.crop_w, crop_h=p.crop_h), p


def timed(fn, seconds, stream):
    import torch

    fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    fn()
    e1.record(stream)
    e1.synchronize()
    steps = max(1, int(seconds * 1e3 / max(e0.elapsed_time(e1), 1e-3)) + 1)
    e0.record(stream)
    for _ in range(steps):
        fn()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1) / steps, steps


class Workload:
    """Device buffers of one (table, sample type) batch and the two backward calls on them."""

    def __init__(self, tab, p, dtype, stream):
        import torch

        self.tab, self.p, self.dtype = tab, p, dtype
        code, sb = SAMPLES[dtype]
        H, W, h, w = p.src_h, p.src_w, p.dst_h, p.dst_w
        per_plane = H * W * (sb + 4) + h * w * (sb + 8)
        self.n = n = int(np.ceil(2 * L2_BYTES / per_plane))
        self.stream = stream
        st = stream.cuda_stream
        dt = getattr(torch, dtype)
        pitch = (w * sb + 15) // 16 * 16 // sb
        with torch.cuda.stream(stream):
            x = torch.rand((n, H, W), device="cuda")
            x[..., : W // 2] += 1.0  # hard edges: every row has clamped outputs beside them
            self.x = x.to(dt)
            self.y = torch.empty((n, h, pitch), dtype=dt, device="cuda")
            self.g = torch.randn((n, h, w), device="cuda")
            self.gy = torch.empty((n, h, w), device="cuda")
            self.gs = torch.empty((n, H, W), device="cuda")
        tab.resize_planes_device(code, 0.0, n, self.x.data_ptr(), W * sb, H * W * sb, self.y.data_ptr(), pitch * sb,
                                 h * pitch * sb, st)
        args = ((self.x.data_ptr(), W * sb, H * W * sb), (self.y.data_ptr(), pitch * sb, h * pitch * sb),
                (self.g.data_ptr(), w * 4, h * w * 4), (self.gy.data_ptr(), w * 4, h * w * 4),
                (self.gs.data_ptr(), W * 4, H * W * 4))
        self.backward = lambda: tab.antiring_adjoint_planes_device(code, 1.0, n, *args, st)
        self.adjoint = lambda: tab.adjoint_planes_device(n, self.g.data_ptr(), w * 4, h * w * 4, self.gs.data_ptr(), W * 4,
                                                         H * W * 4, st)
        torch.cuda.synchronize()

    def clamped_fraction(self):
        """Share of output samples the clamp moves at strength 1 (their g_y is +0 while g is not)."""
        import torch

        self.backward()
        torch.cuda.synchronize()
        return float(((self.gy == 0) & (self.g != 0)).float().mean())

    def pass_bytes(self, clamped):
        """Bytes antiring_grad_out and antiring_route_gather need (module docstring)."""
        sb = SAMPLES[self.dtype][1]
        H, W, h, w = self.p.src_h, self.p.src_w, self.p.dst_h, self.p.dst_w
        anchors = min(H * W, 4 * h * w) * sb
        grad_out = self.n * (h * w * (sb + 8) + anchors)
        gather = self.n * (h * w * (sb + 12 * clamped) + anchors)
        return grad_out, gather


def bench_backward(cid, tab, p, dtype, args):
    import torch

    wl = Workload(tab, p, dtype, torch.cuda.Stream())
    b_ms, a_ms, steps = [], [], []
    for _ in range(args.pairs):
        t, s1 = timed(wl.backward, args.seconds, wl.stream)
        b_ms.append(t)
        t, s2 = timed(wl.adjoint, args.seconds, wl.stream)
        a_ms.append(t)
        steps.append((s1, s2))
    b, a = statistics.median(b_ms), statistics.median(a_ms)
    H, W = p.src_h, p.src_w
    return {"config": cid, "table": "luma", "dtype": dtype, "src": [W, H], "dst": [p.dst_w, p.dst_h],
            "fs": tab.info.filter_size, "path": capi.PATH_NAMES.get(tab.info.fast_path), "planes": wl.n, "steps": steps,
            "backward_ms": [round(v, 4) for v in b_ms], "adjoint_ms": [round(v, 4) for v in a_ms],
            "backward_src_gsamples_s": round(wl.n * H * W / (b * 1e-3) / 1e9, 2),
            "adjoint_src_gsamples_s": round(wl.n * H * W / (a * 1e-3) / 1e9, 2),
            "backward_over_adjoint_time": round(b / a, 3), "clamped_fraction": round(wl.clamped_fraction(), 4)}


def bench_forward(cid, p, dtype, args):
    """jinc_resize with antiring=1 against without, through the tensor API (forward only, no graph)."""
    import torch

    sb = SAMPLES[dtype][1]
    H, W, h, w = p.src_h, p.src_w, p.dst_h, p.dst_w
    n = int(np.ceil(2 * L2_BYTES / (sb * (H * W + h * w))))
    stream = torch.cuda.Stream()
    geo = dict(width=w, height=h, tap=bench.CONFIGS[cid]["tap"], src_left=p.crop_left, src_top=p.crop_top,
               src_width=p.crop_w, src_height=p.crop_h, blur=bench.CONFIGS[cid]["kw"].get("blur", 0.0))
    with torch.cuda.stream(stream):
        x = torch.rand((n, H, W), device="cuda")
        x[..., : W // 2] += 1.0
        x = x.to(getattr(torch, dtype))
    torch.cuda.synchronize()

    def run(s):
        with torch.cuda.stream(stream), torch.no_grad():
            jinc_resize(x, antiring=s, **geo)

    on_ms, off_ms = [], []
    for _ in range(args.pairs):
        on_ms.append(timed(lambda: run(1.0), args.seconds, stream)[0])
        off_ms.append(timed(lambda: run(0.0), args.seconds, stream)[0])
    on, off = statistics.median(on_ms), statistics.median(off_ms)
    return {"config": cid, "table": "luma", "dtype": dtype, "tensor_forward": True, "planes": n,
            "antiring_ms": [round(v, 4) for v in on_ms], "plain_ms": [round(v, 4) for v in off_ms],
            "antiring_over_plain_time": round(on / off, 3)}


def profile(configs):
    """Time per launch of the backward at strength 1 and of the plain adjoint, one table and sample type at a time."""
    import torch
    from torch.profiler import ProfilerActivity

    ctx = capi.Context(0)
    for cid in configs:
        tab, p = luma_table(ctx, bench.CONFIGS[cid])
        for dtype in SAMPLES:
            wl = Workload(tab, p, dtype, torch.cuda.Stream())
            clamped = wl.clamped_fraction()
            reps = 5
            with torch.profiler.profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(reps):
                    wl.backward()
                torch.cuda.synchronize()
            kern = {}
            for e in prof.key_averages():
                t = getattr(e, "device_time_total", None)
                if t is None:
                    t = e.cuda_time_total
                m = re.search(r"antiring_grad_out|antiring_route_gather|adjoint_up2x|adjoint_general", e.key)
                if t and m:
                    kern[m.group(0)] = kern.get(m.group(0), 0.0) + t / reps / 1e3  # ms per backward call
            go, ga = wl.pass_bytes(clamped)
            rec = {"config": cid, "dtype": dtype, "planes": wl.n, "clamped_fraction": round(clamped, 4),
                   "ms_per_call": {k: round(v, 4) for k, v in sorted(kern.items())}}
            for k, b in (("antiring_grad_out", go), ("antiring_route_gather", ga)):
                if k in kern:
                    bw = b / (kern[k] * 1e-3)
                    rec[k] = {"bytes": int(b), "tb_s": round(bw / 1e12, 3), "frac_of_7p7": round(bw / HBM_BYTES_S, 3)}
            print(json.dumps(rec), flush=True)
            del wl
            torch.cuda.empty_cache()
        tab.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="*", default=[2, 4, 5])
    ap.add_argument("--pairs", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--profile", action="store_true")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available() or capi.device_count() < 1:
        sys.exit("bench_antiring_adjoint.py: no CUDA device (there is no CPU fallback)")
    print(json.dumps({"card": card()}), flush=True)
    if args.profile:
        profile(args.configs)
    else:
        ctx = capi.Context(0)
        for cid in args.configs:
            tab, p = luma_table(ctx, bench.CONFIGS[cid])
            for dtype in SAMPLES:
                print(json.dumps(bench_backward(cid, tab, p, dtype, args)), flush=True)
                torch.cuda.empty_cache()
                print(json.dumps(bench_forward(cid, p, dtype, args)), flush=True)
                torch.cuda.empty_cache()
            tab.close()
    print(json.dumps({"card_after": card()}), flush=True)


if __name__ == "__main__":
    main()
