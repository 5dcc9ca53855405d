#!/usr/bin/env python
"""tools/bench_adjoint.py -- the adjoint (jinc_resize_adjoint_planes_device) against the forward resize, kernel-only.

    python tools/bench_adjoint.py [--configs 1 2 3 4 5 6] [--pairs 3] [--seconds 1.0] [--torch-steps 20]
    python tools/bench_adjoint.py --profile OUT_DIR          (a torch.profiler run of its own: configs 2 and 4)

For the luma and chroma tables of bench.py's configs, float32 planes: a batch of planes larger than the 126 MB L2 (source
plus output) goes through jinc_resize_planes_device (forward) and jinc_resize_adjoint_planes_device (adjoint), each timed
with CUDA events over a window of at least `seconds`, forward and adjoint alternated in `pairs` pairs.  Rates are source
samples per second and the FMA fraction: FLOP = 2 * fs^2 per output (bench.py's roofline count) over the FP32-FMA peak
that bench.py measures (avisynth-jincresize_b200/fma_peak).  One JSON line per table, then one line for a torch-level
training step (forward + backward through autograd) of a 32 x 3 x 512^2 -> 1024^2 batch in float16 and float32, and one
line with the card's name, power limit and maximum SM clock.  A GPU is required: there is no CPU fallback."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "avisynth-jincresize_b200"))

import bench  # noqa: E402  (the workloads and the FMA peak)
from jinc_b200 import capi  # noqa: E402
from jinc_b200.tensor import _stream, jinc_resize  # noqa: E402
from oracle import cpu as oc  # noqa: E402  (the per-table geometry, chroma siting included)

L2_BYTES = 126e6


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def tables(ctx, cfg):
    fmt, kw = cfg["fmt"], cfg["kw"]
    sw, sh = fmt.subsampling
    pp = oc.plane_params(cfg["w"], cfg["h"], cfg["tw"], cfg["th"], src_left=kw.get("src_left", 0.0),
                         src_top=kw.get("src_top", 0.0), quant_x=kw.get("quant_x", 256), quant_y=kw.get("quant_y", 256),
                         tap=cfg["tap"], sub_w=sw if len(fmt.planes) > 1 else 0, sub_h=sh if len(fmt.planes) > 1 else 0,
                         cplace=kw.get("cplace", "mpeg2"))
    for k, p in enumerate(pp):
        yield ("luma" if k == 0 else "chroma"), capi.Table(
            ctx, quant_x=p.quant_x, quant_y=p.quant_y, src_w=p.src_w, src_h=p.src_h, dst_w=p.dst_w, dst_h=p.dst_h,
            radius=capi.radius_for_tap(cfg["tap"]), blur=float(np.float32(kw.get("blur", 0.0))), crop_left=p.crop_left,
            crop_top=p.crop_top, crop_w=p.crop_w, crop_h=p.crop_h), p


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


def bench_table(name, tab, p, fs, args, peak_tflops):
    import torch

    H, W, h, w = p.src_h, p.src_w, p.dst_h, p.dst_w
    n = int(np.ceil(2 * L2_BYTES / (4 * (H * W + h * w))))
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        src = torch.rand((n, H, W), device="cuda")
        pitch = (w + 3) // 4 * 4
        dst = torch.empty((n, h, pitch), device="cuda")
        g = torch.randn((n, h, w), device="cuda")
        gs = torch.empty((n, H, W), device="cuda")
    torch.cuda.synchronize()
    st = stream.cuda_stream
    fwd = lambda: tab.resize_planes_device(4, 0.0, n, src.data_ptr(), W * 4, H * W * 4, dst.data_ptr(), pitch * 4, h * pitch * 4, st)
    adj = lambda: tab.adjoint_planes_device(n, g.data_ptr(), w * 4, h * w * 4, gs.data_ptr(), W * 4, H * W * 4, st)
    f_ms, a_ms, steps = [], [], []
    for _ in range(args.pairs):
        t, s1 = timed(fwd, args.seconds, stream)
        f_ms.append(t)
        t, s2 = timed(adj, args.seconds, stream)
        a_ms.append(t)
        steps.append((s1, s2))
    flop = 2.0 * fs * fs * h * w * n
    rate = lambda ms: flop / (ms * 1e-3) / 1e12
    f, a = statistics.median(f_ms), statistics.median(a_ms)
    return {"table": name, "src": [W, H], "dst": [w, h], "fs": fs, "info_path": capi.PATH_NAMES.get(tab.info.fast_path),
            "planes": n, "batch_mb": round(4 * n * (H * W + h * w) / 1e6, 1), "steps": steps,
            "forward_ms": [round(v, 4) for v in f_ms], "adjoint_ms": [round(v, 4) for v in a_ms],
            "forward_src_gsamples_s": round(n * H * W / (f * 1e-3) / 1e9, 2),
            "adjoint_src_gsamples_s": round(n * H * W / (a * 1e-3) / 1e9, 2),
            "forward_fma_frac": round(rate(f) / peak_tflops, 3), "adjoint_fma_frac": round(rate(a) / peak_tflops, 3),
            "adjoint_over_forward_time": round(a / f, 3)}


def torch_step(dtype, steps):
    import torch

    x = torch.rand((32, 3, 512, 512), device="cuda").to(dtype).requires_grad_()
    g = torch.randn((32, 3, 1024, 1024), device="cuda").to(dtype)

    def step():
        x.grad = None
        y = jinc_resize(x, 1024, 1024)
        (y * g).sum().backward()

    for _ in range(3):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    e1.synchronize()
    return round(e0.elapsed_time(e1) / steps, 3)


def profile(out_dir):
    import torch
    from torch.profiler import ProfilerActivity

    ctx = capi.Context(0)
    os.makedirs(out_dir, exist_ok=True)
    lines = []
    for cid in (2, 4):
        cfg = bench.CONFIGS[cid]
        for name, tab, p in tables(ctx, cfg):
            H, W, h, w = p.src_h, p.src_w, p.dst_h, p.dst_w
            g = torch.randn((2, h, w), device="cuda")
            gs = torch.empty((2, H, W), device="cuda")
            st = _stream(torch.device("cuda", 0))
            tab.adjoint_planes_device(2, g.data_ptr(), w * 4, h * w * 4, gs.data_ptr(), W * 4, H * W * 4, st)
            torch.cuda.synchronize()
            with torch.profiler.profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    tab.adjoint_planes_device(2, g.data_ptr(), w * 4, h * w * 4, gs.data_ptr(), W * 4, H * W * 4, st)
                torch.cuda.synchronize()
            lines.append(f"== config {cid} {name} ({W}x{H} -> {w}x{h}, fs {tab.info.filter_size}), 3 calls of 2 planes")
            lines.append(prof.key_averages().table(sort_by="cuda_time_total", row_limit=10))
            tab.close()
    text = "\n".join(lines)
    open(os.path.join(out_dir, "r06_adjoint_profile.txt"), "w").write(text)
    print(text)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="*", default=[1, 2, 3, 4, 5, 6])
    ap.add_argument("--pairs", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--torch-steps", type=int, default=20)
    ap.add_argument("--profile", metavar="OUT_DIR")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available() or capi.device_count() < 1:
        sys.exit("bench_adjoint.py: no CUDA device (there is no CPU fallback)")
    if args.profile:
        profile(args.profile)
        return
    print(json.dumps({"card": card()}), flush=True)
    peak, _ = bench.fma_peak_tflops()
    ctx = capi.Context(0)
    for cid in args.configs:
        cfg = bench.CONFIGS[cid]
        for name, tab, p in tables(ctx, cfg):
            rec = bench_table(name, tab, p, tab.info.filter_size, args, peak)
            rec["config"] = cid
            rec["fma_peak_tflops"] = peak
            print(json.dumps(rec), flush=True)
            tab.close()
    rec = {"torch_step": "32x3x512^2 -> 1024^2, forward + backward", "steps": args.torch_steps}
    for dt in ("float32", "float16"):
        rec[f"{dt}_ms"] = torch_step(getattr(torch, dt), args.torch_steps)
    print(json.dumps(rec), flush=True)
    print(json.dumps({"card_after": card()}), flush=True)


if __name__ == "__main__":
    main()
