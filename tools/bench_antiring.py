#!/usr/bin/env python
"""tools/bench_antiring.py -- cost of the anti-ringing pass (antiring_pass) on bench.py's geometries.

    python tools/bench_antiring.py [--configs 1 2 3 4 5] [--pairs 3] [--steps K] [--e2e-steps K] [--warmup W]

For each config (bench.py's format, geometry, tap, crop and blur) prints one JSON line:
  kernel   jinc_filter_process_device_batch on device-resident frames (CUDA events around `steps` launches per table) at
           strength 0 and strength 1, alternated in `pairs` pairs; every batch is at least twice the 126 MB L2.
           Gpixel/s counts output luma pixels; delta_ms is what the pass adds to a batch
  pass     jinc_antiring_plane_device alone over the same planes, one call per plane (CUDA events around `steps` sweeps),
           at strength 1.  bytes = the algorithmic traffic: every output sample read and written once, and each source
           sample of the anchor rows and columns read once.  GB/s and the fraction of 7.7 TB/s (the data-sheet HBM3e
           bandwidth of one B200, not a measured peak) are given for the per-call timing and for delta_ms above
  e2e      jinc_filter_submit / jinc_filter_wait on caller-pinned host frames, `inflight` frames in flight: frames/s at
           strength 0 and 1, alternated in the same pairs
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

import bench  # noqa: E402  (the workloads)
from jinc_b200 import capi  # noqa: E402
from oracle import cpu as oc  # noqa: E402

L2_BYTES = 126e6
HBM_DATASHEET_BYTES_S = 7.7e12


def make_filter(cfg, slots: int):
    fmt, kw = cfg["fmt"], cfg["kw"]
    sw, sh = fmt.subsampling
    return capi.Filter(src_w=cfg["w"], src_h=cfg["h"], target_w=cfg["tw"], target_h=cfg["th"], n_planes=len(fmt.planes),
                       sample_bytes=np.dtype(fmt.dtype).itemsize, bits=fmt.bits, sub_w=sw, sub_h=sh,
                       src_left=kw.get("src_left", 0.0), src_top=kw.get("src_top", 0.0), quant_x=kw.get("quant_x", 256),
                       quant_y=kw.get("quant_y", 256), tap=cfg["tap"], blur=kw.get("blur", 0.0),
                       cplace=kw.get("cplace", "mpeg2"), devices=[0], slots_per_device=slots)


def frame(cfg, seed: int):
    fmt = cfg["fmt"]
    rng = np.random.default_rng(0x41520000 ^ seed)
    out = []
    for i in range(len(fmt.planes)):
        shape = fmt.plane_shape(i, cfg["w"], cfg["h"])
        if fmt.bits == 32:
            out.append(rng.random(shape, dtype=np.float32))
        else:
            out.append(rng.integers(0, fmt.peak + 1, shape).astype(fmt.dtype))
    return out


def anchor_count(pos, n):
    f = np.floor(pos.astype(np.float64)).astype(np.int64)
    return len(np.union1d(np.clip(f, 0, n - 1), np.clip(f + 1, 0, n - 1)))


def pass_bytes(flt, sb):
    """Algorithmic bytes of the pass over one frame: output read + write, each anchor source sample read once."""
    total = 0
    for i, (sshape, dshape) in enumerate(flt.plane_shapes()):
        t = flt.table(1 if (flt.num_tables > 1 and i in (1, 2)) else 0)
        nx = anchor_count(t.axis(0)[3], sshape[1])
        ny = anchor_count(t.axis(1)[3], sshape[0])
        total += (2 * dshape[0] * dshape[1] + nx * ny) * sb
    return total


def measure(cid: int, args) -> dict:
    import torch

    cfg = bench.CONFIGS[cid]
    fmt = cfg["fmt"]
    sb = np.dtype(fmt.dtype).itemsize
    frame_bytes = sum((fmt.plane_shape(i, cfg["w"], cfg["h"])[0] * fmt.plane_shape(i, cfg["w"], cfg["h"])[1] +
                       fmt.plane_shape(i, cfg["tw"], cfg["th"])[0] * fmt.plane_shape(i, cfg["tw"], cfg["th"])[1]) * sb
                      for i in range(len(fmt.planes)))
    F = max(cfg["frames"], math.ceil(2 * L2_BYTES / frame_bytes))
    frames_np = [frame(cfg, f) for f in range(F)]
    flt = make_filter(cfg, args.inflight)
    shapes = flt.plane_shapes()
    tdt = {1: torch.uint8, 2: torch.int16, 4: torch.float32}[sb]  # 16-bit samples travel as int16 bit patterns
    view = {1: np.uint8, 2: np.int16, 4: np.float32}[sb]
    keep, dev, planes = [], [], []
    for planes_np in frames_np:
        fr = capi.Frame()
        for i, ((sshape, dshape), p) in enumerate(zip(shapes, planes_np)):
            sp = (sshape[1] * sb + 255) // 256 * 256 // sb
            dp = (dshape[1] * sb + 255) // 256 * 256 // sb
            s = torch.zeros((sshape[0], sp), dtype=tdt, device="cuda")
            s[:, : sshape[1]].copy_(torch.from_numpy(p.view(view)))
            d = torch.zeros((dshape[0], dp), dtype=tdt, device="cuda")
            fr.src[i], fr.src_pitch[i] = s.data_ptr(), sp * sb
            fr.dst[i], fr.dst_pitch[i] = d.data_ptr(), dp * sb
            keep += [s, d]
            planes.append((1 if (flt.num_tables > 1 and i in (1, 2)) else 0, s.data_ptr(), sp * sb, d.data_ptr(), dp * sb))
        dev.append(fr)
    frames = (capi.Frame * F)(*dev)
    stream = torch.cuda.Stream()
    st = stream.cuda_stream
    torch.cuda.synchronize()

    def batch():
        for k in range(flt.num_tables):
            flt.process_device_batch(frames, 0, 1 << k, 3, st)

    def timed(fn, steps):
        for _ in range(args.warmup):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / steps

    # tables of the filter's own geometry for the per-plane calls (same parameters, own context)
    ctx = capi.Context(0)
    pp = oc.plane_params(cfg["w"], cfg["h"], cfg["tw"], cfg["th"], src_left=cfg["kw"].get("src_left", 0.0),
                         src_top=cfg["kw"].get("src_top", 0.0), quant_x=cfg["kw"].get("quant_x", 256),
                         quant_y=cfg["kw"].get("quant_y", 256), tap=cfg["tap"], sub_w=fmt.subsampling[0],
                         sub_h=fmt.subsampling[1], cplace=cfg["kw"].get("cplace", "mpeg2"))
    tables = [capi.Table(ctx, quant_x=tp.quant_x, quant_y=tp.quant_y, src_w=tp.src_w, src_h=tp.src_h, dst_w=tp.dst_w,
                         dst_h=tp.dst_h, radius=tp.radius, blur=float(np.float32(cfg["kw"].get("blur", 0.0))),
                         crop_left=tp.crop_left, crop_top=tp.crop_top, crop_w=tp.crop_w, crop_h=tp.crop_h) for tp in pp]
    for k, t in enumerate(tables):
        assert np.array_equal(t.axis(0)[3], flt.table(k).axis(0)[3]) and np.array_equal(t.axis(1)[3], flt.table(k).axis(1)[3])
    L = capi.lib()

    def sweep():
        for k, sp_, spitch, dp_, dpitch in planes:
            rc = L.jinc_antiring_plane_device(ctx.handle, tables[k].handle, sb, 1.0, sp_, spitch, dp_, dpitch, st)
            assert rc == 0, L.jinc_last_error()

    # pinned host frames for the end-to-end leg
    host = []
    for planes_np in frames_np[: max(args.inflight * 2, 4)]:
        src = [torch.from_numpy(p.view(view)).pin_memory() for p in planes_np]
        dst = [torch.zeros(dshape, dtype=tdt).pin_memory() for _, dshape in shapes]
        host.append((src, dst, flt._frame([t.numpy().view(fmt.dtype) for t in src], [t.numpy().view(fmt.dtype) for t in dst])))

    def e2e(steps):
        def run(n):
            tickets = []
            for _ in range(n):
                for _, _, fr in host:
                    if len(tickets) >= args.inflight:
                        flt.wait(tickets.pop(0))
                    tickets.append(flt.submit_raw(fr))
            for t in tickets:
                flt.wait(t)

        run(1)
        t0 = time.perf_counter()
        run(steps)
        return steps * len(host) / (time.perf_counter() - t0)

    kern = {0.0: [], 1.0: []}
    fps = {0.0: [], 1.0: []}
    alone = []
    launches = {}
    for _ in range(args.pairs):
        for s in (0.0, 1.0):
            flt.set_antiring(s)
            l0 = flt.kernel_launches
            kern[s].append(timed(batch, args.steps))
            launches[s] = (flt.kernel_launches - l0) // (args.steps + args.warmup)
        alone.append(timed(sweep, args.steps))
    for _ in range(args.pairs):
        for s in (0.0, 1.0):
            flt.set_antiring(s)
            fps[s].append(e2e(args.e2e_steps))

    bytes_batch = pass_bytes(flt, sb) * F
    gpix = cfg["tw"] * cfg["th"] * F / 1e9
    k0, k1, a = statistics.median(kern[0.0]), statistics.median(kern[1.0]), statistics.median(alone)
    delta = k1 - k0
    infos = [flt.table(k).info for k in range(flt.num_tables)]
    for t in tables:
        t.close()
    ctx.close()
    flt.close()
    del keep
    torch.cuda.empty_cache()

    def rate(ms):
        return {"gb_s": round(bytes_batch / (ms * 1e-3) / 1e9, 1),
                "frac_of_7p7_tb_s_datasheet": round(bytes_batch / (ms * 1e-3) / HBM_DATASHEET_BYTES_S, 3)} if ms > 0 else None

    return {"config": cid, "workload": cfg["name"], "frames_per_batch": F, "batch_mb": round(F * frame_bytes / 1e6, 1),
            "kernel_paths": [bench.KERNEL_NAMES.get(i.fast_path, "resample_strips") for i in infos],
            "steps": args.steps, "pairs": args.pairs,
            "kernel": {"s0_ms": [round(v, 4) for v in kern[0.0]], "s1_ms": [round(v, 4) for v in kern[1.0]],
                       "s0_gpixel_s": round(gpix / (k0 * 1e-3), 2), "s1_gpixel_s": round(gpix / (k1 * 1e-3), 2),
                       "launches_per_batch": {"s0": launches[0.0], "s1": launches[1.0]},
                       "delta_ms": round(delta, 4), "delta_frac_of_s0": round(delta / k0, 4), "delta_rate": rate(delta)},
            "pass": {"api": "jinc_antiring_plane_device, one call per plane, strength 1", "calls_per_sweep": len(planes),
                     "ms_per_sweep": [round(v, 4) for v in alone], "bytes_per_sweep": bytes_batch, **rate(a)},
            "e2e": {"api": "jinc_filter_submit/jinc_filter_wait, caller-pinned host frames, %d in flight" % args.inflight,
                    "frames": len(host), "steps": args.e2e_steps, "s0_fps": [round(v, 2) for v in fps[0.0]],
                    "s1_fps": [round(v, 2) for v in fps[1.0]],
                    "median_fps_ratio_s1_over_s0": round(statistics.median(fps[1.0]) / statistics.median(fps[0.0]), 4)}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[1, 2, 3, 4, 5])
    ap.add_argument("--pairs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--inflight", type=int, default=3)
    args = ap.parse_args()
    import torch

    if capi.device_count() < 1 or not torch.cuda.is_available():
        sys.exit("bench_antiring: no CUDA device (there is no CPU fallback)")
    name = torch.cuda.get_device_name(0)
    for cid in args.configs:
        line = measure(cid, args)
        line["device"] = name
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
