#!/usr/bin/env python
"""bench.py -- throughput of the EWA-Jinc resampling hot path on B200, next to the reference's CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 1..9] [--impl b200|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of `frames_per_step` distinct synthetic frames of the
chosen BASELINE.json config (default: configs[1], 1080p YUV420P8 -> 2160p Jinc36Resize cplace=MPEG2).
Prints ONE JSON line (rank 0):
  value        output Mpixel/s, kernels only, inputs resident in HBM (CUDA events, max over ranks); a sampled row band
               of the timed launches' output is compared with the oracle outside the timed region ("verified")
  e2e          the same metric through the reference-facing call: the AviSynth+ plugin's get_frame under the mini-host,
               PAGEABLE host frames in and out, H2D + kernels + D2H inside the timed region
  e2e_pinned   the C ABI's host-frame call (jinc_filter_submit/wait) with caller-pinned planes
  both carry   ceiling_gbs / frac: a pure-copy run of the same buffers and sizes with no kernels, measured in the
               same process right before (every rank at once under torchrun), and the achieved share of it
  roofline     dominant kernel (luma-table launch) against the FP32-FMA roofline measured on this box
               (avisynth-jincresize_b200/fma_peak), plus roofline_hbm against MEASURED_PEAKS.json
  all_configs  kernel-only value, roofline fraction, end-to-end value and table construction time of the other
               BASELINE configs
  row_bands    latency of ONE 8K frame cut into row bands over the N GPUs of the run (jinc_filter_process_bands)
  cpu_baseline the UNMODIFIED reference (oracle/_ref) on this box's host cores, AVX2 and AVX-512 paths, one thread and
               all threads, on a bounded sample of the same workload, plus its filter construction time
`--impl reference` times only that CPU reference and prints the same line shape with "impl": "reference".
`--dump-outputs DIR` writes what the last kernel-only step computed as DIR/plane<i>.npy (float32, see dump_outputs); the
inputs are seeded, so two builds run with the same arguments can be compared output for output.
Under torchrun (N>1) every rank drives its own GPU with the same per-GPU batch (weak scaling; frames are
independent, so there is no collective on the data path -- NCCL is used for the barrier and the max only).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (which may be read-only)
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "avisynth-jincresize_b200"))

from minihost import avs_host as ah  # noqa: E402
from oracle import ref as oref  # noqa: E402
from jinc_b200 import paths  # noqa: E402

METRIC = "output Mpixel/s"

CONFIGS = {
    1: dict(name="640x360 YV12 -> 1280x720 Jinc36Resize (tap=3)", fmt=ah.YV12, w=640, h=360, tw=1280, th=720,
            fn="Jinc36Resize", kw=dict(), tap=3, frames=128),
    2: dict(name="1920x1080 YUV420P8 -> 3840x2160 Jinc36Resize cplace=MPEG2", fmt=ah.YUV420P8, w=1920, h=1080, tw=3840,
            th=2160, fn="Jinc36Resize", kw=dict(cplace="MPEG2"), tap=3, frames=24),
    3: dict(name="1920x1080 YUV444P16 -> 3840x2160 Jinc64Resize src_left=10.3 src_top=6.7 quant=256", fmt=ah.YUV444P16,
            w=1920, h=1080, tw=3840, th=2160, fn="Jinc64Resize",
            kw=dict(src_left=10.3, src_top=6.7, quant_x=256, quant_y=256), tap=4, frames=8),
    4: dict(name="3840x2160 RGBPS -> 7680x4320 Jinc256Resize (tap=8)", fmt=ah.RGBPS, w=3840, h=2160, tw=7680, th=4320,
            fn="Jinc256Resize", kw=dict(), tap=8, frames=2),
    5: dict(name="7680x4320 YUV420P10 -> 1920x1080 JincResize tap=6 blur=0.9", fmt=ah.YUV420P10, w=7680, h=4320,
            tw=1920, th=1080, fn="JincResize", kw=dict(tap=6, blur=0.9), tap=6, frames=4),
    # not BASELINE configs: the "next" row of SURVEY.md 8(f), ratios that are not exact 2x / 1/n
    6: dict(name="1280x720 YUV420P8 -> 1920x1080 Jinc36Resize (1.5x)", fmt=ah.YUV420P8, w=1280, h=720, tw=1920,
            th=1080, fn="Jinc36Resize", kw=dict(), tap=3, frames=48),
    7: dict(name="1920x1080 YUV420P8 -> 1280x720 Jinc36Resize (2:3 downscale)", fmt=ah.YUV420P8, w=1920, h=1080,
            tw=1280, th=720, fn="Jinc36Resize", kw=dict(), tap=3, frames=48),
    9: dict(name="1920x1080 YUV420P8 -> 2560x1440 Jinc36Resize (4:3 upscale)", fmt=ah.YUV420P8, w=1920, h=1080,
            tw=2560, th=1440, fn="Jinc36Resize", kw=dict(), tap=3, frames=32),
    8: dict(name="1920x1080 YUV444P16 -> 2500x1400 Jinc64Resize (irregular ratio, many phases)", fmt=ah.YUV444P16, w=1920, h=1080,
            tw=2500, th=1400, fn="Jinc64Resize", kw=dict(), tap=4, frames=12),
}

KERNEL_NAMES = {1: "resample_up2x", 2: "resample_down", 3: "resample_down (periodic passes in one launch)",
                4: "resample_cells (piecewise-periodic ratio)"}


def synth_frame(fmt: ah.Format, w: int, h: int, seed: int):
    """Seeded uniform noise over the full sample range (float chroma in [-0.5, 0.5))."""
    rng = np.random.default_rng(0x4A494E43 ^ seed)
    planes = []
    for i in range(len(fmt.planes)):
        ph, pw = fmt.plane_shape(i, w, h)
        if fmt.bits == 32:
            a = rng.random((ph, pw), dtype=np.float32)
            if i in (1, 2) and fmt.family not in ("rgbp", "rgbap"):
                a -= 0.5
        else:
            a = rng.integers(0, fmt.peak + 1, (ph, pw), dtype=np.uint16 if fmt.bits > 8 else np.uint8)
        planes.append(np.ascontiguousarray(a.astype(fmt.dtype)))
    return planes


def filter_size_of(cfg) -> int:
    """filter_size of the luma table (src/JincResize.cpp:349-357), computed on the host for the config record."""
    from oracle import cpu as oc

    radius = oc.radius_for_tap(cfg["tap"])
    sup = 0.0
    for src, dst in ((cfg["w"], cfg["tw"]), (cfg["h"], cfg["th"])):
        sup = max(sup, float(np.float32(radius / min(dst / src, 1.0))))
    return int(math.ceil(sup * 2.0))


def config_record(cfg, config_id: int, byts: float, parts: int = 3) -> dict:
    """The `config` object of the JSON line: identical for the GPU arm and the reference arm of one workload."""
    fmt, F = cfg["fmt"], cfg["frames"]
    rec = {"workload": cfg["name"], "config_id": config_id, "frames_per_step": F,
           "sample_type": f"{fmt.family}{fmt.bits}", "filter_size": filter_size_of(cfg),
           "l2": "inputs larger than L2: every step walks %d distinct frames (%.0f MB of planes)" % (F, F * byts / 1e6),
           "partition": "frame-parallel, one process per GPU, no collective",
           "host_affinity": "ranks bind to the CPUs NVML reports as local to their GPU"}
    if parts != 3:
        rec.update(parts=parts, INVALID="diagnostic run, part of the frame skipped")
    return rec


def algorithmic_work(cfg, fs_luma, fs_chroma):
    """FLOP = 2*fs^2*output samples; bytes = (src + dst samples)*sizeof(T) per plane (SURVEY.md 8d)."""
    fmt = cfg["fmt"]
    sb = np.dtype(fmt.dtype).itemsize
    flop = byts = 0.0
    luma = dict(flop=0.0, bytes=0.0)
    for i in range(len(fmt.planes)):
        sh = fmt.plane_shape(i, cfg["w"], cfg["h"])
        dh = fmt.plane_shape(i, cfg["tw"], cfg["th"])
        chroma_tbl = i in (1, 2) and fmt.subsampling != (0, 0)
        fs = fs_chroma if chroma_tbl else fs_luma
        f = 2.0 * fs * fs * dh[0] * dh[1]
        b = (sh[0] * sh[1] + dh[0] * dh[1]) * sb
        flop += f
        byts += b
        if not chroma_tbl:
            luma["flop"] += f
            luma["bytes"] += b
    return flop, byts, luma


def frame_bytes(cfg) -> float:
    return algorithmic_work(cfg, 1, 1)[1]


class ClockSampler:
    """nvidia-smi clocks/throttle reasons while the timed region runs (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def measured_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs"), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(config_id: int, frames: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel's launch, from the committed `ncu --set full`
    capture of the same bench command (profiles/ncu_traffic.json); None when no capture exists for this workload."""
    try:
        rec = json.load(open(os.path.join(REPO, "profiles", "ncu_traffic.json"))).get(str(config_id))
        if rec and rec.get("frames_per_launch") == frames:
            return float(rec["dram_bytes_per_launch"])
    except Exception:
        pass
    return None


_FMA_PEAK = None


def fma_peak_tflops():
    """FP32 FMA-pipe peak measured on this GPU by the repo's own microbenchmark (best FFMA variant)."""
    global _FMA_PEAK
    if _FMA_PEAK is None:
        tool = paths.fma_peak_tool()
        try:
            out = subprocess.run([tool, "8000"], capture_output=True, text=True, timeout=120).stdout
            best = max(json.loads(l)["tflops"] for l in out.splitlines() if l.startswith("{"))
            _FMA_PEAK = (best, "measured (fma_peak: FFMA reg-reg, 148 SMs)")
        except Exception:
            _FMA_PEAK = (148 * 128 * 2 * 1.965e9 / 1e12, "nominal (148 SM x 128 lanes x 2 x 1.965 GHz)")
    return _FMA_PEAK


# ------------------------------------------------------------------------------------------ CPU reference

def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


OPT_NAMES = {2: "avx2", 3: "avx512"}


def run_reference(cfg, steps: int, warmup: int, budget_s: float, exact_steps: bool = False):
    """Times the reference's own CPU implementation through its plugin API under the mini-host.  For each SIMD path the
    host CPU has (opt=2 AVX2 -- what the reference picks by default, src/JincResize.cpp:898 -- and opt=3 AVX-512, :897):
    filter construction (LUT + generate_coeff_table_c, :795-866), single-thread frames, then frame-parallel get_frame
    with one host thread per core (what AviSynth's Prefetch does for this MT_MULTI_INSTANCE filter).  `value` is the
    faster path's all-thread figure.  The step count is cut to fit `budget_s` unless exact_steps is set.  Falls back to the
    scalar oracle port only if the prebuilt reference is absent."""
    fmt, w, h, tw, th = cfg["fmt"], cfg["w"], cfg["h"], cfg["tw"], cfg["th"]
    threads = host_threads()
    mpix = tw * th / 1e6
    F = cfg["frames"]
    if os.path.exists(oref.REF_PLUGIN):
        env = ah.Env()
        env.load_plugin(oref.REF_PLUGIN)
        try:
            cpu = set(next(l for l in open("/proc/cpuinfo") if l.startswith("flags")).split())
        except Exception:
            cpu = set()
        opts = [o for o, name in ((2, "avx2"), (3, "avx512f")) if name in cpu] or [-1]
        distinct = min(F, 4)
        src = env.source(fmt, w, h, [synth_frame(fmt, w, h, s) for s in range(distinct)], num_frames=1 << 20)
        per_opt = budget_s / len(opts)
        sub, best = {}, None
        for opt in opts:
            t0 = time.perf_counter()
            clip = env.invoke(cfg["fn"] if opt < 0 else "JincResize", src, tw, th,
                              **(cfg["kw"] if opt < 0 else dict(cfg["kw"], tap=cfg["tap"], opt=opt)))
            construct_s = time.perf_counter() - t0
            t1 = clip.pull(0, 1, 1)  # single-thread probe: sizes the bounded sample
            n1 = max(1, min(4, int(0.15 * per_opt / max(t1, 1e-6))))
            t1 = clip.pull(1, n1, 1) / n1
            est = t1 * F / max(1, min(threads, F))
            n_steps, n_warm = max(1, steps), warmup
            if not exact_steps:
                while n_steps > 1 and est * (n_steps + warmup) > 0.7 * per_opt:
                    n_steps -= 1
                n_warm = warmup if est * (n_steps + warmup) <= 0.7 * per_opt else 0
            f0 = 8
            for _ in range(n_warm):
                clip.pull(f0, F, threads)
                f0 += F
            tt = time.perf_counter()
            for _ in range(n_steps):
                clip.pull(f0, F, threads)
                f0 += F
            dt = time.perf_counter() - tt
            rec = dict(value=n_steps * F * mpix / dt, single_thread_value=mpix / t1, construct_ms=construct_s * 1e3,
                       ms_per_step=dt / n_steps * 1e3, steps=n_steps, warmup=n_warm, threads=threads)
            sub[OPT_NAMES.get(opt, "default")] = rec
            if best is None or rec["value"] > sub[best]["value"]:
                best = OPT_NAMES.get(opt, "default")
            clip.release()
        src.release()
        b = sub[best]
        return dict(value=b["value"], unit=METRIC, cores=threads, kind="reference",
                    sample=f"{b['steps']} steps x {F} frames per SIMD path, frame-parallel on {threads} host threads; value = the faster "
                           f"path ({best}); the reference's default on this CPU is avx2",
                    ms_per_step=b["ms_per_step"], steps=b["steps"], warmup=b["warmup"], frames_per_step=F,
                    single_thread_value=b["single_thread_value"], construct_ms=b["construct_ms"], best_path=best,
                    **{k: v for k, v in sub.items()})
    # scalar port (oracle) -- only when oracle/_ref did not travel
    from oracle import cpu as oc

    planes = synth_frame(fmt, w, h, 0)
    sw, sh = fmt.subsampling
    pp = oc.plane_params(w, h, tw, th, tap=cfg["tap"], sub_w=sw, sub_h=sh, **{k: v for k, v in cfg["kw"].items() if k not in ("tap", "blur")})
    lut = oc.make_lut(cfg["tap"], cfg["kw"].get("blur", 0.0))
    t0 = time.perf_counter()
    t = oc.Table(pp[0], lut)
    construct_s = time.perf_counter() - t0
    rows = max(8, th // 64)
    peak = float(fmt.peak) if fmt.bits < 32 else 0.0
    for _ in range(warmup):
        t.resize(planes[0], peak, rows=(th // 2, th // 2 + rows))
    t0 = time.perf_counter()
    for _ in range(steps):
        t.resize(planes[0], peak, rows=(th // 2, th // 2 + rows))
    dt = time.perf_counter() - t0
    value = steps * (rows * tw / 1e6) / dt
    return dict(value=value, unit=METRIC, cores=1, kind="port", sample=f"{rows} luma rows of one frame, scalar oracle port",
                ms_per_step=dt / steps * 1e3, steps=steps, warmup=warmup, frames_per_step=rows / th, construct_ms=construct_s * 1e3)


def bind_to_gpu_numa(device_index: int):
    """One process per GPU: pin this process to the CPUs NVML reports as local to its GPU BEFORE any pinned host buffer is
    allocated, so the frames it DMAs live on the GPU's own NUMA node.  Returns the number of CPUs bound to, or None when
    NVML gives no answer."""
    try:
        import pynvml
        import torch

        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(device_index)
        bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * i + b for i, wd in enumerate(mask) for b in range(64) if (wd >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


# ------------------------------------------------------------------------------------------ GPU arm

class Dist:
    """barrier / max-over-ranks; single-process when WORLD_SIZE is 1."""

    def __init__(self):
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    def init(self):
        import torch
        import torch.distributed as dist

        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))

    def barrier(self):
        import torch
        import torch.distributed as dist

        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max(self, *vals):
        import torch
        import torch.distributed as dist

        if self.world == 1:
            return [float(v) for v in vals]
        t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def sum(self, *vals):
        import torch
        import torch.distributed as dist

        if self.world == 1:
            return [float(v) for v in vals]
        t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
        dist.all_reduce(t)
        return [float(v) for v in t]

    def close(self):
        import torch.distributed as dist

        if self.world > 1:
            dist.destroy_process_group()


def make_filter(cfg, devices, slots=0, flags=0):
    from jinc_b200 import capi

    fmt, kw = cfg["fmt"], cfg["kw"]
    sw, sh = fmt.subsampling
    return capi.Filter(src_w=cfg["w"], src_h=cfg["h"], target_w=cfg["tw"], target_h=cfg["th"], n_planes=len(fmt.planes),
                       sample_bytes=np.dtype(fmt.dtype).itemsize, bits=fmt.bits, sub_w=sw, sub_h=sh,
                       src_left=kw.get("src_left", 0.0), src_top=kw.get("src_top", 0.0), quant_x=kw.get("quant_x", 256),
                       quant_y=kw.get("quant_y", 256), tap=cfg["tap"], blur=kw.get("blur", 0.0), cplace=kw.get("cplace", "mpeg2"),
                       devices=list(devices), slots_per_device=slots, flags=flags)


def capture_output_rows(cfg, planes_by_frame, dst_by_frame, shapes):
    """Right after the kernel-only leg: rows of its OUTPUT (first and last frame of the batch: top, a tile seam in the
    middle, bottom of every plane) are downloaded; verify_against_oracle compares them once every timed leg is done."""
    cap = []
    for fi, (planes, dsts) in enumerate(zip(planes_by_frame, dst_by_frame)):
        for i, pl in enumerate(planes):
            H, W = shapes[i][1]
            for (y0, y1) in ((0, 3), (H // 2 - 1, H // 2 + 2), (H - 3, H)):
                cap.append((fi, i, y0, y1, pl, dsts[i][y0:y1, :W].cpu().numpy()))
    return cap


def verify_against_oracle(cfg, captured):
    """Outside the timed regions: the captured rows of the kernel-only leg's output against the CPU oracle (parity bar)."""
    from oracle import cpu as oc

    fmt, kw = cfg["fmt"], cfg["kw"]
    sw, sh = fmt.subsampling
    pp = oc.plane_params(cfg["w"], cfg["h"], cfg["tw"], cfg["th"], src_left=kw.get("src_left", 0.0), src_top=kw.get("src_top", 0.0),
                         quant_x=kw.get("quant_x", 256), quant_y=kw.get("quant_y", 256), tap=cfg["tap"], sub_w=sw, sub_h=sh,
                         cplace=kw.get("cplace", "mpeg2"))
    lut = oc.make_lut(cfg["tap"], kw.get("blur", 0.0))
    tabs = [oc.Table(p, lut) for p in pp]
    peak = float(fmt.peak) if fmt.bits < 32 else 0.0
    worst, rows_checked = 0.0, 0
    for fi, i, y0, y1, pl, got in captured:
        t = tabs[1] if (len(tabs) > 1 and i in (1, 2)) else tabs[0]
        ref = t.resize(pl, peak, rows=(y0, y1))[y0:y1]
        if fmt.bits == 32:
            err = float((np.abs(got.astype(np.float64) - ref) / np.maximum(1.0, np.abs(ref))).max())
            ok = err <= 1e-5
        else:
            err = float(np.abs(got.astype(np.int64) - ref.astype(np.int64)).max())
            ok = err <= 1
        worst = max(worst, err)
        rows_checked += y1 - y0
        if not ok:
            raise SystemExit(f"bench.py: kernel-only output differs from the oracle (frame {fi} plane {i} rows {y0}-{y1}: {err})")
    for t in tabs:
        t.close()
    return {"ok": True, "against": "CPU oracle (oracle/jinc_oracle.c)", "frames_checked": len({c[0] for c in captured}),
            "rows_checked": rows_checked, "max_err": worst, "bar": "1e-5 relative" if fmt.bits == 32 else "1 LSB"}


DUMP_BYTES = 60 << 20  # below 64 MB with the .npy headers


def dump_outputs(out_dir, dst_by_frame, shapes):
    """The output planes of the batch as out_dir/plane<i>.npy, float32, one array row per output row (row y of frame f
    is batch row f * H + y).  When the batch holds more than DUMP_BYTES of float32 samples, every plane keeps the same
    fraction of its batch rows, drawn by a fixed-seed generator and kept in batch order, so that runs with the same
    arguments write the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    F = len(dst_by_frame)
    frac = min(1.0, DUMP_BYTES / (4 * F * sum(h * w for _, (h, w) in shapes)))
    rng = np.random.default_rng(0x4A494E43)
    for i, (_, (H, W)) in enumerate(shapes):
        n = F * H
        rows = np.arange(n) if frac == 1.0 else np.sort(rng.choice(n, int(n * frac), replace=False))
        out = np.empty((rows.size, W), np.float32)
        for f in range(F):
            sel = (rows >= f * H) & (rows < (f + 1) * H)
            if sel.any():
                out[sel] = dst_by_frame[f][i][:, :W].cpu().numpy()[rows[sel] - f * H]
        np.save(os.path.join(out_dir, f"plane{i}.npy"), out)


def copy_ceiling(D, host_src, host_dst, dev_src, dev_dst, inflight: int, steps: int):
    """The same pinned buffers and sizes as the end-to-end legs, moved with plain copies and NO kernels: per frame the
    source planes go H2D and the destination planes come D2H, `inflight` frames in flight on their own streams.  Every
    rank runs it at once.  Returns (seconds per step, bytes per step)."""
    import torch

    streams = [torch.cuda.Stream() for _ in range(inflight)]
    F = len(host_src)
    nbytes = sum(t.numel() * t.element_size() for f in range(F) for t in host_src[f] + host_dst[f])
    # tightly packed device planes, one set per stream: every plane moves as ONE linear transfer (the best a copy can do)
    tight_src = [[torch.empty_like(h, device="cuda") for h in host_src[0]] for _ in range(inflight)]
    tight_dst = [[torch.empty_like(h, device="cuda") for h in host_dst[0]] for _ in range(inflight)]
    del dev_src, dev_dst

    def step():
        for f in range(F):
            k = f % inflight
            with torch.cuda.stream(streams[k]):
                for h, d in zip(host_src[f], tight_src[k]):
                    d.copy_(h, non_blocking=True)
                for h, d in zip(host_dst[f], tight_dst[k]):
                    h.copy_(d, non_blocking=True)

    step()
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    D.barrier()
    return (time.perf_counter() - t0) / steps, nbytes


def run_plugin_leg(D, cfg, threads: int, steps: int, warm_steps: int):
    """The drop-in path itself: the AviSynth+ C plugin (libjincresize_b200.so) under the mini-host, PAGEABLE host frames
    in and out through get_frame, `threads` concurrent get_frame callers (what Prefetch(threads) does).  The plugin
    page-locks the host's recycled frame buffers as they come back (first sightings are staged through pinned mirrors)."""
    from jinc_b200 import capi

    fmt, w, h, tw, th, F = cfg["fmt"], cfg["w"], cfg["h"], cfg["tw"], cfg["th"], cfg["frames"]
    os.environ["JINCRESIZE_B200_DEVICES"] = str(D.local_rank)
    env = ah.Env()
    env.load_plugin(paths.b200_plugin())
    src = env.source(fmt, w, h, [synth_frame(fmt, w, h, 7000 + 10 * D.rank + s) for s in range(min(F, 4))], num_frames=1 << 20)
    t0 = time.perf_counter()
    clip = env.invoke(cfg["fn"], src, tw, th, **cfg["kw"])
    construct_s = time.perf_counter() - t0
    f0 = 0
    st0 = capi.host_buffer_stats()
    # warm-up: table build, slot allocation, first touch of the frame pool, and the page-locking of the pool's buffers
    # (done by a helper thread while the frames that found them pageable are staged) -- until a pull stages nothing
    for k in range(12):
        before = capi.host_buffer_stats()
        clip.pull(f0, max(F, 3 * threads), threads)
        f0 += max(F, 3 * threads)
        after = capi.host_buffer_stats()
        if k + 1 >= max(1, warm_steps) and after["staged_frames"] == before["staged_frames"] and after["registrations"] == before["registrations"]:
            break
    D.barrier()
    t0 = time.perf_counter()
    clip.pull(f0, steps * F, threads)  # the K steps back to back, as a host streams a clip: no barrier between steps
    D.barrier()
    dt = time.perf_counter() - t0
    st1 = capi.host_buffer_stats()
    clip.release()
    src.release()
    return dt, construct_s, {k: st1[k] - st0[k] for k in st1 if k != "registered_bytes"} | {"registered_bytes": st1["registered_bytes"]}


def measure_config(D, args, cfg, config_id: int, steps: int, warmup: int, full: bool):
    """All GPU legs of one workload on this rank's GPU.  full = False: kernel-only + plugin end-to-end only (all_configs)."""
    import torch

    from jinc_b200 import capi

    fmt, w, h, tw, th, F = cfg["fmt"], cfg["w"], cfg["h"], cfg["tw"], cfg["th"], cfg["frames"]
    sb = np.dtype(fmt.dtype).itemsize
    t0 = time.perf_counter()
    flt = make_filter(cfg, [D.local_rank], slots=args.inflight)
    filter_create_s = time.perf_counter() - t0
    infos = [flt.table(k).info for k in range(flt.num_tables)]
    fs_l, fs_c = infos[0].filter_size, infos[-1].filter_size
    tdtype = {1: torch.uint8, 2: torch.uint16, 4: torch.float32}[sb]

    def pitched(shape):  # device plane with a 256-byte aligned pitch, like a pitched allocation
        rows, cols = shape
        pitch_elems = ((cols * sb + 255) // 256 * 256) // sb
        return torch.zeros((rows, pitch_elems), dtype=tdtype, device="cuda")

    shapes = flt.plane_shapes()
    host_src, host_dst, dev_frames, dev_src, dev_dst, planes_np = [], [], [], [], [], []
    for f in range(F):
        planes = synth_frame(fmt, w, h, seed=1000 * D.rank + f)
        hs = [torch.from_numpy(p).pin_memory() for p in planes]
        hd = [torch.zeros(dshape, dtype=tdtype).pin_memory() for _, dshape in shapes]
        ds, dd = [], []
        fr = capi.Frame()
        for i, ((sshape, dshape), p) in enumerate(zip(shapes, hs)):
            s = pitched(sshape)
            s[:, : sshape[1]].copy_(p, non_blocking=True)
            d = pitched(dshape)
            ds.append(s)
            dd.append(d)
            fr.src[i], fr.src_pitch[i] = s.data_ptr(), s.stride(0) * sb
            fr.dst[i], fr.dst_pitch[i] = d.data_ptr(), d.stride(0) * sb
        host_src.append(hs)
        host_dst.append(hd)
        dev_frames.append(fr)
        dev_src.append(ds)
        dev_dst.append(dd)
        planes_np.append(planes if f in (0, F - 1) else None)
    torch.cuda.synchronize()

    stream = torch.cuda.Stream()
    sh_ = stream.cuda_stream
    n_tables = flt.num_tables
    frames_arr = (capi.Frame * F)(*dev_frames)

    def kernel_step(pairs=None):
        # one launch per coefficient table covers every frame of the batch: interior tiles + border strips together
        if pairs is not None:
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            flt.process_device_batch(frames_arr, 0, 1, args.parts, sh_)
            e1.record(stream)
            pairs.append((e0, e1))
        else:
            flt.process_device_batch(frames_arr, 0, 1, args.parts, sh_)
        if n_tables > 1:
            flt.process_device_batch(frames_arr, 0, 2, args.parts, sh_)

    # ---------------- kernel-only
    for _ in range(warmup):
        kernel_step()
    D.barrier()
    sampler = ClockSampler(D.local_rank) if (full and D.rank == 0) else None
    if sampler:
        sampler.start()
    launches0 = flt.kernel_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pairs = []
    ev0.record(stream)
    for _ in range(steps):
        kernel_step(pairs)
    ev1.record(stream)
    D.barrier()
    gpu_launches = flt.kernel_launches - launches0
    ms_total = ev0.elapsed_time(ev1)
    dom_ms = [a.elapsed_time(b) for a, b in pairs]
    res = dict(F=F, fs_l=fs_l, fs_c=fs_c, infos=infos, ms_total=ms_total, dom_ms=dom_ms, gpu_launches=gpu_launches,
               construct_ms=sum(i.build_ms for i in infos), filter_create_ms=filter_create_s * 1e3, shapes=shapes)
    if full and D.rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, dev_dst, shapes)
    captured = None
    if D.rank == 0 and args.parts == 3 and not args.no_verify:
        captured = capture_output_rows(cfg, [planes_np[0], planes_np[F - 1]], [dev_dst[0], dev_dst[F - 1]], shapes)

    if full:
        # ---------------- pure-copy ceiling of the same buffers (no kernels)
        res["ceiling_s"], res["copy_bytes"] = copy_ceiling(D, host_src, host_dst, dev_src, dev_dst, args.inflight, max(2, min(steps, 10)))

        # ---------------- end to end through the host-frame C ABI (caller-pinned host buffers)
        src_np = [[t.numpy() for t in hs] for hs in host_src]
        dst_np = [[t.numpy() for t in hd] for hd in host_dst]
        raw = [flt._frame(s, d) for s, d in zip(src_np, dst_np)]

        def e2e_steps(k):  # k steps back to back, `inflight` frames in flight throughout
            tickets = []
            for _ in range(k):
                for f in range(F):
                    if len(tickets) >= args.inflight:
                        flt.wait(tickets.pop(0))
                    tickets.append(flt.submit_raw(raw[f]))
            for t in tickets:
                flt.wait(t)

        e2e_steps(max(1, warmup // 2))
        D.barrier()
        t0 = time.perf_counter()
        e2e_steps(steps)
        D.barrier()
        res["pinned_s"] = time.perf_counter() - t0
    if sampler:
        res["clocks"] = sampler.stop()
    flt.close()
    del frames_arr, dev_frames, dev_src, dev_dst, host_src, host_dst
    torch.cuda.empty_cache()

    # ---------------- end to end through the plugin (the reference-facing call), pageable frames
    if args.plugin_threads > 0:
        try:
            psteps = max(1, min(steps, 10)) if full else max(1, min(steps, 5))
            psteps = max(psteps, -(-24 // F))  # a stream of at least 24 frames
            dt, construct_s, stats = run_plugin_leg(D, cfg, args.plugin_threads, psteps, 2 if full else 1)
            res["plugin_s"], res["plugin_steps"] = dt, psteps
            res["plugin_construct_ms"], res["plugin_host_buffers"] = construct_s * 1e3, stats
        except Exception as ex:  # the other legs stand on their own
            res["plugin_error"] = str(ex)[:200]
    if captured is not None:  # last: the other ranks wait at the next barrier, not inside a timed leg's warm-up
        res["verified"] = verify_against_oracle(cfg, captured)
    return res


def run_row_bands(D, args, config_id: int):
    """Latency of ONE frame of an 8K config cut into row bands over the GPUs of this run (rank 0 drives all of them
    in-process; the other ranks wait at the barrier).  Caller-pinned planes; median of several frames."""
    import torch

    cfg = CONFIGS[config_id]
    fmt, w, h, tw, th = cfg["fmt"], cfg["w"], cfg["h"], cfg["tw"], cfg["th"]
    out = None
    if D.rank == 0:
        tdtype = {1: torch.uint8, 2: torch.uint16, 4: torch.float32}[np.dtype(fmt.dtype).itemsize]
        planes = synth_frame(fmt, w, h, seed=555)
        hs = [torch.from_numpy(p).pin_memory() for p in planes]
        res = {}
        for label, devices, bands in (("whole_frame_1gpu", [0], 0), ("bands", list(range(D.world)), args.bands * D.world)):
            flt = make_filter(cfg, devices, slots=max(2, args.bands))
            hd = [torch.zeros(d, dtype=tdtype).pin_memory() for _, d in flt.plane_shapes()]
            src_np, dst_np = [t.numpy() for t in hs], [t.numpy() for t in hd]
            times = []
            for it in range(7):
                t0 = time.perf_counter()
                flt.process(src_np, dst_np, bands=bands)
                times.append(time.perf_counter() - t0)
            res[label] = statistics.median(times[2:]) * 1e3
            flt.close()
            del hd
        mpix = tw * th / 1e6
        out = {"workload": cfg["name"], "config_id": config_id, "gpus": D.world, "bands": args.bands * D.world,
               "api": "jinc_filter_process_bands (rank 0 drives every GPU of the run in-process), caller-pinned planes",
               "ms_per_frame_whole_frame_1gpu": res["whole_frame_1gpu"], "ms_per_frame_bands": res["bands"],
               "mpixel_s_bands": mpix / (res["bands"] * 1e-3), "speedup_vs_whole_frame_1gpu": res["whole_frame_1gpu"] / res["bands"]}
    D.barrier()
    return out


def run_b200(args, cfg):
    import torch

    D = Dist()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback")
    numa_cpus = bind_to_gpu_numa(D.local_rank) if D.world > 1 else None
    D.init()
    fmt, tw, th = cfg["fmt"], cfg["tw"], cfg["th"]
    mpix = tw * th / 1e6

    r = measure_config(D, args, cfg, args.config, args.steps, args.warmup, True)
    F = r["F"]
    ms_total, pinned_s, ceiling_s = D.max(r["ms_total"], r["pinned_s"], r["ceiling_s"])
    plugin_s = D.max(r.get("plugin_s", float("nan")))[0]
    gpu_launches = int(D.sum(r["gpu_launches"])[0])

    others = {}
    if not args.no_all_configs and args.config in (1, 2, 3, 4, 5):
        for cid in (1, 2, 3, 4, 5):
            if cid == args.config:
                continue
            c = CONFIGS[cid]
            o = measure_config(D, args, c, cid, max(2, min(args.steps, 5)), 3, False)
            o_ms = D.max(o["ms_total"])[0]
            o_plugin = D.max(o.get("plugin_s", float("nan")))[0]
            steps_o = max(2, min(args.steps, 5))
            flop_o, byts_o, luma_o = algorithmic_work(c, o["fs_l"], o["fs_c"])
            dom = statistics.mean(o["dom_ms"])
            fma_peak, _ = fma_peak_tflops() if D.rank == 0 else (1.0, "")
            others[str(cid)] = {
                "workload": c["name"], "frames_per_step": o["F"],
                "value": D.world * steps_o * o["F"] * (c["tw"] * c["th"] / 1e6) / (o_ms * 1e-3), "unit": "Mpixel/s",
                "launch_ms": dom, "frac": luma_o["flop"] * o["F"] / (dom * 1e-3) / 1e12 / fma_peak,
                "whole_step_frac": flop_o * o["F"] * steps_o / (o["ms_total"] * 1e-3) / 1e12 / fma_peak,
                "e2e": (D.world * o["plugin_steps"] * o["F"] * (c["tw"] * c["th"] / 1e6) / o_plugin) if "plugin_s" in o else None,
                "e2e_host_buffers": o.get("plugin_host_buffers"),
                "construct_ms": o["construct_ms"], "plugin_construct_ms": o.get("plugin_construct_ms"),
                "kernel": KERNEL_NAMES.get(o["infos"][0].fast_path, "resample_strips"),
                "verified": o.get("verified", {}).get("ok")}

    bands = None
    if args.bands > 0:
        try:
            bands = run_row_bands(D, args, args.bands_config)
        except Exception as ex:
            bands = {"error": str(ex)[:200]}
            D.barrier()

    if D.rank == 0:
        infos = r["infos"]
        frames_total = D.world * args.steps * F
        value = frames_total * mpix / (ms_total * 1e-3)
        flop, byts, luma = algorithmic_work(cfg, r["fs_l"], r["fs_c"])
        i0 = infos[0]
        dom_avg_ms = statistics.mean(r["dom_ms"])
        fma_peak, fma_how = fma_peak_tflops()
        hbm_peak, hbm_how = measured_peaks()
        dom_flop = luma["flop"] * F
        dom_bytes = luma["bytes"] * F
        achieved_tf = dom_flop / (dom_avg_ms * 1e-3) / 1e12
        achieved_gbs = dom_bytes / (dom_avg_ms * 1e-3) / 1e9
        shapes = r["shapes"]
        sb = np.dtype(fmt.dtype).itemsize
        h2d = sum(int(np.prod(s)) for s, _ in shapes) * sb * F
        d2h = sum(int(np.prod(d)) for _, d in shapes) * sb * F
        ceiling_gbs = D.world * r["copy_bytes"] / ceiling_s / 1e9
        ceiling_mpix = D.world * F * mpix / ceiling_s

        def e2e_obj(seconds, steps, api, extra=None):
            v = D.world * steps * F * mpix / seconds
            gbs = D.world * (h2d + d2h) * steps / seconds / 1e9
            o = {"value": v, "unit": "Mpixel/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "api": api,
                 "ms_per_step": seconds / steps * 1e3, "pcie_gbs": gbs, "ceiling_gbs": ceiling_gbs,
                 "ceiling_value": ceiling_mpix, "frac": gbs / ceiling_gbs,
                 "ceiling": "pure copies of the same pinned buffers and sizes, no kernels, %d frames in flight per GPU, all %d ranks at once"
                            % (args.inflight, D.world)}
            if extra:
                o.update(extra)
            return o

        pinned = e2e_obj(pinned_s, args.steps, "jinc_filter_submit/jinc_filter_wait (C ABI host-frame call, %d frames in flight per GPU), "
                                               "caller-pinned host planes" % args.inflight)
        if "plugin_s" in r:
            e2e = e2e_obj(plugin_s, r["plugin_steps"],
                          "avisynth_c_plugin_init / get_frame under the mini-host, pageable AviSynth frames, %d concurrent callers per GPU"
                          % args.plugin_threads,
                          {"host_buffers": r["plugin_host_buffers"], "construct_ms": r["plugin_construct_ms"]})
        else:
            e2e = dict(pinned, note="plugin leg unavailable (%s): this is the pinned C-ABI figure" % r.get("plugin_error", "disabled"))
        cpu = None
        if D.world == 1 and not args.no_cpu:
            cpu = run_reference(cfg, steps=3, warmup=1, budget_s=25.0)
            cpu = {k: v for k, v in cpu.items() if k not in ("ms_per_step", "steps", "warmup", "frames_per_step")}
        line = {
            "metric": METRIC, "value": value, "unit": "Mpixel/s", "n_gpus": D.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": config_record(cfg, args.config, byts, args.parts),
            "e2e": e2e,
            "e2e_pinned": pinned,
            "gpu_launches": gpu_launches,
            "clocks": r.get("clocks"),
            "verified": r.get("verified"),
            "construct_ms": {"tables_gpu": r["construct_ms"], "jinc_filter_create": r["filter_create_ms"],
                             "plugin_invoke": r.get("plugin_construct_ms"),
                             "what": "tables_gpu = jinc_table_create wall time summed over the filter's tables (LUT + device table kernels + "
                                     "plans; the reference's counterpart is cpu_baseline.construct_ms); jinc_filter_create adds the CUDA "
                                     "context, streams and pinned frame slots"},
            "roofline": {"bound": "fp32_fma", "kernel": KERNEL_NAMES.get(i0.fast_path, "resample_strips") +
                         " (luma-table planes of all %d frames: interior tiles + border strips)" % F,
                         "achieved": achieved_tf, "peak": fma_peak, "unit": "TFLOP/s", "frac": achieved_tf / fma_peak,
                         "peak_source": fma_how, "traffic": ncu_traffic(args.config, F), "launch_ms": dom_avg_ms,
                         "algorithmic_flop_per_launch": dom_flop, "share_of_step": sum(r["dom_ms"]) / r["ms_total"]},
            "roofline_hbm": {"bound": "hbm", "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s",
                             "frac": achieved_gbs / hbm_peak, "peak_source": hbm_how,
                             "algorithmic_bytes_per_launch": dom_bytes},
            "whole_frame": {"gflop_per_frame": flop / 1e9, "mbytes_per_frame": byts / 1e6,
                            "tflops": flop * args.steps * F / (r["ms_total"] * 1e-3) / 1e12,
                            "frac": flop * args.steps * F / (r["ms_total"] * 1e-3) / 1e12 / fma_peak},
            "all_configs": others or None,
            "row_bands": bands,
            "host": {"threads": host_threads(), "numa_bound_cpus": numa_cpus},
            "cpu_baseline": cpu,
        }
        print(json.dumps(line))
    D.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-all-configs", action="store_true", help="skip the all_configs legs (the other BASELINE configs)")
    ap.add_argument("--no-verify", action="store_true", help="skip the oracle check of the kernel-only output")
    ap.add_argument("--plugin-threads", type=int, default=8,
                    help="concurrent get_frame callers of the plugin end-to-end leg (0 skips it)")
    ap.add_argument("--inflight", type=int, default=3, help="frames in flight per GPU in the pinned end-to-end leg (= pipeline slots)")
    ap.add_argument("--bands", type=int, default=2, help="row bands per GPU in the row_bands leg (0 skips it)")
    ap.add_argument("--bands-config", type=int, default=4, choices=[4, 5], help="the 8K config whose single frame is cut into bands")
    ap.add_argument("--parts", type=int, default=3, choices=[1, 2, 3],
                    help="diagnosis only: 1 = interior tiles, 2 = border strips, 3 = both (the only valid bench setting)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the output planes of the last kernel-only step to DIR/plane<i>.npy (float32; a fixed-seed "
                         "sample of whole rows when the batch exceeds 60 MiB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; it does not apply to --impl reference")
    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return
        r = run_reference(cfg, steps=args.steps, warmup=args.warmup, budget_s=150.0, exact_steps=True)
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "Mpixel/s", "n_gpus": args.gpus,
                "steps": r["steps"], "warmup": r["warmup"], "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config_record(cfg, args.config, frame_bytes(cfg)),
                "cpu_baseline": {k: v for k, v in r.items() if k not in ("ms_per_step", "steps", "warmup", "frames_per_step")},
                "e2e": {"value": r["value"], "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return
    run_b200(args, cfg)


if __name__ == "__main__":
    main()
