"""ctypes binding of the C ABI in include/jinc_b200.h (libjinc_b200.so).

The library is the product; this module only loads it and marshals arguments.  There is no CPU
fallback: if the shared library is missing, or no CUDA device is present, calls raise JincError.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import paths

MAX_PLANES = 4
MAX_DEVICES = 16
CPLACE = {"mpeg2": 0, "mpeg1": 1, "topleft": 2}
SAMPLE_F16 = 0x102  # JINC_SAMPLE_F16: IEEE binary16 planes (numpy float16), passed where the ABI takes sample_bytes
DTYPES = {1: np.uint8, 2: np.uint16, 4: np.float32, SAMPLE_F16: np.float16}
PATH_NAMES = {0: "general", 1: "up2x", 2: "down_int", 3: "periodic", 4: "piecewise"}


class JincError(RuntimeError):
    pass


class TableParams(C.Structure):
    _fields_ = [("quant_x", C.c_int32), ("quant_y", C.c_int32), ("src_w", C.c_int32), ("src_h", C.c_int32),
                ("dst_w", C.c_int32), ("dst_h", C.c_int32), ("radius", C.c_double), ("blur", C.c_double),
                ("crop_left", C.c_double), ("crop_top", C.c_double), ("crop_w", C.c_double), ("crop_h", C.c_double)]


class TableInfo(C.Structure):
    _fields_ = [("filter_size", C.c_int32), ("n_phase_x", C.c_int32), ("n_phase_y", C.c_int32),
                ("n_border_cols", C.c_int32), ("n_border_rows", C.c_int32), ("fast_path", C.c_int32),
                ("interior_x0", C.c_int32), ("interior_x1", C.c_int32), ("interior_y0", C.c_int32),
                ("interior_y1", C.c_int32), ("filter_support", C.c_float), ("build_ms", C.c_float),
                ("up2x_taps", C.c_int32)]


class FilterParams(C.Structure):
    _fields_ = [("src_w", C.c_int32), ("src_h", C.c_int32), ("target_w", C.c_int32), ("target_h", C.c_int32),
                ("src_left", C.c_double), ("src_top", C.c_double), ("src_width", C.c_double), ("src_height", C.c_double),
                ("quant_x", C.c_int32), ("quant_y", C.c_int32), ("tap", C.c_int32), ("blur", C.c_double),
                ("cplace", C.c_int32), ("n_planes", C.c_int32), ("sub_w", C.c_int32), ("sub_h", C.c_int32),
                ("sample_bytes", C.c_int32), ("bits", C.c_int32), ("n_devices", C.c_int32),
                ("devices", C.c_int32 * MAX_DEVICES), ("slots_per_device", C.c_int32), ("flags", C.c_int32)]

FLAG_HOST_REGISTER = 1
FLAG_DST_PADDING_WRITABLE = 2
E_BUSY = -5


class Frame(C.Structure):
    _fields_ = [("src", C.c_void_p * MAX_PLANES), ("src_pitch", C.c_ssize_t * MAX_PLANES),
                ("dst", C.c_void_p * MAX_PLANES), ("dst_pitch", C.c_ssize_t * MAX_PLANES)]


# every symbol include/jinc_b200.h declares (tests check the library exports all of them)
EXPORTS = [
    "jinc_abi_version", "jinc_last_error", "jinc_device_count", "jinc_radius_for_tap", "jinc_eval_sqr",
    "jinc_lut_build", "jinc_ctx_create", "jinc_ctx_destroy", "jinc_ctx_device", "jinc_table_create",
    "jinc_table_destroy", "jinc_table_get_info", "jinc_table_axis", "jinc_table_pixel_weights",
    "jinc_table_pixel_block", "jinc_resize_plane_device", "jinc_table_launches_per_plane", "jinc_table_strip_plan",
    "jinc_filter_create",
    "jinc_filter_destroy", "jinc_filter_table", "jinc_filter_num_tables", "jinc_filter_num_devices",
    "jinc_filter_process", "jinc_filter_submit", "jinc_filter_wait", "jinc_filter_process_split",
    "jinc_filter_kernel_launches", "jinc_filter_process_device", "jinc_filter_process_device_batch",
    "jinc_plan_frame_owner", "jinc_plan_row_bands", "jinc_filter_num_slots", "jinc_filter_try_submit",
    "jinc_filter_process_bands", "jinc_host_buffer_stats", "jinc_filter_live_count", "jinc_filter_set_antiring",
    "jinc_antiring_plane_device", "jinc_resize_planes_device", "jinc_resize_adjoint_planes_device",
    "jinc_antiring_planes_device", "jinc_antiring_adjoint_planes_device",
]

_lib = None


def lib():
    global _lib
    if _lib is None:
        path = paths.cuda_lib()
        if not os.path.exists(path):
            raise JincError(f"{path} is missing: build it with `make cuda` (or __graft_entry__.build()); "
                            "there is no CPU fallback")
        L = C.CDLL(path)
        vp, ci, cd = C.c_void_p, C.c_int, C.c_double
        L.jinc_abi_version.restype = ci
        L.jinc_last_error.restype = C.c_char_p
        L.jinc_device_count.restype = ci
        L.jinc_radius_for_tap.restype, L.jinc_radius_for_tap.argtypes = cd, [ci]
        L.jinc_eval_sqr.restype, L.jinc_eval_sqr.argtypes = cd, [cd]
        L.jinc_lut_build.restype, L.jinc_lut_build.argtypes = ci, [cd, cd, C.POINTER(cd)]
        L.jinc_ctx_create.restype, L.jinc_ctx_create.argtypes = ci, [ci, C.POINTER(vp)]
        L.jinc_ctx_destroy.restype, L.jinc_ctx_destroy.argtypes = None, [vp]
        L.jinc_ctx_device.restype, L.jinc_ctx_device.argtypes = ci, [vp]
        L.jinc_table_create.restype, L.jinc_table_create.argtypes = ci, [vp, C.POINTER(TableParams), C.POINTER(vp)]
        L.jinc_table_destroy.restype, L.jinc_table_destroy.argtypes = None, [vp]
        L.jinc_table_get_info.restype, L.jinc_table_get_info.argtypes = ci, [vp, C.POINTER(TableInfo)]
        L.jinc_table_axis.restype, L.jinc_table_axis.argtypes = ci, [vp, ci, vp, vp, vp, vp]
        L.jinc_table_pixel_weights.restype, L.jinc_table_pixel_weights.argtypes = ci, [vp, ci, ci, vp]
        L.jinc_table_pixel_block.restype, L.jinc_table_pixel_block.argtypes = ci, [vp, ci, ci, C.POINTER(C.c_int64)]
        L.jinc_resize_plane_device.restype = ci
        L.jinc_resize_plane_device.argtypes = [vp, vp, ci, C.c_float, vp, C.c_ssize_t, vp, C.c_ssize_t, vp]
        L.jinc_resize_planes_device.restype = ci
        L.jinc_resize_planes_device.argtypes = [vp, vp, ci, C.c_float, ci, vp, C.c_ssize_t, C.c_ssize_t, vp, C.c_ssize_t,
                                                C.c_ssize_t, vp]
        L.jinc_resize_adjoint_planes_device.restype = ci
        L.jinc_resize_adjoint_planes_device.argtypes = [vp, vp, ci, vp, C.c_ssize_t, C.c_ssize_t, vp, C.c_ssize_t, C.c_ssize_t, vp]
        L.jinc_antiring_planes_device.restype = ci
        L.jinc_antiring_planes_device.argtypes = [vp, vp, ci, C.c_float, ci, vp, C.c_ssize_t, C.c_ssize_t, vp, C.c_ssize_t,
                                                  C.c_ssize_t, vp]
        L.jinc_antiring_adjoint_planes_device.restype = ci
        L.jinc_antiring_adjoint_planes_device.argtypes = [vp, vp, ci, C.c_float, ci] + [vp, C.c_ssize_t, C.c_ssize_t] * 5 + [vp]
        L.jinc_antiring_plane_device.restype = ci
        L.jinc_antiring_plane_device.argtypes = [vp, vp, ci, C.c_float, vp, C.c_ssize_t, vp, C.c_ssize_t, vp]
        L.jinc_filter_set_antiring.restype, L.jinc_filter_set_antiring.argtypes = ci, [vp, C.c_float]
        L.jinc_table_launches_per_plane.restype, L.jinc_table_launches_per_plane.argtypes = ci, [vp]
        L.jinc_table_strip_plan.restype, L.jinc_table_strip_plan.argtypes = ci, [vp, C.POINTER(ci)]
        L.jinc_filter_create.restype, L.jinc_filter_create.argtypes = ci, [C.POINTER(FilterParams), C.POINTER(vp)]
        L.jinc_filter_destroy.restype, L.jinc_filter_destroy.argtypes = None, [vp]
        L.jinc_filter_table.restype, L.jinc_filter_table.argtypes = vp, [vp, ci]
        L.jinc_filter_num_tables.restype, L.jinc_filter_num_tables.argtypes = ci, [vp]
        L.jinc_filter_num_devices.restype, L.jinc_filter_num_devices.argtypes = ci, [vp]
        L.jinc_filter_process.restype, L.jinc_filter_process.argtypes = ci, [vp, C.POINTER(Frame)]
        L.jinc_filter_submit.restype, L.jinc_filter_submit.argtypes = ci, [vp, C.POINTER(Frame), C.POINTER(C.c_int64)]
        L.jinc_filter_wait.restype, L.jinc_filter_wait.argtypes = ci, [vp, C.c_int64]
        L.jinc_filter_process_split.restype, L.jinc_filter_process_split.argtypes = ci, [vp, C.POINTER(Frame)]
        L.jinc_filter_process_device.restype = ci
        L.jinc_filter_process_device.argtypes = [vp, ci, C.POINTER(Frame), ci, ci, vp]
        L.jinc_filter_process_device_batch.restype = ci
        L.jinc_filter_process_device_batch.argtypes = [vp, ci, C.POINTER(Frame), ci, ci, ci, vp]
        L.jinc_filter_kernel_launches.restype, L.jinc_filter_kernel_launches.argtypes = C.c_int64, [vp]
        L.jinc_filter_num_slots.restype, L.jinc_filter_num_slots.argtypes = ci, [vp]
        L.jinc_filter_try_submit.restype = ci
        L.jinc_filter_try_submit.argtypes = [vp, C.POINTER(Frame), C.POINTER(C.c_int64)]
        L.jinc_filter_process_bands.restype, L.jinc_filter_process_bands.argtypes = ci, [vp, C.POINTER(Frame), ci]
        L.jinc_host_buffer_stats.restype = None
        L.jinc_host_buffer_stats.argtypes = [C.POINTER(C.c_int64)] * 5
        L.jinc_filter_live_count.restype = ci
        L.jinc_plan_frame_owner.restype, L.jinc_plan_frame_owner.argtypes = ci, [C.c_int64, ci]
        L.jinc_plan_row_bands.restype = ci
        L.jinc_plan_row_bands.argtypes = [ci, ci, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        _lib = L
    return _lib


def _check(rc: int):
    if rc != 0:
        raise JincError(f"[{rc}] {lib().jinc_last_error().decode()}")


def device_count() -> int:
    return lib().jinc_device_count()


def live_filters() -> int:
    return lib().jinc_filter_live_count()


def host_buffer_stats() -> dict:
    """Process-wide bookkeeping of the frame pipeline's view of caller buffers (jinc_host_buffer_stats)."""
    v = [C.c_int64() for _ in range(5)]
    lib().jinc_host_buffer_stats(*[C.byref(x) for x in v])
    return dict(zip(("registered_bytes", "registrations", "direct_src_frames", "direct_dst_frames", "staged_frames"),
                    (x.value for x in v)))


def frame_owner(frame: int, n_parts: int) -> int:
    """Part (GPU of a filter, or rank of a multi-process job) that frame `frame` belongs to.  Host-only."""
    r = lib().jinc_plan_frame_owner(frame, n_parts)
    if r < 0:
        _check(r)
    return r


def frames_of(part: int, n_parts: int, n_frames: int) -> list[int]:
    """Frames of a clip of n_frames that part `part` processes (frame-parallel partition, no exchange)."""
    return [n for n in range(n_frames) if frame_owner(n, n_parts) == part]


def row_bands(target_h: int, n_parts: int) -> list[tuple[int, int]]:
    """Output-row bands [y0, y1) of the row-band split of one frame over n_parts GPUs.  Host-only."""
    y0 = (C.c_int32 * n_parts)()
    y1 = (C.c_int32 * n_parts)()
    _check(lib().jinc_plan_row_bands(target_h, n_parts, y0, y1))
    return [(int(a), int(b)) for a, b in zip(y0, y1)]


def radius_for_tap(tap: int) -> float:
    return lib().jinc_radius_for_tap(tap)


def lut_build(tap: int, blur: float = 0.0) -> np.ndarray:
    out = np.zeros(1024, dtype=np.float64)
    _check(lib().jinc_lut_build(radius_for_tap(tap), float(np.float32(blur)), out.ctypes.data_as(C.POINTER(C.c_double))))
    return out


class Context:
    def __init__(self, device: int = 0):
        h = C.c_void_p()
        _check(lib().jinc_ctx_create(device, C.byref(h)))
        self.handle = h

    def close(self):
        if self.handle:
            lib().jinc_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class TableView:
    """Read-only wrapper over a jinc_table* (owned by a Table or by a Filter)."""

    def __init__(self, handle, dst_w: int, dst_h: int):
        self.handle, self.dst_w, self.dst_h = handle, dst_w, dst_h

    @property
    def info(self) -> TableInfo:
        i = TableInfo()
        _check(lib().jinc_table_get_info(self.handle, C.byref(i)))
        return i

    def axis(self, axis: int):
        n = self.dst_w if axis == 0 else self.dst_h
        start = np.zeros(n, np.int32)
        phase = np.zeros(n, np.int32)
        border = np.zeros(n, np.uint8)
        pos = np.zeros(n, np.float32)
        _check(lib().jinc_table_axis(self.handle, axis, start.ctypes.data, phase.ctypes.data, border.ctypes.data,
                                     pos.ctypes.data))
        return start, phase, border, pos

    def pixel_weights(self, x: int, y: int) -> np.ndarray:
        fs = self.info.filter_size
        out = np.zeros((fs, fs), np.float32)
        _check(lib().jinc_table_pixel_weights(self.handle, x, y, out.ctypes.data))
        return out

    def pixel_block(self, x: int, y: int) -> int:
        v = C.c_int64()
        _check(lib().jinc_table_pixel_block(self.handle, x, y, C.byref(v)))
        return v.value

    @property
    def launches_per_plane(self) -> int:
        return lib().jinc_table_launches_per_plane(self.handle)

    @property
    def strip_plan(self) -> tuple:
        """(strip patches per plane, patches with their weight blocks in shared memory); (0, 0) without a plan"""
        staged = C.c_int(0)
        n = lib().jinc_table_strip_plan(self.handle, C.byref(staged))
        return n, staged.value


class Table(TableView):
    def __init__(self, ctx: Context, *, quant_x=256, quant_y=256, src_w, src_h, dst_w, dst_h, radius, blur=0.0,
                 crop_left=0.0, crop_top=0.0, crop_w=None, crop_h=None):
        p = TableParams(quant_x, quant_y, src_w, src_h, dst_w, dst_h, radius, blur, crop_left, crop_top,
                        float(src_w) if crop_w is None else crop_w, float(src_h) if crop_h is None else crop_h)
        h = C.c_void_p()
        _check(lib().jinc_table_create(ctx.handle, C.byref(p), C.byref(h)))
        super().__init__(h, dst_w, dst_h)
        self.ctx = ctx

    def resize_device(self, sample_bytes: int, peak: float, d_src: int, src_pitch: int, d_dst: int, dst_pitch: int,
                      stream: int = 0):
        """One device-resident plane; sample_bytes is 1, 2, 4 or SAMPLE_F16 (peak is then ignored)."""
        _check(lib().jinc_resize_plane_device(self.ctx.handle, self.handle, sample_bytes, peak, d_src, src_pitch,
                                              d_dst, dst_pitch, stream or None))

    def resize_planes_device(self, sample_bytes: int, peak: float, n_planes: int, d_src: int, src_pitch: int,
                             src_plane_stride: int, d_dst: int, dst_pitch: int, dst_plane_stride: int, stream: int = 0):
        """n_planes device-resident planes of this table's geometry in one call (jinc_resize_planes_device); pitches and
        plane strides in bytes."""
        _check(lib().jinc_resize_planes_device(self.ctx.handle, self.handle, sample_bytes, peak, n_planes, d_src, src_pitch,
                                               src_plane_stride, d_dst, dst_pitch, dst_plane_stride, stream or None))

    def adjoint_planes_device(self, n_planes: int, d_grad_dst: int, grad_dst_pitch: int, grad_dst_plane_stride: int,
                              d_grad_src: int, grad_src_pitch: int, grad_src_plane_stride: int, stream: int = 0):
        """Adjoint (transpose) of the resize on n_planes float32 gradient planes (jinc_resize_adjoint_planes_device)."""
        _check(lib().jinc_resize_adjoint_planes_device(self.ctx.handle, self.handle, n_planes, d_grad_dst, grad_dst_pitch,
                                                       grad_dst_plane_stride, d_grad_src, grad_src_pitch,
                                                       grad_src_plane_stride, stream or None))

    def antiring_planes_device(self, sample_bytes: int, strength: float, n_planes: int, d_src: int, src_pitch: int,
                               src_plane_stride: int, d_dst: int, dst_pitch: int, dst_plane_stride: int, stream: int = 0):
        """Anti-ringing clamp in place on n_planes planes resize_planes_device produced (jinc_antiring_planes_device)."""
        _check(lib().jinc_antiring_planes_device(self.ctx.handle, self.handle, sample_bytes, strength, n_planes, d_src,
                                                 src_pitch, src_plane_stride, d_dst, dst_pitch, dst_plane_stride,
                                                 stream or None))

    def antiring_adjoint_planes_device(self, sample_bytes: int, strength: float, n_planes: int, src, y, grad_dst, grad_y,
                                       grad_src, stream: int = 0):
        """Gradient of resize + anti-ringing clamp (jinc_antiring_adjoint_planes_device) for float32 / SAMPLE_F16 planes.
        src, y, grad_dst, grad_y, grad_src: (device pointer, pitch, plane stride) in bytes; writes grad_y and grad_src."""
        planes = [v for t in (src, y, grad_dst, grad_y, grad_src) for v in t]
        _check(lib().jinc_antiring_adjoint_planes_device(self.ctx.handle, self.handle, sample_bytes, strength, n_planes,
                                                         *planes, stream or None))

    def antiring_device(self, sample_bytes: int, strength: float, d_src: int, src_pitch: int, d_dst: int, dst_pitch: int,
                        stream: int = 0):
        """Anti-ringing clamp in place on a plane resize_device produced from d_src (jinc_antiring_plane_device)."""
        _check(lib().jinc_antiring_plane_device(self.ctx.handle, self.handle, sample_bytes, strength, d_src, src_pitch,
                                                d_dst, dst_pitch, stream or None))

    def close(self):
        if self.handle:
            lib().jinc_table_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Filter:
    """A filter instance over host frames: the call a plugin's GetFrame makes (jinc_filter_process)."""

    def __init__(self, *, src_w, src_h, target_w, target_h, n_planes, sample_bytes, bits, sub_w=0, sub_h=0,
                 src_left=0.0, src_top=0.0, src_width=None, src_height=None, quant_x=256, quant_y=256, tap=3,
                 blur=0.0, cplace="mpeg2", devices=None, slots_per_device=0, flags=0):
        f32 = lambda v: float(np.float32(v))  # script floats are 32-bit
        p = FilterParams()
        p.src_w, p.src_h, p.target_w, p.target_h = src_w, src_h, target_w, target_h
        p.src_left, p.src_top = f32(src_left), f32(src_top)
        p.src_width = f32(src_width) if src_width is not None else float(src_w)
        p.src_height = f32(src_height) if src_height is not None else float(src_h)
        p.quant_x, p.quant_y, p.tap, p.blur = quant_x, quant_y, tap, f32(blur)
        p.cplace = CPLACE[cplace.lower()]
        p.n_planes, p.sub_w, p.sub_h, p.sample_bytes, p.bits = n_planes, sub_w, sub_h, sample_bytes, bits
        devices = list(devices) if devices is not None else []
        p.n_devices = len(devices)
        for i, d in enumerate(devices[:MAX_DEVICES]):
            p.devices[i] = d
        p.slots_per_device = slots_per_device
        p.flags = flags
        self.params = p
        h = C.c_void_p()
        _check(lib().jinc_filter_create(C.byref(p), C.byref(h)))
        self.handle = h
        self.dtype = DTYPES[sample_bytes]

    def plane_shapes(self):
        p = self.params
        out = []
        for i in range(p.n_planes):
            sub = i in (1, 2) and (p.sub_w or p.sub_h)
            out.append(((p.src_h >> p.sub_h, p.src_w >> p.sub_w) if sub else (p.src_h, p.src_w),
                        (p.target_h >> p.sub_h, p.target_w >> p.sub_w) if sub else (p.target_h, p.target_w)))
        return out

    def table(self, k: int) -> TableView:
        h = lib().jinc_filter_table(self.handle, k)
        if not h:
            raise IndexError(k)
        p = self.params
        if k == 0:
            return TableView(h, p.target_w, p.target_h)
        return TableView(h, p.target_w >> p.sub_w, p.target_h >> p.sub_h)

    @property
    def num_tables(self) -> int:
        return lib().jinc_filter_num_tables(self.handle)

    @property
    def num_devices(self) -> int:
        return lib().jinc_filter_num_devices(self.handle)

    @property
    def num_slots(self) -> int:
        return lib().jinc_filter_num_slots(self.handle)

    @property
    def kernel_launches(self) -> int:
        return lib().jinc_filter_kernel_launches(self.handle)

    def set_antiring(self, strength: float):
        """Anti-ringing strength of frames submitted from now on: 0 (off, the default) .. 1 (jinc_filter_set_antiring)."""
        _check(lib().jinc_filter_set_antiring(self.handle, strength))

    def _frame(self, src_planes, dst_planes) -> Frame:
        fr = Frame()
        for i, (s, d) in enumerate(zip(src_planes, dst_planes)):
            assert s.dtype == self.dtype and d.dtype == self.dtype
            assert s.strides[1] == s.itemsize and d.strides[1] == d.itemsize
            fr.src[i], fr.src_pitch[i] = s.ctypes.data, s.strides[0]
            fr.dst[i], fr.dst_pitch[i] = d.ctypes.data, d.strides[0]
        return fr

    def alloc_dst(self):
        return [np.zeros(dst, dtype=self.dtype) for _, dst in self.plane_shapes()]

    def process(self, src_planes, dst_planes=None, split=False, bands=0):
        """One frame through jinc_filter_process; split=True: jinc_filter_process_split (one row band per GPU);
        bands=n: jinc_filter_process_bands with n row bands."""
        dst_planes = dst_planes if dst_planes is not None else self.alloc_dst()
        fr = self._frame(src_planes, dst_planes)
        if bands:
            _check(lib().jinc_filter_process_bands(self.handle, C.byref(fr), bands))
        else:
            fn = lib().jinc_filter_process_split if split else lib().jinc_filter_process
            _check(fn(self.handle, C.byref(fr)))
        return dst_planes

    def process_raw(self, frame: Frame):
        _check(lib().jinc_filter_process(self.handle, C.byref(frame)))

    def process_device(self, frame: Frame, device_index: int = 0, table_mask: int = 3, parts: int = 3, stream: int = 0):
        """Device-resident frame (Frame holds device pointers); asynchronous on `stream`."""
        _check(lib().jinc_filter_process_device(self.handle, device_index, C.byref(frame), table_mask, parts,
                                                stream or None))

    def process_device_batch(self, frames, device_index: int = 0, table_mask: int = 3, parts: int = 3, stream: int = 0):
        """frames: a ctypes array (Frame * n) of device-pointer frames; one launch per table for the whole batch."""
        _check(lib().jinc_filter_process_device_batch(self.handle, device_index, frames, len(frames), table_mask, parts,
                                                      stream or None))

    def submit(self, src_planes, dst_planes) -> int:
        fr = self._frame(src_planes, dst_planes)
        t = C.c_int64()
        _check(lib().jinc_filter_submit(self.handle, C.byref(fr), C.byref(t)))
        return t.value

    def submit_raw(self, frame: Frame) -> int:
        t = C.c_int64()
        _check(lib().jinc_filter_submit(self.handle, C.byref(frame), C.byref(t)))
        return t.value

    def try_submit(self, src_planes, dst_planes):
        """Ticket, or None when every in-flight slot is taken (JINC_E_BUSY)."""
        fr = self._frame(src_planes, dst_planes)
        t = C.c_int64()
        rc = lib().jinc_filter_try_submit(self.handle, C.byref(fr), C.byref(t))
        if rc == E_BUSY:
            return None
        _check(rc)
        return t.value

    def wait(self, ticket: int):
        _check(lib().jinc_filter_wait(self.handle, ticket))

    def close(self):
        if self.handle:
            lib().jinc_filter_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
