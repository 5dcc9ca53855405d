"""ctypes driver for the in-process VapourSynth (API 4) stand-in (minihost/vs_minihost.cpp).

Used by tests to drive the VapourSynth front-end of the B200 plugin through the host's call sequence: load the
plugin, build a source node, call jinc.JincResize with an argument map, pull frames (two-phase getFrame), read planes and
frame properties.  Test infrastructure; not on the product path.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

VS_MINIHOST_LIB = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libvs_minihost.so")

CF_GRAY, CF_RGB, CF_YUV = 1, 2, 3
ST_INT, ST_FLOAT = 0, 1

_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(VS_MINIHOST_LIB)
        vp, ci = C.c_void_p, C.c_int
        L.vsmh_core_create.restype = vp
        L.vsmh_core_destroy.argtypes = [vp]
        L.vsmh_load_plugin.restype, L.vsmh_load_plugin.argtypes = vp, [vp, C.c_char_p, C.c_char_p, ci]
        L.vsmh_plugin_namespace.restype, L.vsmh_plugin_namespace.argtypes = C.c_char_p, [vp]
        L.vsmh_plugin_id.restype, L.vsmh_plugin_id.argtypes = C.c_char_p, [vp]
        L.vsmh_function_args.restype, L.vsmh_function_args.argtypes = C.c_char_p, [vp, C.c_char_p]
        L.vsmh_source_create.restype, L.vsmh_source_create.argtypes = vp, [vp] + [ci] * 9
        L.vsmh_source_fill_plane.restype, L.vsmh_source_fill_plane.argtypes = ci, [vp, ci, ci, vp, C.c_ssize_t]
        L.vsmh_source_set_prop_int.argtypes = [vp, C.c_char_p, C.c_int64]
        L.vsmh_map_create.restype = vp
        L.vsmh_map_free.argtypes = [vp]
        L.vsmh_map_set_node.argtypes = [vp, C.c_char_p, vp]
        L.vsmh_map_set_int.argtypes = [vp, C.c_char_p, C.c_int64]
        L.vsmh_map_set_float.argtypes = [vp, C.c_char_p, C.c_double]
        L.vsmh_map_set_data.argtypes = [vp, C.c_char_p, C.c_char_p]
        L.vsmh_invoke.restype, L.vsmh_invoke.argtypes = vp, [vp, C.c_char_p, vp, C.c_char_p, ci]
        L.vsmh_node_info.argtypes = [vp] + [C.POINTER(ci)] * 5
        L.vsmh_node_format.argtypes = [vp, C.POINTER(ci), C.POINTER(ci)]
        L.vsmh_get_frame.restype, L.vsmh_get_frame.argtypes = vp, [vp, ci, C.c_char_p, ci]
        L.vsmh_frame_plane.argtypes = [vp, ci, C.POINTER(vp), C.POINTER(C.c_ssize_t), C.POINTER(ci), C.POINTER(ci)]
        L.vsmh_frame_prop_int.restype, L.vsmh_frame_prop_int.argtypes = ci, [vp, C.c_char_p, C.POINTER(C.c_int64)]
        L.vsmh_free_frame.argtypes = [vp]
        L.vsmh_free_node.argtypes = [vp]
        L.vsmh_live_frames.restype = C.c_long
        L.vsmh_live_nodes.restype = C.c_long
        L.vsmh_pull_frames.restype, L.vsmh_pull_frames.argtypes = C.c_double, [vp, ci, ci, ci]
        _lib = L
    return _lib


class VsError(RuntimeError):
    pass


class Node:
    def __init__(self, handle, dtype):
        self.handle, self.dtype = handle, dtype

    @property
    def info(self):
        v = [C.c_int() for _ in range(5)]
        lib().vsmh_node_info(self.handle, *[C.byref(x) for x in v])
        return dict(zip(("width", "height", "num_frames", "num_planes", "bytes_per_sample"), (x.value for x in v)))

    @property
    def format(self):
        """(sample type, bits per sample) of the clip: ST_INT or ST_FLOAT."""
        st, bits = C.c_int(), C.c_int()
        lib().vsmh_node_format(self.handle, C.byref(st), C.byref(bits))
        return st.value, bits.value

    def get_frame(self, n: int):
        """(planes, props): planes in VapourSynth order (Y,U,V or R,G,B)."""
        L = lib()
        err = C.create_string_buffer(512)
        f = L.vsmh_get_frame(self.handle, n, err, 512)
        if not f:
            raise VsError(err.value.decode())
        try:
            planes = []
            for p in range(self.info["num_planes"]):
                ptr, stride, w, h = C.c_void_p(), C.c_ssize_t(), C.c_int(), C.c_int()
                L.vsmh_frame_plane(f, p, C.byref(ptr), C.byref(stride), C.byref(w), C.byref(h))
                raw = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(h.value, stride.value))
                planes.append(raw[:, : w.value * np.dtype(self.dtype).itemsize].copy().view(self.dtype))
            props = {}
            v = C.c_int64()
            for key in ("_ChromaLocation", "_Matrix", "_ColorRange"):
                if L.vsmh_frame_prop_int(f, key.encode(), C.byref(v)):
                    props[key] = v.value
            return planes, props
        finally:
            L.vsmh_free_frame(f)

    def pull(self, first: int, count: int, threads: int = 1) -> float:
        t = lib().vsmh_pull_frames(self.handle, first, count, threads)
        if t < 0:
            raise VsError("getFrame failed while pulling frames")
        return t

    def release(self):
        if self.handle:
            lib().vsmh_free_node(self.handle)
            self.handle = None


class Core:
    def __init__(self):
        self.handle = lib().vsmh_core_create()

    def load_plugin(self, path: str) -> "Plugin":
        err = C.create_string_buffer(512)
        h = lib().vsmh_load_plugin(self.handle, path.encode(), err, 512)
        if not h:
            raise VsError(err.value.decode())
        return Plugin(h)

    def source(self, family: int, dtype, bits: int, ssw: int, ssh: int, width: int, height: int, frames, num_frames=None, props=None) -> Node:
        """frames: list (one per stored frame) of lists of 2-D numpy planes in VapourSynth order."""
        st = ST_FLOAT if np.issubdtype(np.dtype(dtype), np.floating) else ST_INT
        h = lib().vsmh_source_create(self.handle, family, st, bits, ssw, ssh, width, height, num_frames or len(frames), len(frames))
        for k, planes in enumerate(frames):
            for p, arr in enumerate(planes):
                arr = np.ascontiguousarray(arr, dtype=dtype)
                assert lib().vsmh_source_fill_plane(h, k, p, arr.ctypes.data, arr.strides[0]) == 0
        for key, val in (props or {}).items():
            lib().vsmh_source_set_prop_int(h, key.encode(), int(val))
        return Node(h, dtype)

    @staticmethod
    def live_objects():
        return lib().vsmh_live_frames(), lib().vsmh_live_nodes()


class Plugin:
    def __init__(self, handle):
        self.handle = handle

    @property
    def namespace(self) -> str:
        return lib().vsmh_plugin_namespace(self.handle).decode()

    def function_args(self, name: str):
        s = lib().vsmh_function_args(self.handle, name.encode())
        return s.decode() if s else None

    def invoke(self, name: str, clip: Node, **named) -> Node:
        L = lib()
        m = L.vsmh_map_create()
        try:
            if clip is not None:
                L.vsmh_map_set_node(m, b"clip", clip.handle)
            for k, v in named.items():
                if v is None:
                    continue
                if isinstance(v, (int, np.integer)):
                    L.vsmh_map_set_int(m, k.encode(), int(v))
                elif isinstance(v, (float, np.floating)):
                    L.vsmh_map_set_float(m, k.encode(), float(v))
                elif isinstance(v, str):
                    L.vsmh_map_set_data(m, k.encode(), v.encode())
                else:
                    raise TypeError(type(v))
            err = C.create_string_buffer(512)
            h = L.vsmh_invoke(self.handle, name.encode(), m, err, 512)
            if not h:
                raise VsError(err.value.decode())
            return Node(h, clip.dtype)
        finally:
            L.vsmh_map_free(m)
