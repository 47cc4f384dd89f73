"""ctypes wrapper of the batch extension (include/jsmpeg_b200.h, part 2): N independent streams on
one GPU, device-resident planes, one call decodes the next pictures of every stream."""
from __future__ import annotations

import ctypes

import numpy as np

OUT_DEVICE = 0
OUT_HOST = 1
OUT_RGBA = 2


class Stats(ctypes.Structure):
    _fields_ = [
        ("pictures", ctypes.c_uint64), ("pictures_decoded", ctypes.c_uint64),
        ("coded_blocks", ctypes.c_uint64), ("macroblocks", ctypes.c_uint64),
        ("algorithmic_bytes", ctypes.c_uint64), ("es_bytes", ctypes.c_uint64),
        ("h2d_bytes", ctypes.c_uint64), ("d2h_bytes", ctypes.c_uint64),
        ("kernel_launches", ctypes.c_uint64), ("recon_launches", ctypes.c_uint64),
        ("parse_ms", ctypes.c_double), ("recon_ms", ctypes.c_double), ("scan_ms", ctypes.c_double),
        ("parse_errors", ctypes.c_uint64), ("walk_ms", ctypes.c_double),
        ("lane_walk_pictures", ctypes.c_uint64),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


_VP = ctypes.c_void_p
_BATCH_ABI = {
    "jsmpeg_b200_batch_create": (_VP, [ctypes.c_int, ctypes.c_int, ctypes.c_uint]),
    "jsmpeg_b200_batch_destroy": (None, [_VP]),
    "jsmpeg_b200_batch_get_write_ptr": (_VP, [_VP, ctypes.c_int, ctypes.c_uint]),
    "jsmpeg_b200_batch_did_write": (None, [_VP, ctypes.c_int, ctypes.c_uint]),
    "jsmpeg_b200_batch_get_index": (ctypes.c_int, [_VP, ctypes.c_int]),
    "jsmpeg_b200_batch_set_index": (None, [_VP, ctypes.c_int, ctypes.c_uint]),
    "jsmpeg_b200_batch_stream_info": (ctypes.c_int, [_VP, ctypes.c_int, ctypes.POINTER(ctypes.c_int),
                                                     ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int),
                                                     ctypes.POINTER(ctypes.c_float)]),
    "jsmpeg_b200_batch_write_ts": (ctypes.c_long, [_VP, ctypes.c_int, ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int,
                                                   _VP, _VP, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]),
    "jsmpeg_b200_batch_upload": (ctypes.c_long, [_VP]),
    "jsmpeg_b200_batch_rewind": (None, [_VP]),
    "jsmpeg_b200_batch_reset": (None, [_VP]),
    "jsmpeg_b200_batch_decode": (ctypes.c_long, [_VP, ctypes.c_int, ctypes.c_int]),
    "jsmpeg_b200_batch_get_planes": (ctypes.c_int, [_VP, ctypes.c_int, ctypes.POINTER(_VP), ctypes.POINTER(_VP), ctypes.POINTER(_VP)]),
    "jsmpeg_b200_batch_get_host_planes": (ctypes.c_int, [_VP, ctypes.c_int, ctypes.POINTER(_VP), ctypes.POINTER(_VP), ctypes.POINTER(_VP)]),
    "jsmpeg_b200_batch_get_rgba": (ctypes.c_int, [_VP, ctypes.c_int, ctypes.POINTER(_VP)]),
    "jsmpeg_b200_batch_read_planes": (ctypes.c_int, [_VP, ctypes.c_int, _VP, _VP, _VP]),
    "jsmpeg_b200_batch_read_rgba": (ctypes.c_int, [_VP, ctypes.c_int, _VP]),
    "jsmpeg_b200_batch_last_picture": (ctypes.c_int, [_VP, ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
    "jsmpeg_b200_batch_get_stats": (None, [_VP, ctypes.POINTER(Stats)]),
    "jsmpeg_b200_batch_reset_stats": (None, [_VP]),
    "jsmpeg_b200_debug_parse_picture": (ctypes.c_int, [_VP, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int, ctypes.c_int,
                                                       _VP, _VP, _VP, _VP, _VP]),
    "jsmpeg_b200_debug_reconstruct": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "jsmpeg_b200_debug_reconstruct_batch": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, _VP, ctypes.c_size_t, ctypes.c_size_t,
                                                           ctypes.c_size_t, _VP, _VP, _VP, _VP, _VP, _VP]),
    "jsmpeg_b200_set_default_device": (None, [ctypes.c_int]),
    "jsmpeg_b200_batch_last_error": (ctypes.c_char_p, [_VP]),
    "jsmpeg_b200_batch_set_option": (ctypes.c_int, [_VP, ctypes.c_char_p, ctypes.c_int]),
    "jsmpeg_b200_decoder_last_error": (ctypes.c_char_p, [_VP]),
    "jsmpeg_b200_decoder_set_option": (ctypes.c_int, [_VP, ctypes.c_char_p, ctypes.c_int]),
    "jsmpeg_b200_decoder_last_picture": (ctypes.c_int, [_VP, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
    "jsmpeg_b200_bind_host_to_device": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(ctypes.c_int)]),
    "jsmpeg_b200_version": (ctypes.c_char_p, []),
}


def bind_batch_abi(lib):
    for name, (res, args) in _BATCH_ABI.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


class BatchDecoder:
    """``n_streams`` independent MPEG-1 video decoders on one B200."""

    def __init__(self, n_streams, device=0, max_slots=0, lib=None, chunk_pictures=None, decode_b=None, slice_walk=None):
        from . import capi
        self.lib = lib if lib is not None else capi.product_library()
        self.n_streams = n_streams
        self.handle = self.lib.jsmpeg_b200_batch_create(n_streams, device, max_slots)
        err = self.lib.jsmpeg_b200_batch_last_error(self.handle)
        if err:  # no usable CUDA device: the C ABI answers "false" for ever; the Python host says so loudly
            self.close()
            raise RuntimeError(err.decode(errors="replace"))
        if chunk_pictures is not None:
            self.set_option("chunk_pictures", chunk_pictures)
        if slice_walk is not None:  # I/P pictures of many slices: one lane per slice (same records, another walk kernel)
            self.set_option("slice_walk", slice_walk)
        if decode_b is not None:  # the B-picture extension (the reference skips B pictures, and so does the default)
            self.set_option("decode_b", decode_b)

    def close(self):
        if self.handle:
            self.lib.jsmpeg_b200_batch_destroy(self.handle)
            self.handle = None

    __del__ = close

    def set_option(self, name, value):
        if self.lib.jsmpeg_b200_batch_set_option(self.handle, name.encode(), int(value)) != 0:
            raise ValueError(f"unknown option {name!r}")

    def last_error(self):
        err = self.lib.jsmpeg_b200_batch_last_error(self.handle)
        return err.decode(errors="replace") if err else None

    def write(self, stream, data):
        """Two-phase write of the reference ABI (get_write_ptr / memcpy / did_write)."""
        data = bytes(data) if not isinstance(data, bytes) else data
        ptr = self.lib.jsmpeg_b200_batch_get_write_ptr(self.handle, stream, len(data))
        ctypes.memmove(ptr, data, len(data))
        self.lib.jsmpeg_b200_batch_did_write(self.handle, stream, len(data))

    def write_ts(self, stream, ts_bytes, stream_id=0xE0):
        """MPEG-TS in, demultiplexed on the GPU (any chunking, resyncs like src/ts.js).  Returns (ES bytes
        appended, [(payload byte offset, pts seconds), ...] per PES packet of `stream_id` that starts in it)."""
        ts_bytes = bytes(ts_bytes)
        n_max = len(ts_bytes) // 188 + 1
        pts = np.zeros(n_max, np.uint64)
        off = np.zeros(n_max, np.uint32)
        n = ctypes.c_int()
        total = self.lib.jsmpeg_b200_batch_write_ts(self.handle, stream, ts_bytes, len(ts_bytes), stream_id,
                                                    pts.ctypes.data, off.ctypes.data, n_max, ctypes.byref(n))
        if total < 0:
            raise RuntimeError(self.last_error() or "jsmpeg_b200_batch_write_ts failed")
        return total, [(int(off[i]), float(pts[i]) / 90000.0) for i in range(n.value)]

    def get_index(self, stream):
        return self.lib.jsmpeg_b200_batch_get_index(self.handle, stream)

    def set_index(self, stream, index):
        self.lib.jsmpeg_b200_batch_set_index(self.handle, stream, index)

    def stream_info(self, stream):
        w, h, cs, fr = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_float()
        has = self.lib.jsmpeg_b200_batch_stream_info(self.handle, stream, w, h, cs, fr)
        return {"has_sequence_header": bool(has), "width": w.value, "height": h.value,
                "coded_size": cs.value, "frame_rate": fr.value}

    def upload(self):
        return self.lib.jsmpeg_b200_batch_upload(self.handle)

    def rewind(self):
        self.lib.jsmpeg_b200_batch_rewind(self.handle)

    def reset(self):
        self.lib.jsmpeg_b200_batch_reset(self.handle)

    def decode(self, n_pictures=1, flags=OUT_DEVICE):
        return self.lib.jsmpeg_b200_batch_decode(self.handle, n_pictures, flags)

    def device_planes(self, stream):
        y, cr, cb = _VP(), _VP(), _VP()
        if self.lib.jsmpeg_b200_batch_get_planes(self.handle, stream, y, cr, cb) != 0:
            return None
        return y.value, cr.value, cb.value

    def read_planes(self, stream):
        n = self.stream_info(stream)["coded_size"]
        y = np.empty(n, np.uint8)
        cr = np.empty(n >> 2, np.uint8)
        cb = np.empty(n >> 2, np.uint8)
        rc = self.lib.jsmpeg_b200_batch_read_planes(self.handle, stream, y.ctypes.data, cr.ctypes.data, cb.ctypes.data)
        if rc != 0:
            raise RuntimeError("stream has no sequence header yet")
        return y, cr, cb

    def host_planes(self, stream):
        n = self.stream_info(stream)["coded_size"]
        y, cr, cb = _VP(), _VP(), _VP()
        if self.lib.jsmpeg_b200_batch_get_host_planes(self.handle, stream, y, cr, cb) != 0:
            return None

        def view(p, size):
            return np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctypes.c_uint8)), shape=(size,))

        return view(y, n), view(cr, n >> 2), view(cb, n >> 2)

    def read_rgba(self, stream):
        info = self.stream_info(stream)
        out = np.empty((info["height"], info["width"], 4), np.uint8)
        if self.lib.jsmpeg_b200_batch_read_rgba(self.handle, stream, out.ctypes.data) != 0:
            raise RuntimeError("no RGBA picture (decode with OUT_RGBA first)")
        return out

    def last_picture(self, stream):
        """(picture_coding_type, temporal_reference) of the picture the stream's last decode() consumed, or None."""
        t, r = ctypes.c_int(), ctypes.c_int()
        if self.lib.jsmpeg_b200_batch_last_picture(self.handle, stream, t, r) != 0:
            return None
        return t.value, r.value

    def stats(self):
        st = Stats()
        self.lib.jsmpeg_b200_batch_get_stats(self.handle, ctypes.byref(st))
        return st.as_dict()

    def reset_stats(self):
        self.lib.jsmpeg_b200_batch_reset_stats(self.handle)
