"""ctypes view of the C ABI in include/sxgpu.h (libsxgpu.so).

Python is not on the data path: these bindings exist so that tests/ and bench.py can call
the same entry points a C++ host (the driver=sx device in csrc/host) calls.  There is no
CPU fallback -- if the library cannot be loaded, or no sm_100 GPU is present, this raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

from . import _build

SXGPU_OK = 0
ERR_INVALID, ERR_CUDA, ERR_NO_DEVICE, ERR_NOMEM, ERR_UNSUPPORTED = -1, -2, -3, -4, -5


class SxGpuError(RuntimeError):
    def __init__(self, code: int, what: str, detail: str = ""):
        super().__init__(f"{what}: {code} {detail}".strip())
        self.code = code


class Info(C.Structure):
    _fields_ = [("device", C.c_int), ("sm_count", C.c_int), ("cc_major", C.c_int), ("cc_minor", C.c_int),
                ("l2_bytes", C.c_uint64), ("hbm_bytes", C.c_uint64), ("name", C.c_char * 64)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("sum", "wsum", "x", "count", "tx_on", "rail")]

    def as_tuple(self):
        return (self.sum, self.wsum, self.x, self.count, self.tx_on, self.rail)


class BankConfig(C.Structure):
    _fields_ = [("nstreams", C.c_uint32), ("period", C.c_uint32), ("sample_rate", C.c_double),
                ("tx_threshold2", C.c_float), ("reserved", C.c_uint32), ("seed", C.c_uint64)]


class Block(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dest", C.c_void_p), ("length", C.c_uint64),
                ("tx_threshold2", C.c_float), ("reserved", C.c_uint32)]


_P, _S, _F = C.c_void_p, C.c_size_t, C.c_float

# name -> (restype, argtypes); every symbol include/sxgpu.h declares
SIGNATURES = {
    "sxgpu_init": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "sxgpu_destroy": (C.c_int, [_P]),
    "sxgpu_abi_version": (C.c_int, []),
    "sxgpu_strerror": (C.c_char_p, [C.c_int]),
    "sxgpu_last_error": (C.c_char_p, [_P]),
    "sxgpu_device_info": (C.c_int, [_P, C.POINTER(Info)]),
    "sxgpu_convert_rx_buffer": (C.c_int, [_P, _P, _S, _P, _S, _S, _P]),
    "sxgpu_convert_tx_buffer": (C.c_int, [_P, _P, _S, _P, _S, _S, _F, _P]),
    "sxgpu_convert_rx_buffer_cs16": (C.c_int, [_P, _P, _S, _P, _S, _S, _P]),
    "sxgpu_convert_tx_buffer_cs16": (C.c_int, [_P, _P, _S, _P, _S, _S, _F, _P]),
    "sxgpu_convert_rx_buffer_s16": (C.c_int, [_P, _P, _S, _P, _S, _S, _P]),
    "sxgpu_convert_tx_buffer_s16": (C.c_int, [_P, _P, _S, _P, _S, _S, _F, _P]),
    "sxgpu_convert_rx_batch": (C.c_int, [_P, _P, C.c_uint32, C.c_int, _S, _P]),
    "sxgpu_convert_tx_batch": (C.c_int, [_P, _P, C.c_uint32, C.c_int, _S, _P]),
    "sxgpu_convert_loopback": (C.c_int, [_P, _P, _P, _P, _S, _F, _P]),
    "sxgpu_fill_silence": (C.c_int, [_P, _P, _S, _S, _P]),
    "sxgpu_bank_create": (C.c_int, [_P, C.POINTER(BankConfig), C.POINTER(_P)]),
    "sxgpu_bank_destroy": (C.c_int, [_P]),
    "sxgpu_bank_advance": (C.c_int, [_P, C.c_int64, _P]),
    "sxgpu_bank_read": (C.c_int, [_P, _P, _P]),
    "sxgpu_bank_write": (C.c_int, [_P, _P, C.c_int, _P, C.c_longlong, _P]),
    "sxgpu_bank_repeat": (C.c_int, [_P, _P, C.c_longlong, _P]),
    "sxgpu_bank_repeat_begin": (C.c_int, [_P, _P, _P]),
    "sxgpu_bank_repeat_end": (C.c_int, [_P, _P, C.c_longlong, _P]),
    "sxgpu_bank_ingest": (C.c_int, [_P, C.c_uint32, C.c_uint32, _P, _P]),
    "sxgpu_bank_drain": (C.c_int, [_P, C.c_uint32, C.c_uint32, _S, _P, _P]),
    "sxgpu_bank_device_view": (C.c_int, [_P, _P, _S, C.POINTER(C.c_int)]),
    "sxgpu_bank_last_read": (C.c_int, [_P, _P, _P, _P, _P]),
    "sxgpu_bank_last_write": (C.c_int, [_P, _P, _P]),
    "sxgpu_bank_positions": (C.c_int, [_P, _P, _P, _P, _P]),
    "sxgpu_bank_playback": (C.c_int, [_P, C.c_uint32, C.c_int64, _S, _P, _P]),
    "sxgpu_bank_ring_frames": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "sxgpu_iir_create": (C.c_int, [_P, C.c_uint32, C.c_uint32, _P, C.POINTER(_P)]),
    "sxgpu_iir_destroy": (C.c_int, [_P]),
    "sxgpu_iir_set_state": (C.c_int, [_P, _P, _P]),
    "sxgpu_iir_get_state": (C.c_int, [_P, _P, _P]),
    "sxgpu_iir_apply": (C.c_int, [_P, _P, C.c_uint32, _P]),
    "sxgpu_bank_repeat_filtered": (C.c_int, [_P, _P, _P, _P, C.c_longlong, _P]),
    "sxgpu_bank_read_filtered": (C.c_int, [_P, _P, _P, _P]),
    "sxgpu_bank_write_filtered": (C.c_int, [_P, _P, _P, C.c_int, _P, C.c_longlong, _P]),
    "sxgpu_iir_device_view": (C.c_int, [_P, _P, _S]),
    "sxgpu_convert_rx_buffer_host": (C.c_int, [_P, _P, _S, _P, _S, _S]),
    "sxgpu_convert_rx_buffer_host_gated": (C.c_int, [_P, _P, _S, _P, _S, _S, _P, _P]),
    "sxgpu_convert_tx_buffer_host": (C.c_int, [_P, _P, _S, _P, _S, _S, _F]),
    "sxgpu_convert_rx_buffer_cs16_host": (C.c_int, [_P, _P, _S, _P, _S, _S]),
    "sxgpu_convert_tx_buffer_cs16_host": (C.c_int, [_P, _P, _S, _P, _S, _S, _F]),
    "sxgpu_convert_rx_buffer_s16_host": (C.c_int, [_P, _P, _S, _P, _S, _S]),
    "sxgpu_convert_tx_buffer_s16_host": (C.c_int, [_P, _P, _S, _P, _S, _S, _F]),
    "sxgpu_stats_words": (C.c_int, [_P, _P, _S, C.c_uint64, C.POINTER(Stats), _P]),
    "sxgpu_synth_frames": (C.c_int, [_P, _P, C.c_uint64, _S, C.c_uint64, _P]),
    "sxgpu_malloc": (C.c_int, [_P, C.POINTER(_P), _S]),
    "sxgpu_free": (C.c_int, [_P, _P]),
    "sxgpu_malloc_host": (C.c_int, [_P, C.POINTER(_P), _S]),
    "sxgpu_free_host": (C.c_int, [_P, _P]),
    "sxgpu_host_register": (C.c_int, [_P, _P, _S]),
    "sxgpu_host_unregister": (C.c_int, [_P, _P]),
    "sxgpu_memcpy_h2d": (C.c_int, [_P, _P, _P, _S, _P]),
    "sxgpu_memcpy_d2h": (C.c_int, [_P, _P, _P, _S, _P]),
    "sxgpu_stream_create": (C.c_int, [_P, C.POINTER(_P)]),
    "sxgpu_stream_destroy": (C.c_int, [_P, _P]),
    "sxgpu_stream_sync": (C.c_int, [_P, _P]),
    "sxgpu_multi_create": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(_P)]),
    "sxgpu_multi_destroy": (C.c_int, [_P]),
    "sxgpu_multi_size": (C.c_int, [_P]),
    "sxgpu_multi_context": (_P, [_P, C.c_int]),
    "sxgpu_multi_last_error": (C.c_char_p, [_P]),
    "sxgpu_multi_convert_rx_host": (C.c_int, [_P, _P, C.c_uint32]),
    "sxgpu_multi_convert_tx_host": (C.c_int, [_P, _P, C.c_uint32]),
    "sxgpu_multi_convert_rx_batch": (C.c_int, [_P, _P, C.c_uint32]),
    "sxgpu_multi_convert_tx_batch": (C.c_int, [_P, _P, C.c_uint32]),
    "sxgpu_multi_sync": (C.c_int, [_P]),
    "sxgpu_set_option": (C.c_int, [_P, C.c_char_p, C.c_int64]),
    "sxgpu_get_option": (C.c_int, [_P, C.c_char_p, C.POINTER(C.c_int64)]),
    "sxgpu_get_counter": (C.c_int, [_P, C.c_char_p, C.POINTER(C.c_uint64)]),
}

_lib = None


def library_path() -> Path:
    return _build.GPU_LIB


def load_library(build: bool = True) -> C.CDLL:
    """Load libsxgpu.so (building it in-tree first if it is missing or stale)."""
    global _lib
    if _lib is None:
        path = _build.build_gpu_library() if build else _build.GPU_LIB
        if not Path(path).exists():
            raise RuntimeError(f"{path} is missing: build it with __graft_entry__.build(); there is no CPU fallback")
        lib = C.CDLL(str(path))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError here = header and library disagree
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


class Context:
    """One sxgpu context = one GPU.  Thin, checked wrappers over the C ABI."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = _P()
        rc = self.lib.sxgpu_init(device, C.byref(h))
        if rc != SXGPU_OK:
            raise SxGpuError(rc, "sxgpu_init", self.lib.sxgpu_strerror(rc).decode())
        self.handle = h
        self.device = device

    def close(self):
        if self.handle:
            self.lib.sxgpu_destroy(self.handle)
            self.handle = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def check(self, rc: int, what: str) -> None:
        if rc != SXGPU_OK:
            raise SxGpuError(rc, what, self.lib.sxgpu_last_error(self.handle).decode())

    # -- hot path, device pointers (ints, e.g. torch.Tensor.data_ptr()) ---------------------
    def convert_rx_buffer(self, d_src, src_offset, d_dest, dest_offset, length, stream=None):
        self.check(self.lib.sxgpu_convert_rx_buffer(self.handle, d_src, src_offset, d_dest, dest_offset, length, stream),
                   "sxgpu_convert_rx_buffer")

    def convert_tx_buffer(self, d_src, src_offset, d_dest, dest_offset, length, tx_threshold2, stream=None):
        self.check(self.lib.sxgpu_convert_tx_buffer(self.handle, d_src, src_offset, d_dest, dest_offset, length,
                                                    tx_threshold2, stream), "sxgpu_convert_tx_buffer")

    def convert_rx_buffer_cs16(self, d_src, src_offset, d_dest, dest_offset, length, stream=None):
        self.check(self.lib.sxgpu_convert_rx_buffer_cs16(self.handle, d_src, src_offset, d_dest, dest_offset, length,
                                                         stream), "sxgpu_convert_rx_buffer_cs16")

    def convert_tx_buffer_cs16(self, d_src, src_offset, d_dest, dest_offset, length, tx_threshold2, stream=None):
        self.check(self.lib.sxgpu_convert_tx_buffer_cs16(self.handle, d_src, src_offset, d_dest, dest_offset, length,
                                                         tx_threshold2, stream), "sxgpu_convert_tx_buffer_cs16")

    def convert_rx_buffer_s16(self, d_src, src_offset, d_dest, dest_offset, length, stream=None):
        self.check(self.lib.sxgpu_convert_rx_buffer_s16(self.handle, d_src, src_offset, d_dest, dest_offset, length,
                                                        stream), "sxgpu_convert_rx_buffer_s16")

    def convert_tx_buffer_s16(self, d_src, src_offset, d_dest, dest_offset, length, tx_threshold2, stream=None):
        self.check(self.lib.sxgpu_convert_tx_buffer_s16(self.handle, d_src, src_offset, d_dest, dest_offset, length,
                                                        tx_threshold2, stream), "sxgpu_convert_tx_buffer_s16")

    def convert_batch(self, direction: str, blocks, on_device=False, max_length=0, stream=None, nblocks=None):
        fn = self.lib.sxgpu_convert_rx_batch if direction == "rx" else self.lib.sxgpu_convert_tx_batch
        if on_device:
            ptr, n = blocks, nblocks
        else:
            arr = (Block * len(blocks))(*blocks)
            ptr, n = C.cast(arr, _P), len(blocks)
        self.check(fn(self.handle, ptr, n, 1 if on_device else 0, max_length, stream), f"sxgpu_convert_{direction}_batch")

    def convert_loopback(self, d_i2s_in, d_cf32, d_i2s_out, length, tx_threshold2, stream=None):
        self.check(self.lib.sxgpu_convert_loopback(self.handle, d_i2s_in, d_cf32, d_i2s_out, length, tx_threshold2,
                                                   stream), "sxgpu_convert_loopback")

    def fill_silence(self, d_i2s, offset, length, stream=None):
        self.check(self.lib.sxgpu_fill_silence(self.handle, d_i2s, offset, length, stream), "sxgpu_fill_silence")

    # -- hot path, host pointers ---------------------------------------------------------------
    def convert_rx_buffer_host(self, h_src, src_offset, h_dest, dest_offset, length):
        self.check(self.lib.sxgpu_convert_rx_buffer_host(self.handle, h_src, src_offset, h_dest, dest_offset, length),
                   "sxgpu_convert_rx_buffer_host")

    def convert_tx_buffer_host(self, h_src, src_offset, h_dest, dest_offset, length, tx_threshold2):
        self.check(self.lib.sxgpu_convert_tx_buffer_host(self.handle, h_src, src_offset, h_dest, dest_offset, length,
                                                         tx_threshold2), "sxgpu_convert_tx_buffer_host")

    def convert_rx_buffer_cs16_host(self, h_src, src_offset, h_dest, dest_offset, length):
        self.check(self.lib.sxgpu_convert_rx_buffer_cs16_host(self.handle, h_src, src_offset, h_dest, dest_offset,
                                                              length), "sxgpu_convert_rx_buffer_cs16_host")

    def convert_tx_buffer_cs16_host(self, h_src, src_offset, h_dest, dest_offset, length, tx_threshold2):
        self.check(self.lib.sxgpu_convert_tx_buffer_cs16_host(self.handle, h_src, src_offset, h_dest, dest_offset,
                                                              length, tx_threshold2), "sxgpu_convert_tx_buffer_cs16_host")

    def convert_rx_buffer_s16_host(self, h_src, src_offset, h_dest, dest_offset, length):
        self.check(self.lib.sxgpu_convert_rx_buffer_s16_host(self.handle, h_src, src_offset, h_dest, dest_offset,
                                                             length), "sxgpu_convert_rx_buffer_s16_host")

    def convert_tx_buffer_s16_host(self, h_src, src_offset, h_dest, dest_offset, length, tx_threshold2):
        self.check(self.lib.sxgpu_convert_tx_buffer_s16_host(self.handle, h_src, src_offset, h_dest, dest_offset,
                                                             length, tx_threshold2), "sxgpu_convert_tx_buffer_s16_host")

    # -- statistics, synthetic source -----------------------------------------------------------
    def stats_words(self, d_words, nwords, base_index=0, stream=None):
        out = Stats()
        self.check(self.lib.sxgpu_stats_words(self.handle, d_words, nwords, base_index, C.byref(out), stream),
                   "sxgpu_stats_words")
        return out.as_tuple()

    def synth_frames(self, d_i2s, first_frame, nframes, seed, stream=None):
        self.check(self.lib.sxgpu_synth_frames(self.handle, d_i2s, first_frame, nframes, seed, stream),
                   "sxgpu_synth_frames")

    # -- plumbing ----------------------------------------------------------------------------------
    def malloc(self, nbytes):
        p = _P()
        self.check(self.lib.sxgpu_malloc(self.handle, C.byref(p), nbytes), "sxgpu_malloc")
        return p.value

    def free(self, d_ptr):
        self.check(self.lib.sxgpu_free(self.handle, d_ptr), "sxgpu_free")

    def malloc_host(self, nbytes):
        p = _P()
        self.check(self.lib.sxgpu_malloc_host(self.handle, C.byref(p), nbytes), "sxgpu_malloc_host")
        return p.value

    def free_host(self, h_ptr):
        self.check(self.lib.sxgpu_free_host(self.handle, h_ptr), "sxgpu_free_host")

    def memcpy_h2d(self, d_dst, h_src, nbytes, stream=None):
        self.check(self.lib.sxgpu_memcpy_h2d(self.handle, d_dst, h_src, nbytes, stream), "sxgpu_memcpy_h2d")

    def memcpy_d2h(self, h_dst, d_src, nbytes, stream=None):
        self.check(self.lib.sxgpu_memcpy_d2h(self.handle, h_dst, d_src, nbytes, stream), "sxgpu_memcpy_d2h")

    def stream_sync(self, stream=None):
        self.check(self.lib.sxgpu_stream_sync(self.handle, stream), "sxgpu_stream_sync")

    def set_option(self, key: str, value: int):
        self.check(self.lib.sxgpu_set_option(self.handle, key.encode(), value), f"sxgpu_set_option({key})")

    def get_option(self, key: str) -> int:
        v = C.c_int64()
        self.check(self.lib.sxgpu_get_option(self.handle, key.encode(), C.byref(v)), f"sxgpu_get_option({key})")
        return v.value

    def counter(self, key: str) -> int:
        v = C.c_uint64()
        self.check(self.lib.sxgpu_get_counter(self.handle, key.encode(), C.byref(v)), f"sxgpu_get_counter({key})")
        return v.value

    def info(self) -> Info:
        out = Info()
        self.check(self.lib.sxgpu_device_info(self.handle, C.byref(out)), "sxgpu_device_info")
        return out


class Bank:
    """A bank of HBM-resident stream pairs (sxgpu_bank_* in include/sxgpu.h)."""

    def __init__(self, ctx: Context, nstreams: int, period: int = 0, sample_rate: float = 75000.0,
                 tx_threshold2: float = 1.0e-6, seed: int = 0x53581255):
        import numpy as np
        self.np = np
        self.ctx, self.lib = ctx, ctx.lib
        cfg = BankConfig(nstreams, period, sample_rate, tx_threshold2, 0, seed)
        h = _P()
        ctx.check(self.lib.sxgpu_bank_create(ctx.handle, C.byref(cfg), C.byref(h)), "sxgpu_bank_create")
        self.handle, self.nstreams = h, nstreams
        r = C.c_uint64()
        self.lib.sxgpu_bank_ring_frames(h, C.byref(r))
        self.ring = r.value
        self.period = period if 0 < period <= 65536 else (256 if period == 0 else 65536)

    def close(self):
        if self.handle:
            self.lib.sxgpu_bank_destroy(self.handle)
            self.handle = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def advance(self, frames, stream=None):
        self.ctx.check(self.lib.sxgpu_bank_advance(self.handle, frames, stream), "sxgpu_bank_advance")

    def read(self, d_cf32, stream=None):
        self.ctx.check(self.lib.sxgpu_bank_read(self.handle, d_cf32, stream), "sxgpu_bank_read")

    def write(self, d_cf32, flags=4, d_time_ns=None, rx_time_offset_ns=0, stream=None):
        self.ctx.check(self.lib.sxgpu_bank_write(self.handle, d_cf32, flags, d_time_ns, rx_time_offset_ns, stream),
                       "sxgpu_bank_write")

    def repeat(self, d_cf32, rx_time_offset_ns=0, stream=None):
        """read(d_cf32) then write(d_cf32, HAS_TIME, rx time + offset) in one launch."""
        self.ctx.check(self.lib.sxgpu_bank_repeat(self.handle, d_cf32, rx_time_offset_ns, stream), "sxgpu_bank_repeat")

    def repeat_filtered(self, d_cf32, pre: "Iir | None" = None, post: "Iir | None" = None, rx_time_offset_ns=0,
                        stream=None):
        """repeat() with the channel filters: read, `pre` filter, `post` filter, timed write, in one
        iteration that carries both filters' state (either may be None)."""
        self.ctx.check(self.lib.sxgpu_bank_repeat_filtered(self.handle, pre.handle if pre else None,
                                                           post.handle if post else None, d_cf32, rx_time_offset_ns,
                                                           stream), "sxgpu_bank_repeat_filtered")

    def read_filtered(self, d_cf32, f: "Iir | None", stream=None):
        """read(d_cf32) then f.apply(d_cf32, period) in one pass (f None: read)."""
        self.ctx.check(self.lib.sxgpu_bank_read_filtered(self.handle, f.handle if f else None, d_cf32, stream),
                       "sxgpu_bank_read_filtered")

    def write_filtered(self, d_cf32, f: "Iir | None", flags=4, d_time_ns=None, rx_time_offset_ns=0, stream=None):
        """write() of d_cf32 filtered by f, in one pass that leaves d_cf32 as it was (f None: write)."""
        self.ctx.check(self.lib.sxgpu_bank_write_filtered(self.handle, f.handle if f else None, d_cf32, flags, d_time_ns,
                                                          rx_time_offset_ns, stream), "sxgpu_bank_write_filtered")

    def repeat_begin(self, d_cf32, stream=None):
        self.ctx.check(self.lib.sxgpu_bank_repeat_begin(self.handle, d_cf32, stream), "sxgpu_bank_repeat_begin")

    def repeat_end(self, d_cf32, rx_time_offset_ns=0, stream=None):
        self.ctx.check(self.lib.sxgpu_bank_repeat_end(self.handle, d_cf32, rx_time_offset_ns, stream),
                       "sxgpu_bank_repeat_end")

    def ingest(self, first_stream, nstreams, i2s, stream=None):
        """One period of I2S frames per stream from outside (host or device address)."""
        self.ctx.check(self.lib.sxgpu_bank_ingest(self.handle, first_stream, nstreams, i2s, stream), "sxgpu_bank_ingest")

    def drain(self, first_stream, nstreams, nframes, i2s, stream=None):
        """The last nframes frames each stream wrote, to a device or pinned-host address."""
        self.ctx.check(self.lib.sxgpu_bank_drain(self.handle, first_stream, nstreams, nframes, i2s, stream),
                       "sxgpu_bank_drain")

    def last_read(self, stream=None):
        np = self.np
        ret, fl, t = np.empty(self.nstreams, np.int32), np.empty(self.nstreams, np.int32), np.empty(self.nstreams, np.int64)
        self.ctx.check(self.lib.sxgpu_bank_last_read(self.handle, ret.ctypes.data, fl.ctypes.data, t.ctypes.data, stream),
                       "sxgpu_bank_last_read")
        return ret, fl, t

    def last_write(self, stream=None):
        ret = self.np.empty(self.nstreams, self.np.int32)
        self.ctx.check(self.lib.sxgpu_bank_last_write(self.handle, ret.ctypes.data, stream), "sxgpu_bank_last_write")
        return ret

    def positions(self, stream=None):
        np = self.np
        c, r, t = (np.empty(self.nstreams, np.int64) for _ in range(3))
        self.ctx.check(self.lib.sxgpu_bank_positions(self.handle, c.ctypes.data, r.ctypes.data, t.ctypes.data, stream),
                       "sxgpu_bank_positions")
        return c, r, t

    def playback(self, index, position, nframes, stream=None):
        out = self.np.empty(2 * nframes, self.np.int32)
        self.ctx.check(self.lib.sxgpu_bank_playback(self.handle, index, position, nframes, out.ctypes.data, stream),
                       "sxgpu_bank_playback")
        return out


class Iir:
    """A cascade of second-order sections with one state per stream (sxgpu_iir_* in include/sxgpu.h):
    scipy.signal.sosfilt(sos, x, zi=state) along each stream's block, carried from call to call.
    `sos` is what scipy's filter design functions return with output="sos": (nsections, 6)."""

    def __init__(self, ctx: Context, nstreams: int, sos):
        import numpy as np
        self.np = np
        self.ctx, self.lib = ctx, ctx.lib
        self.handle = None
        sos = np.ascontiguousarray(np.asarray(sos, dtype=np.float64))
        if sos.ndim != 2 or sos.shape[1] != 6:
            raise ValueError(f"sos must have shape (nsections, 6), got {sos.shape}")
        h = _P()
        ctx.check(self.lib.sxgpu_iir_create(ctx.handle, nstreams, sos.shape[0], sos.ctypes.data, C.byref(h)),
                  "sxgpu_iir_create")
        self.handle, self.nstreams, self.nsections = h, nstreams, sos.shape[0]

    def close(self):
        if self.handle:
            self.lib.sxgpu_iir_destroy(self.handle)
            self.handle = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def apply(self, d_cf32, period, stream=None):
        """Filter d_cf32[nstreams][period] (complex64 on the device) in place."""
        self.ctx.check(self.lib.sxgpu_iir_apply(self.handle, d_cf32, period, stream), "sxgpu_iir_apply")

    def state(self, stream=None):
        """The state as scipy's zf: (nsections, nstreams, 2) complex64."""
        zf = self.np.empty((self.nsections, self.nstreams, 2), self.np.complex64)
        self.ctx.check(self.lib.sxgpu_iir_get_state(self.handle, zf.ctypes.data, stream), "sxgpu_iir_get_state")
        return zf

    def set_state(self, zi=None, stream=None):
        """Set the state from scipy's zi layout, (nsections, nstreams, 2); None = zeros."""
        ptr = None
        if zi is not None:
            zi = self.np.ascontiguousarray(zi, dtype=self.np.complex64)
            if zi.shape != (self.nsections, self.nstreams, 2):
                raise ValueError(f"zi must have shape {(self.nsections, self.nstreams, 2)}, got {zi.shape}")
            ptr = zi.ctypes.data
        self.ctx.check(self.lib.sxgpu_iir_set_state(self.handle, ptr, stream), "sxgpu_iir_set_state")


class Multi:
    """Several GPUs from one process (sxgpu_multi_* in include/sxgpu.h): one context and one host
    thread per GPU, block lists split between them, no collective."""

    def __init__(self, devices):
        self.lib = load_library()
        arr = (C.c_int * len(devices))(*devices)
        h = _P()
        rc = self.lib.sxgpu_multi_create(arr, len(devices), C.byref(h))
        if rc != SXGPU_OK:
            raise SxGpuError(rc, "sxgpu_multi_create", self.lib.sxgpu_strerror(rc).decode())
        self.handle, self.devices = h, list(devices)

    def close(self):
        if self.handle:
            self.lib.sxgpu_multi_destroy(self.handle)
            self.handle = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def check(self, rc, what):
        if rc != SXGPU_OK:
            raise SxGpuError(rc, what, self.lib.sxgpu_multi_last_error(self.handle).decode())

    def context(self, index: int) -> "Context":
        """The index-th GPU's own context (owned by the Multi: do not close it)."""
        c = Context.__new__(Context)
        c.lib, c.handle, c.device = self.lib, _P(self.lib.sxgpu_multi_context(self.handle, index)), self.devices[index]
        return c

    def _call(self, fn, blocks, what):
        arr = (Block * len(blocks))(*blocks)
        self.check(fn(self.handle, C.cast(arr, _P), len(blocks)), what)

    def convert_rx_host(self, blocks):
        self._call(self.lib.sxgpu_multi_convert_rx_host, blocks, "sxgpu_multi_convert_rx_host")

    def convert_tx_host(self, blocks):
        self._call(self.lib.sxgpu_multi_convert_tx_host, blocks, "sxgpu_multi_convert_tx_host")

    def convert_rx_batch(self, blocks):
        self._call(self.lib.sxgpu_multi_convert_rx_batch, blocks, "sxgpu_multi_convert_rx_batch")

    def convert_tx_batch(self, blocks):
        self._call(self.lib.sxgpu_multi_convert_tx_batch, blocks, "sxgpu_multi_convert_tx_batch")

    def sync(self):
        self.check(self.lib.sxgpu_multi_sync(self.handle), "sxgpu_multi_sync")
