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
    "sxgpu_iir_apply_long": (C.c_int, [_P, _P, C.c_uint64, _P]),
    "sxgpu_bank_repeat_filtered": (C.c_int, [_P, _P, _P, _P, C.c_longlong, _P]),
    "sxgpu_bank_read_filtered": (C.c_int, [_P, _P, _P, _P]),
    "sxgpu_bank_write_filtered": (C.c_int, [_P, _P, _P, C.c_int, _P, C.c_longlong, _P]),
    "sxgpu_iir_device_view": (C.c_int, [_P, _P, _S]),
    "sxgpu_fir_create": (C.c_int, [_P, C.c_uint32, C.c_uint32, _P, C.c_uint32, C.c_uint32, C.POINTER(_P)]),
    "sxgpu_fir_destroy": (C.c_int, [_P]),
    "sxgpu_fir_output_frames": (C.c_int, [_P, C.c_uint64, C.POINTER(C.c_uint64)]),
    "sxgpu_fir_apply": (C.c_int, [_P, _P, C.c_uint64, _P, C.POINTER(C.c_uint64), _P]),
    "sxgpu_fir_get_state": (C.c_int, [_P, _P, C.POINTER(C.c_uint32), _P]),
    "sxgpu_fir_set_state": (C.c_int, [_P, _P, C.c_uint32, _P]),
    "sxgpu_bank_read_fir": (C.c_int, [_P, _P, _P, C.POINTER(C.c_uint64), _P]),
    "sxgpu_bank_write_fir": (C.c_int, [_P, _P, _P, C.c_uint64, C.c_int, _P, C.c_longlong, _P]),
    "sxgpu_nco_create": (C.c_int, [_P, C.c_uint32, _P, C.POINTER(_P)]),
    "sxgpu_nco_destroy": (C.c_int, [_P]),
    "sxgpu_nco_apply": (C.c_int, [_P, _P, C.c_uint64, _P]),
    "sxgpu_nco_set_frequencies": (C.c_int, [_P, _P, _P]),
    "sxgpu_nco_get_state": (C.c_int, [_P, _P, _P, _P]),
    "sxgpu_nco_set_state": (C.c_int, [_P, _P, _P, _P]),
    "sxgpu_bank_read_ddc": (C.c_int, [_P, _P, _P, _P, C.POINTER(C.c_uint64), _P]),
    "sxgpu_bank_write_duc": (C.c_int, [_P, _P, _P, _P, C.c_uint64, C.c_int, _P, C.c_longlong, _P]),
    "sxgpu_chan_create": (C.c_int, [_P, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, _P, C.POINTER(_P)]),
    "sxgpu_chan_destroy": (C.c_int, [_P]),
    "sxgpu_chan_output_frames": (C.c_int, [_P, C.c_uint64, C.POINTER(C.c_uint64)]),
    "sxgpu_chan_apply": (C.c_int, [_P, _P, C.c_uint64, _P, C.POINTER(C.c_uint64), _P]),
    "sxgpu_chan_get_state": (C.c_int, [_P, _P, C.POINTER(C.c_uint32), _P]),
    "sxgpu_chan_set_state": (C.c_int, [_P, _P, C.c_uint32, _P]),
    "sxgpu_chan_synth_create": (C.c_int, [_P, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, _P, C.POINTER(_P)]),
    "sxgpu_chan_synth_destroy": (C.c_int, [_P]),
    "sxgpu_chan_synth_apply": (C.c_int, [_P, _P, C.c_uint64, _P, _P]),
    "sxgpu_chan_synth_get_state": (C.c_int, [_P, _P, C.POINTER(C.c_uint32), _P]),
    "sxgpu_chan_synth_set_state": (C.c_int, [_P, _P, C.c_uint32, _P]),
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


class _Owned:
    """An object behind a C handle: `close` (also on leaving a `with` block) frees it with the type's
    destroy function, named by `_destroy`, once."""

    handle = None
    _destroy = ""

    def close(self):
        if self.handle:
            getattr(self.lib, self._destroy)(self.handle)
            self.handle = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class Context(_Owned):
    """One sxgpu context = one GPU.  Thin, checked wrappers over the C ABI."""

    _destroy = "sxgpu_destroy"

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = _P()
        rc = self.lib.sxgpu_init(device, C.byref(h))
        if rc != SXGPU_OK:
            raise SxGpuError(rc, "sxgpu_init", self.lib.sxgpu_strerror(rc).decode())
        self.handle = h
        self.device = device

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


class Bank(_Owned):
    """A bank of HBM-resident stream pairs (sxgpu_bank_* in include/sxgpu.h)."""

    _destroy = "sxgpu_bank_destroy"

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

    def read_fir(self, f: "Fir", d_out, stream=None) -> int:
        """read() then f.apply(that block, period, d_out) in one call, without the full-rate block;
        returns nout, the frames per stream written to d_out."""
        n = C.c_uint64()
        self.ctx.check(self.lib.sxgpu_bank_read_fir(self.handle, f.handle if f else None, d_out, C.byref(n), stream),
                       "sxgpu_bank_read_fir")
        return n.value

    def write_fir(self, f: "Fir", d_in, nin, flags=4, d_time_ns=None, rx_time_offset_ns=0, stream=None):
        """write() of f.apply(d_in, nin), which must be one period, in one call that leaves d_in as it was."""
        self.ctx.check(self.lib.sxgpu_bank_write_fir(self.handle, f.handle if f else None, d_in, nin, flags, d_time_ns,
                                                     rx_time_offset_ns, stream), "sxgpu_bank_write_fir")

    def read_ddc(self, nco: "Nco", f: "Fir", d_out, stream=None) -> int:
        """read(), nco.apply(that block, period), then f.apply(it, period, d_out) in one call, without
        the full-rate block; returns nout, the frames per stream written to d_out."""
        n = C.c_uint64()
        self.ctx.check(self.lib.sxgpu_bank_read_ddc(self.handle, nco.handle if nco else None, f.handle if f else None,
                                                    d_out, C.byref(n), stream), "sxgpu_bank_read_ddc")
        return n.value

    def write_duc(self, f: "Fir", nco: "Nco", d_in, nin, flags=4, d_time_ns=None, rx_time_offset_ns=0, stream=None):
        """write() of nco.apply(f.apply(d_in, nin), period), in one call that leaves d_in as it was."""
        self.ctx.check(self.lib.sxgpu_bank_write_duc(self.handle, f.handle if f else None, nco.handle if nco else None,
                                                     d_in, nin, flags, d_time_ns, rx_time_offset_ns, stream),
                       "sxgpu_bank_write_duc")

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


class Iir(_Owned):
    """A cascade of second-order sections with one state per stream (sxgpu_iir_* in include/sxgpu.h):
    scipy.signal.sosfilt(sos, x, zi=state) along each stream's block, carried from call to call.
    `sos` is what scipy's filter design functions return with output="sos": (nsections, 6)."""

    _destroy = "sxgpu_iir_destroy"

    def __init__(self, ctx: Context, nstreams: int, sos):
        import numpy as np
        self.np = np
        self.ctx, self.lib = ctx, ctx.lib
        sos = np.ascontiguousarray(np.asarray(sos, dtype=np.float64))
        if sos.ndim != 2 or sos.shape[1] != 6:
            raise ValueError(f"sos must have shape (nsections, 6), got {sos.shape}")
        h = _P()
        ctx.check(self.lib.sxgpu_iir_create(ctx.handle, nstreams, sos.shape[0], sos.ctypes.data, C.byref(h)),
                  "sxgpu_iir_create")
        self.handle, self.nstreams, self.nsections = h, nstreams, sos.shape[0]

    def apply(self, d_cf32, period, stream=None):
        """Filter d_cf32[nstreams][period] (complex64 on the device) in place."""
        self.ctx.check(self.lib.sxgpu_iir_apply(self.handle, d_cf32, period, stream), "sxgpu_iir_apply")

    def apply_long(self, d_cf32, nframes, stream=None):
        """Filter d_cf32[nstreams][nframes] in place for any nframes, in parallel along the block: bit
        for bit `apply` on each stream's first chunk, within float32 rounding of it after that
        (sxgpu_iir_apply_long in include/sxgpu.h)."""
        self.ctx.check(self.lib.sxgpu_iir_apply_long(self.handle, d_cf32, nframes, stream), "sxgpu_iir_apply_long")

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


class Fir(_Owned):
    """Real FIR taps with an up/down rate change and one history per stream (sxgpu_fir_* in
    include/sxgpu.h): scipy.signal.upfirdn(taps, x, up, down) on each stream's concatenated input,
    bit for bit, carried from call to call.  up = down = 1 is a plain FIR filter."""

    _destroy = "sxgpu_fir_destroy"

    def __init__(self, ctx: Context, nstreams: int, taps, up: int = 1, down: int = 1):
        import numpy as np
        self.np = np
        self.ctx, self.lib = ctx, ctx.lib
        taps = np.ascontiguousarray(np.asarray(taps, dtype=np.float64))
        if taps.ndim != 1:
            raise ValueError(f"taps must be one-dimensional, got shape {taps.shape}")
        h = _P()
        ctx.check(self.lib.sxgpu_fir_create(ctx.handle, nstreams, taps.size, taps.ctypes.data if taps.size else None,
                                            up, down, C.byref(h)), "sxgpu_fir_create")
        self.handle, self.nstreams, self.ntaps, self.up, self.down = h, nstreams, taps.size, up, down
        self.hp = -(-taps.size // up)

    def output_frames(self, nin) -> int:
        """Frames each stream's next apply of nin frames emits."""
        n = C.c_uint64()
        self.ctx.check(self.lib.sxgpu_fir_output_frames(self.handle, nin, C.byref(n)), "sxgpu_fir_output_frames")
        return n.value

    def apply(self, d_in, nin, d_out, stream=None) -> int:
        """d_in[nstreams][nin] -> d_out[nstreams][nout] (complex64 on the device); returns nout."""
        n = C.c_uint64()
        self.ctx.check(self.lib.sxgpu_fir_apply(self.handle, d_in, nin, d_out, C.byref(n), stream), "sxgpu_fir_apply")
        return n.value

    def state(self, stream=None):
        """(history, phase): the last hp - 1 inputs of each stream, (nstreams, hp - 1) complex64 oldest
        first, and the frames fed so far mod down."""
        hist = self.np.empty((self.nstreams, self.hp - 1), self.np.complex64)
        phase = C.c_uint32()
        self.ctx.check(self.lib.sxgpu_fir_get_state(self.handle, hist.ctypes.data, C.byref(phase), stream),
                       "sxgpu_fir_get_state")
        return hist, phase.value

    def set_state(self, hist=None, phase=0, stream=None):
        """Set the history, (nstreams, hp - 1) complex64 (None = zeros), and the phase."""
        ptr = None
        if hist is not None:
            hist = self.np.ascontiguousarray(hist, dtype=self.np.complex64)
            if hist.shape != (self.nstreams, self.hp - 1):
                raise ValueError(f"hist must have shape {(self.nstreams, self.hp - 1)}, got {hist.shape}")
            ptr = hist.ctypes.data
        self.ctx.check(self.lib.sxgpu_fir_set_state(self.handle, ptr, phase, stream), "sxgpu_fir_set_state")


class Nco(_Owned):
    """One numerically controlled oscillator per stream (sxgpu_nco_* in include/sxgpu.h): each
    frame multiplied by exp(+2j pi phase / 2^32), the 32-bit phase advancing by the increment
    rint(f 2^32) per frame, carried from call to call.  `freqs` in cycles per sample, -0.5 .. 0.5
    (None: all 0); to bring a channel at +f0 to DC, use -f0."""

    _destroy = "sxgpu_nco_destroy"

    def __init__(self, ctx: Context, nstreams: int, freqs=None):
        import numpy as np
        self.np = np
        self.ctx, self.lib = ctx, ctx.lib
        f = self._freqs(nstreams, freqs)
        h = _P()
        ctx.check(self.lib.sxgpu_nco_create(ctx.handle, nstreams, f.ctypes.data if f is not None else None, C.byref(h)),
                  "sxgpu_nco_create")
        self.handle, self.nstreams = h, nstreams

    def _freqs(self, nstreams, freqs):
        if freqs is None:
            return None
        return self.np.ascontiguousarray(self.np.broadcast_to(self.np.asarray(freqs, dtype=self.np.float64), (nstreams,)))

    def apply(self, d_cf32, nframes, stream=None):
        """Mix d_cf32[nstreams][nframes] (complex64 on the device) in place."""
        self.ctx.check(self.lib.sxgpu_nco_apply(self.handle, d_cf32, nframes, stream), "sxgpu_nco_apply")

    def set_frequencies(self, freqs, stream=None):
        """Retune every stream (one frequency, or one per stream; None: all 0), the phases kept."""
        f = self._freqs(self.nstreams, freqs)
        self.ctx.check(self.lib.sxgpu_nco_set_frequencies(self.handle, f.ctypes.data if f is not None else None, stream),
                       "sxgpu_nco_set_frequencies")

    def state(self, stream=None):
        """(phases, increments), each (nstreams,) uint32."""
        ph, inc = self.np.empty(self.nstreams, self.np.uint32), self.np.empty(self.nstreams, self.np.uint32)
        self.ctx.check(self.lib.sxgpu_nco_get_state(self.handle, ph.ctypes.data, inc.ctypes.data, stream),
                       "sxgpu_nco_get_state")
        return ph, inc

    def set_state(self, phases=None, incs=None, stream=None):
        """Set the phases and/or the increments, (nstreams,) uint32 each; None leaves that one as it is."""
        ptrs = []
        for a in (phases, incs):
            if a is None:
                ptrs.append((None, None))
                continue
            a = self.np.ascontiguousarray(a, dtype=self.np.uint32)
            if a.shape != (self.nstreams,):
                raise ValueError(f"phases and incs must have shape {(self.nstreams,)}, got {a.shape}")
            ptrs.append((a, a.ctypes.data))
        self.ctx.check(self.lib.sxgpu_nco_set_state(self.handle, ptrs[0][1], ptrs[1][1], stream), "sxgpu_nco_set_state")


class Chan(_Owned):
    """A polyphase DFT channelizer per stream (sxgpu_chan_* in include/sxgpu.h): each stream split
    into `channels` channel-rate streams, channel k centred at k / channels cycles per sample (numpy's
    fft order), low-passed by the real prototype `taps` and decimated by `down` (default: channels,
    critically sampled), the last inputs carried from call to call."""

    _destroy = "sxgpu_chan_destroy"

    def __init__(self, ctx: Context, nstreams: int, taps, channels: int, down: int | None = None):
        import numpy as np
        self.np = np
        self.ctx, self.lib = ctx, ctx.lib
        down = channels if down is None else down
        taps = np.ascontiguousarray(np.asarray(taps, dtype=np.float64))
        if taps.ndim != 1:
            raise ValueError(f"taps must be one-dimensional, got shape {taps.shape}")
        h = _P()
        ctx.check(self.lib.sxgpu_chan_create(ctx.handle, nstreams, channels, down, taps.size,
                                             taps.ctypes.data if taps.size else None, C.byref(h)), "sxgpu_chan_create")
        self.handle, self.nstreams, self.ntaps, self.channels, self.down = h, nstreams, taps.size, channels, down

    def output_frames(self, nin) -> int:
        """Frames each channel's next apply of nin frames emits."""
        n = C.c_uint64()
        self.ctx.check(self.lib.sxgpu_chan_output_frames(self.handle, nin, C.byref(n)), "sxgpu_chan_output_frames")
        return n.value

    def apply(self, d_in, nin, d_out, stream=None) -> int:
        """d_in[nstreams][nin] -> d_out[nstreams][channels][nout] (complex64 on the device); returns nout."""
        n = C.c_uint64()
        self.ctx.check(self.lib.sxgpu_chan_apply(self.handle, d_in, nin, d_out, C.byref(n), stream), "sxgpu_chan_apply")
        return n.value

    def state(self, stream=None):
        """(history, phase): the last ntaps - 1 inputs of each stream, (nstreams, ntaps - 1) complex64
        oldest first, and the frames fed so far mod channels."""
        hist = self.np.empty((self.nstreams, self.ntaps - 1), self.np.complex64)
        phase = C.c_uint32()
        self.ctx.check(self.lib.sxgpu_chan_get_state(self.handle, hist.ctypes.data, C.byref(phase), stream),
                       "sxgpu_chan_get_state")
        return hist, phase.value

    def set_state(self, hist=None, phase=0, stream=None):
        """Set the history, (nstreams, ntaps - 1) complex64 (None = zeros), and the phase."""
        ptr = None
        if hist is not None:
            hist = self.np.ascontiguousarray(hist, dtype=self.np.complex64)
            if hist.shape != (self.nstreams, self.ntaps - 1):
                raise ValueError(f"hist must have shape {(self.nstreams, self.ntaps - 1)}, got {hist.shape}")
            ptr = hist.ctypes.data
        self.ctx.check(self.lib.sxgpu_chan_set_state(self.handle, ptr, phase, stream), "sxgpu_chan_set_state")


class ChanSynth(_Owned):
    """A polyphase synthesis channelizer per stream (sxgpu_chan_synth_* in include/sxgpu.h): the
    `channels` channel-rate streams of each stream, in Chan.apply's layout, interpolated by `up`
    (default: channels, critically sampled) with the real prototype `taps`, channel k moved to
    k / channels cycles per output sample (numpy's fft order) and summed into one stream, the last
    inputs carried from call to call."""

    _destroy = "sxgpu_chan_synth_destroy"

    def __init__(self, ctx: Context, nstreams: int, taps, channels: int, up: int | None = None):
        import numpy as np
        self.np = np
        self.ctx, self.lib = ctx, ctx.lib
        up = channels if up is None else up
        taps = np.ascontiguousarray(np.asarray(taps, dtype=np.float64))
        if taps.ndim != 1:
            raise ValueError(f"taps must be one-dimensional, got shape {taps.shape}")
        h = _P()
        ctx.check(self.lib.sxgpu_chan_synth_create(ctx.handle, nstreams, channels, up, taps.size,
                                                   taps.ctypes.data if taps.size else None, C.byref(h)),
                  "sxgpu_chan_synth_create")
        self.handle, self.nstreams, self.ntaps, self.channels, self.up = h, nstreams, taps.size, channels, up
        self.hp = -(-taps.size // up)

    def apply(self, d_in, nin, d_out, stream=None):
        """d_in[nstreams][channels][nin] -> d_out[nstreams][nin * up] (complex64 on the device)."""
        self.ctx.check(self.lib.sxgpu_chan_synth_apply(self.handle, d_in, nin, d_out, stream), "sxgpu_chan_synth_apply")

    def state(self, stream=None):
        """(history, phase): each channel's last hp - 1 inputs, (nstreams, channels, hp - 1) complex64
        oldest first, and the input frames fed so far mod channels / up."""
        hist = self.np.empty((self.nstreams, self.channels, self.hp - 1), self.np.complex64)
        phase = C.c_uint32()
        self.ctx.check(self.lib.sxgpu_chan_synth_get_state(self.handle, hist.ctypes.data, C.byref(phase), stream),
                       "sxgpu_chan_synth_get_state")
        return hist, phase.value

    def set_state(self, hist=None, phase=0, stream=None):
        """Set the history, (nstreams, channels, hp - 1) complex64 (None = zeros), and the phase."""
        ptr = None
        if hist is not None:
            hist = self.np.ascontiguousarray(hist, dtype=self.np.complex64)
            shape = (self.nstreams, self.channels, self.hp - 1)
            if hist.shape != shape:
                raise ValueError(f"hist must have shape {shape}, got {hist.shape}")
            ptr = hist.ctypes.data
        self.ctx.check(self.lib.sxgpu_chan_synth_set_state(self.handle, ptr, phase, stream), "sxgpu_chan_synth_set_state")


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
