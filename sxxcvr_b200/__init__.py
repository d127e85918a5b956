"""sxxcvr_b200 -- B200-native IQ sample path for the SoapySX (SX1255) driver.

The product is native: CUDA kernels behind the C ABI of include/sxgpu.h (lib/libsxgpu.so)
and a C++ driver=sx SoapySDR device above it (lib/libsxsoapy.so).  This package only holds
the build recipes and ctypes views that tests/ and bench.py use.
"""
from .capi import Bank, Chan, ChanSynth, Context, Fir, Iir, Multi, Nco, SxGpuError, load_library, library_path  # noqa: F401

__all__ = ["Bank", "Chan", "ChanSynth", "Context", "Fir", "Iir", "Multi", "Nco", "SxGpuError", "load_library", "library_path"]
