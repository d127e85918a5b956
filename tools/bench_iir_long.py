#!/usr/bin/env python
"""Iir.apply_long (sxgpu_iir_apply_long) on long blocks, with one 4-section filter (butter(8, 0.25)).

For 1 x 2^27, 16 x 2^23 and 1 x 2^22 frames: the median over rounds of the CUDA-event time per call
(each round times back-to-back warmed calls on one block of 8 B/frame, 1 GB for 2^27 frames, far
above the 126 MB of L2 except at 2^22), and beside it the least time the shapes allow:
    HBM bound   24 B/frame (pass 1 reads 8, pass 3 reads 8 and writes 8) / 7.7 TB/s (the B200's
                data-sheet bandwidth)
    FP32 bound  2 passes x 9 FP32 instructions per section, component and frame (un-contracted
                transposed direct form II) / (SMs x 128 lanes x the card's maximum SM clock)
and achieved / max(bounds), as in tools/bench_iir.py.  At 1 x 2^22 also the sequential way of the
same work: 64 calls of Iir.apply on consecutive 65536-frame pieces.  A separate torch.profiler run
of a few calls per shape breaks each call down by kernel, giving the carry's share (reduce, scan
levels and fix-up).  The card's name, power limit and maximum SM clock are read in the same run.

    python tools/bench_iir_long.py --out bench_iir_long.json
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import torch  # noqa: E402
from scipy import signal  # noqa: E402

from bench_iir import FLOPS_PER_SECTION_SAMPLE, FP32_LANES_PER_SM, HBM_BYTES_PER_S, card  # noqa: E402
from sxxcvr_b200 import Context, Iir  # noqa: E402

BYTES_PER_FRAME = 24
PASSES = 2


def bounds_us(frames, nsections, sms, clock_mhz):
    hbm = BYTES_PER_FRAME * frames / HBM_BYTES_PER_S
    fp32 = PASSES * FLOPS_PER_SECTION_SAMPLE * nsections * 2 * frames / (sms * FP32_LANES_PER_SM * clock_mhz * 1e6)
    return hbm * 1e6, fp32 * 1e6


def timed(fn, side, iters, rounds):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        fn()
    side.synchronize()
    times = []
    for _ in range(rounds):
        a.record(side)
        for _ in range(iters):
            fn()
        b.record(side)
        b.synchronize()
        times.append(a.elapsed_time(b) * 1e3 / iters)
    return times


def kernel_breakdown(fn, side, calls):
    """Device time per call by kernel, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    side.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        side.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type.name != "CUDA":
            continue
        name = ev.key
        if "iir_carry" in name:
            key = name.split("(")[0].split("::")[-1]
        elif "iir_apply_kernel<1>" in name:
            key = "pass1"
        elif "iir_apply_kernel<2>" in name:
            key = "pass3"
        elif "iir_apply_kernel" in name:
            key = "apply"
        else:
            continue
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = ev.cuda_time_total
        out[key] = out.get(key, 0.0) + us / calls
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="bench_iir_long.json", help="where the JSON result goes")
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()

    info = card()
    ctx = Context(0)
    sms = ctx.info().sm_count
    side = torch.cuda.Stream()
    st = side.cuda_stream
    sos = signal.butter(8, 0.25, output="sos")
    nsec = sos.shape[0]
    result = {"card": info, "sm_count": sms, "filter": "butter(8, 0.25), 4 sections", "rounds": args.rounds,
              "hbm_bytes_per_s": HBM_BYTES_PER_S, "points": []}
    for S, N, iters in ((1, 1 << 27, 10), (16, 1 << 23, 10), (1, 1 << 22, 50)):
        with Iir(ctx, S, sos) as f:
            cf = torch.randn(S * N * 2, dtype=torch.float32, device="cuda")
            torch.cuda.synchronize()  # the calls run on another stream
            d = cf.data_ptr()
            long_call = lambda: f.apply_long(d, N, st)  # noqa: E731
            times = timed(long_call, side, iters, args.rounds)
            us = statistics.median(times)
            hbm, fp32 = bounds_us(S * N, nsec, sms, info["max_sm_clock_mhz"])
            before = ctx.counter("launches")
            long_call()
            side.synchronize()
            point = {"streams": S, "frames": N, "mode": "apply_long", "us_per_call": us, "min_us": min(times),
                     "max_us": max(times), "launches_per_call": ctx.counter("launches") - before,
                     "hbm_bound_us": hbm, "fp32_bound_us": fp32, "bound": "hbm" if hbm >= fp32 else "fp32",
                     "achieved_over_bound": us / max(hbm, fp32)}
            kernels = kernel_breakdown(long_call, side, 5)
            carry = sum(v for k, v in kernels.items() if k.startswith("iir_carry"))
            point["profiled_kernel_us"] = kernels
            point["carry_us"] = carry
            point["carry_share_of_kernel_time"] = carry / sum(kernels.values())
            result["points"].append(point)
            print(json.dumps(point), flush=True)
            if S == 1 and N == 1 << 22:
                piece = 65536

                def sequential():
                    for k in range(N // piece):
                        f.apply(d + k * piece * 8, piece, st)
                times = timed(sequential, side, 2, args.rounds)
                seq = {"streams": S, "frames": N, "mode": "apply_64_pieces", "us_per_call": statistics.median(times),
                       "min_us": min(times), "max_us": max(times), "speedup_of_apply_long": statistics.median(times) / us}
                result["points"].append(seq)
                print(json.dumps(seq), flush=True)
            del cf
    ctx.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
