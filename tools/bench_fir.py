#!/usr/bin/env python
"""Fir.apply (sxgpu_fir_apply) on four shapes, against the bounds their dimensions allow.

    A  65 536 streams x 256 frames, 64 taps, down 4    (the bank's block, decimated)
    B  1 x 2^27 frames, 127 taps, 1/1                   (a long channel filter)
    C  16 x 2^20 frames, 96 taps, up 3 down 2
    D  64 x 256 frames, 64 taps, down 4                 (latency-bound; reported only)

For each: the median over rounds of the CUDA-event time per call (each round times back-to-back
warmed calls; every call keeps the phase, so every call does the same work), and beside it
    FP32 bound  4 FP32 instructions (2 FMUL, 2 FADD: no FFMA, by the bit-exact specification) per
                polyphase tap and output frame / (SMs x 128 lanes x the card's maximum SM clock)
    HBM bound   (input + output + the history read and written) bytes / 7.7 TB/s (the B200's
                data-sheet bandwidth)
and achieved / max(bounds).  A, B and C move more than the 126 MB of L2 per call.  A separate
torch.profiler run splits each call into its two kernels.  Beside each shape, what a user does
today: torch.nn.functional.conv1d in float32 (TF32 off) with I and Q as two channels and
stride = down (C: the input zero-stuffed by 3 first), neither stateful nor bit-exact -- informative
only.  The card's name, power limit and maximum SM clock are read in the same run.

    python tools/bench_fir.py --out bench_fir.json
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

from bench_iir import FP32_LANES_PER_SM, HBM_BYTES_PER_S, card  # noqa: E402
from sxxcvr_b200 import Context, Fir  # noqa: E402

FP32_PER_TAP_OUTPUT = 4
SHAPES = [  # name, streams, frames, taps, up, down, calls per round
    ("A", 65536, 256, 64, 1, 4, 50),
    ("B", 1, 1 << 27, 127, 1, 1, 5),
    ("C", 16, 1 << 20, 96, 3, 2, 20),
    ("D", 64, 256, 64, 1, 4, 500),
]


def bounds_us(S, N, nout, ntaps, up, sms, clock_mhz):
    hp = -(-ntaps // up)
    fp32 = FP32_PER_TAP_OUTPUT * hp * S * nout / (sms * FP32_LANES_PER_SM * clock_mhz * 1e6)
    nbytes = 8 * S * N + 8 * S * nout + 2 * 8 * S * (hp - 1)
    return nbytes, fp32 * 1e6, nbytes / HBM_BYTES_PER_S * 1e6


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
        if ev.device_type.name != "CUDA" or "fir_" not in ev.key:
            continue
        key = "history" if "fir_history_kernel" in ev.key else "apply"
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = ev.cuda_time_total
        out[key] = out.get(key, 0.0) + us / calls
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="bench_fir.json", help="where the JSON result goes")
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()

    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    info = card()
    ctx = Context(0)
    sms = ctx.info().sm_count
    side = torch.cuda.Stream()
    st = side.cuda_stream
    result = {"card": info, "sm_count": sms, "rounds": args.rounds, "hbm_bytes_per_s": HBM_BYTES_PER_S,
              "fp32_per_tap_output": FP32_PER_TAP_OUTPUT, "points": []}
    for name, S, N, ntaps, up, down, iters in SHAPES:
        h = signal.firwin(ntaps, 0.8 / max(up, down))
        with Fir(ctx, S, h, up, down) as f:
            nout = f.output_frames(N)
            x = torch.randn(S * N * 2, dtype=torch.float32, device="cuda")
            y = torch.empty(S * nout * 2, dtype=torch.float32, device="cuda")
            torch.cuda.synchronize()  # the calls run on another stream
            dx, dy = x.data_ptr(), y.data_ptr()
            call = lambda: f.apply(dx, N, dy, st)  # noqa: E731
            times = timed(call, side, iters, args.rounds)
            us = statistics.median(times)
            nbytes, fp32, hbm = bounds_us(S, N, nout, ntaps, up, sms, info["max_sm_clock_mhz"])
            before = ctx.counter("launches")
            call()
            side.synchronize()
            point = {"shape": name, "streams": S, "frames": N, "taps": ntaps, "up": up, "down": down,
                     "outputs": nout, "us_per_call": us, "min_us": min(times), "max_us": max(times),
                     "launches_per_call": ctx.counter("launches") - before, "bytes": nbytes,
                     "fp32_bound_us": fp32, "hbm_bound_us": hbm, "bound": "hbm" if hbm >= fp32 else "fp32",
                     "achieved_over_bound": us / max(hbm, fp32)}
            point["profiled_kernel_us"] = kernel_breakdown(call, side, 5)

            # what a user does today: conv1d, I and Q as channels, stateless, not bit-exact
            xc = x.view(S, N, 2).permute(0, 2, 1).contiguous()
            w = torch.from_numpy(h[::-1].astype("float32").copy()).cuda().view(1, 1, -1).repeat(2, 1, 1)
            if up > 1:
                stuffed = torch.zeros(S, 2, N * up, dtype=torch.float32, device="cuda")
                conv = lambda: torch.nn.functional.conv1d(  # noqa: E731
                    stuffed.index_copy_(2, torch.arange(0, N * up, up, device="cuda"), xc), w, stride=down, groups=2)
            else:
                conv = lambda: torch.nn.functional.conv1d(xc, w, stride=down, groups=2)  # noqa: E731
            with torch.cuda.stream(side):
                ctimes = timed(conv, side, max(1, iters // 5), args.rounds)
            point["conv1d_us_per_call"] = statistics.median(ctimes)
            result["points"].append(point)
            print(json.dumps(point), flush=True)
            del x, y, xc
            torch.cuda.empty_cache()
    ctx.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
