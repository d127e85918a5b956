#!/usr/bin/env python
"""Chan.apply (sxgpu_chan_apply) on four shapes, against the bounds their dimensions allow, beside
the per-channel split form users have today and a float32 torch form.

    A  65 536 streams x 256 frames, M = 16, D = 16, 256 taps    (the bank's block)
    B  the same with D = 8                                      (oversampled by 2)
    C  1 x 2^27 frames, M = 64, D = 32, 1 024 taps              (a long capture)
    D  16 x 2^20 frames, M = 1024, D = 1024, 16 384 taps

For each: the median over rounds of the CUDA-event time per call (each round times back-to-back
warmed calls; every call keeps the phase, so every call does the same work), and beside it
    FP32 bound  (4 ntaps + 10 (M/2) log2 M) FP32 instructions per output frame of a stream (FMUL
                and FADD for I and Q: no FFMA, by the bit-exact specification) / (SMs x 128 lanes x
                the card's maximum SM clock)
    HBM bound   (input + output + the history read and written) bytes / 7.7 TB/s (the B200's
                data-sheet bandwidth)
and achieved / max(bounds).  Every shape moves more than the 126 MB of L2 per call.  A separate
torch.profiler run splits each call into the apply and history kernels.  In the same rounds,
alternating with the channelizer:
    split  (A, B, C) per channel k: a device-to-device cudaMemcpyAsync of the block, Nco.apply at
           -k/M on the copy, Fir.apply(h, 1, D) into that channel's rows -- M oscillators and M
           filters, one per channel
    torch  the branch sums as one float32 conv1d with M output channels (the taps of branch r at
           the lags r mod M), then torch.fft.ifft over the channels and the rotation e^{-j 2 pi k N / M};
           TF32 off, neither stateful nor bit-exact -- informative only
The card's name, power limit and maximum SM clock are read in the same run.

    python tools/bench_chan.py --out profiles/r03_bench_chan.json
"""
from __future__ import annotations

import argparse
import json
import math
import statistics
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import torch  # noqa: E402
from scipy import signal  # noqa: E402

from bench_fir_bank import kernel_breakdown, timed_pair  # noqa: E402
from bench_iir import FP32_LANES_PER_SM, HBM_BYTES_PER_S, card  # noqa: E402
from sxxcvr_b200 import Chan, Context, Fir, Nco  # noqa: E402

SHAPES = [  # name, streams, frames, M, D, taps, calls per round, split form
    ("A", 65536, 256, 16, 16, 256, 20, True),
    ("B", 65536, 256, 16, 8, 256, 20, True),
    ("C", 1, 1 << 27, 64, 32, 1024, 3, True),
    ("D", 16, 1 << 20, 1024, 1024, 16384, 20, False),
]


def bounds(S, N, M, nout, ntaps, sms, clock_mhz):
    fp32 = (4 * ntaps + 10 * (M // 2) * int(math.log2(M))) * S * nout / (sms * FP32_LANES_PER_SM * clock_mhz * 1e6)
    nbytes = 8 * S * N + 8 * S * M * nout + 2 * 8 * S * (ntaps - 1)
    return nbytes, fp32 * 1e6, nbytes / HBM_BYTES_PER_S * 1e6


def split_bytes(S, N, M, nout, ntaps):
    """Per channel: the copy (read + write), the oscillator in place (read + write), the filter
    (input, output, history read and written)."""
    return M * (4 * 8 * S * N + 8 * S * N + 8 * S * nout + 2 * 8 * S * (ntaps - 1))


def torch_form(x, S, N, M, D, h):
    """Branch sums by conv1d, then ifft and the rotation: (S, M, nout) complex64, stateless."""
    ntaps = len(h)
    lag = torch.arange(ntaps)
    w = torch.zeros(M, 1, ntaps, dtype=torch.float32)
    taps = torch.tensor(h, dtype=torch.float32)
    for r in range(M):  # conv1d correlates: weight j meets lag ntaps - 1 - j
        sel = lag % M == r
        w[r, 0, ntaps - 1 - lag[sel]] = taps[sel]
    w = w.cuda()
    nout = -(-N // D)
    k = torch.arange(M, device="cuda").view(M, 1)
    n = torch.arange(nout, device="cuda").view(1, nout) * D
    rot = torch.exp(torch.complex(torch.zeros((), device="cuda"), -2 * math.pi * ((k * n) % M).float() / M)) * M
    xv = x.view(S, N, 2).permute(0, 2, 1).reshape(2 * S, 1, N)

    def call():
        u = torch.nn.functional.conv1d(torch.nn.functional.pad(xv, (ntaps - 1, 0)), w, stride=D)  # (2S, M, nout)
        u = u.view(S, 2, M, nout)
        return torch.fft.ifft(torch.complex(u[:, 0], u[:, 1]), dim=1) * rot
    return call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="bench_chan.json", help="where the JSON result goes")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--shapes", nargs="*", default=[s[0] for s in SHAPES])
    args = ap.parse_args()

    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    info = card()
    ctx = Context(0)
    sms = ctx.info().sm_count
    side = torch.cuda.Stream()
    st = side.cuda_stream
    result = {"card": info, "sm_count": sms, "rounds": args.rounds, "hbm_bytes_per_s": HBM_BYTES_PER_S, "points": []}
    for name, S, N, M, D, ntaps, iters, with_split in SHAPES:
        if name not in args.shapes:
            continue
        h = signal.firwin(ntaps, 1.0 / M)
        with Chan(ctx, S, h, M, D) as c:
            nout = c.output_frames(N)
            x = torch.randn(S * N * 2, dtype=torch.float32, device="cuda")
            y = torch.empty(S * M * nout * 2, dtype=torch.float32, device="cuda")
            dx, dy = x.data_ptr(), y.data_ptr()
            forms = {"chan": lambda: c.apply(dx, N, dy, st)}
            extra = []
            if with_split:
                freqs = [(-k / M + 1.0) if -k / M < -0.5 else -k / M for k in range(M)]
                ncos = [Nco(ctx, S, f) for f in freqs]
                firs = [Fir(ctx, S, h, 1, D) for _ in range(M)]
                extra = ncos + firs
                copy = torch.empty_like(x)
                dcopy = copy.data_ptr()

                def split():
                    with torch.cuda.stream(side):
                        for k in range(M):
                            copy.copy_(x, non_blocking=True)  # a device-to-device cudaMemcpyAsync
                            ncos[k].apply(dcopy, N, st)
                            firs[k].apply(dcopy, N, dy + 8 * k * S * nout, st)
                forms["split"] = split
            tcall = torch_form(x, S, N, M, D, h)

            def torch_call():
                with torch.cuda.stream(side):
                    tcall()
            torch_error = None
            try:
                torch_call()
                side.synchronize()
                forms["torch"] = torch_call
            except RuntimeError as e:  # informative only: a shape cuDNN cannot take is reported, not fatal
                torch_error = str(e).splitlines()[0]
            torch.cuda.synchronize()  # the calls run on another stream
            times = timed_pair(forms, side, iters, args.rounds)
            nbytes, fp32, hbm = bounds(S, N, M, nout, ntaps, sms, info["max_sm_clock_mhz"])
            before = ctx.counter("launches")
            forms["chan"]()
            side.synchronize()
            us = statistics.median(times["chan"])
            point = {"shape": name, "streams": S, "frames": N, "channels": M, "down": D, "taps": ntaps,
                     "outputs": nout, "us_per_call": us, "min_us": min(times["chan"]), "max_us": max(times["chan"]),
                     "launches_per_call": ctx.counter("launches") - before, "bytes": nbytes,
                     "fp32_bound_us": fp32, "hbm_bound_us": hbm, "bound": "hbm" if hbm >= fp32 else "fp32",
                     "achieved_over_bound": us / max(hbm, fp32)}
            point["profiled_kernel_us"] = kernel_breakdown(forms["chan"], side, 5)
            for k in forms:
                if k == "chan":
                    continue
                point[k] = {"us_per_call": statistics.median(times[k]), "min_us": min(times[k]),
                            "max_us": max(times[k])}
                point[f"{k}_over_chan"] = point[k]["us_per_call"] / us
            if torch_error:
                point["torch"] = {"error": torch_error}
            if with_split:
                point["split"]["bytes"] = split_bytes(S, N, M, nout, ntaps)
                point["split"]["hbm_bound_us"] = point["split"]["bytes"] / HBM_BYTES_PER_S * 1e6
            result["points"].append(point)
            print(json.dumps(point), flush=True)
            for obj in extra:
                obj.close()
            del x, y, tcall
            torch.cuda.empty_cache()
    ctx.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
