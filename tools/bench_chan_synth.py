#!/usr/bin/env python
"""ChanSynth.apply (sxgpu_chan_synth_apply) on four shapes, against the bounds their dimensions allow,
beside the split form users have today.

    A  65 536 streams x 16 frames per channel, M = 16, D = 16, 256 taps   (256 outputs: the bank's block)
    B  65 536 x 32, M = 16, D = 8, 256 taps                              (oversampled by 2)
    C  1 x 2^22, M = 64, D = 32, 1 024 taps                              (2^27 outputs: a long burst)
    D  16 x 1 024, M = 1024, D = 1024, 16 384 taps                       (2^20 outputs)

For each: the median over rounds of the CUDA-event time per call (each round times back-to-back
warmed calls; every call keeps the phase, so every call does the same work), and beside it
    FP32 bound  (4 ceil(ntaps / D) + 10 (M/2) log2 M / D) FP32 instructions per output frame (FMUL and
                FADD for I and Q: no FFMA, by the bit-exact specification) / (SMs x 128 lanes x the
                card's maximum SM clock)
    HBM bound   (input + output + the history read and written) bytes / 7.7 TB/s (the B200's
                data-sheet bandwidth)
and achieved / max(bounds).  Every shape moves more than the 126 MB of L2 per call.  A separate
torch.profiler run splits each call into the synthesis and history kernels.  In the same rounds,
alternating with the synthesizer, the split form:
    A, B  one Fir.apply(h, D, 1) over all S M channel rows, one Nco.apply with row (s, k) at +k/M,
          in place, and a torch sum over the channels
    C     the same channel by channel (its M-times block would be 64 GiB): per channel a
          Fir.apply into one full-rate block, Nco.apply on it, and a torch add into the output
    D     none
The card's name, power limit and maximum SM clock are read in the same run.

    python tools/bench_chan_synth.py --out profiles/r03_bench_chan_synth.json
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
from sxxcvr_b200 import ChanSynth, Context, Fir, Nco  # noqa: E402

SHAPES = [  # name, streams, frames per channel, M, D, taps, calls per round, split form
    ("A", 65536, 16, 16, 16, 256, 20, "rows"),
    ("B", 65536, 32, 16, 8, 256, 20, "rows"),
    ("C", 1, 1 << 22, 64, 32, 1024, 3, "channels"),
    ("D", 16, 1024, 1024, 1024, 16384, 20, None),
]


def bounds(S, N, M, D, ntaps, sms, clock_mhz):
    hp, nout = -(-ntaps // D), N * D
    fp32 = (4 * hp + 10 * (M // 2) * int(math.log2(M)) / D) * S * nout / (sms * FP32_LANES_PER_SM * clock_mhz * 1e6)
    nbytes = 8 * S * M * N + 8 * S * nout + 2 * 8 * S * M * (hp - 1)
    return nbytes, fp32 * 1e6, nbytes / HBM_BYTES_PER_S * 1e6


def split_bytes(S, N, M, D, ntaps):
    """The interpolators (input, M full-rate blocks, history read and written), the oscillators in
    place (read + write), the sum (read the M blocks, write the output)."""
    hp, nout = -(-ntaps // D), N * D
    return 8 * S * M * N + 8 * S * M * nout + 2 * 8 * S * M * (hp - 1) + 2 * 8 * S * M * nout + 8 * S * M * nout + 8 * S * nout


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="bench_chan_synth.json", help="where the JSON result goes")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--shapes", nargs="*", default=[s[0] for s in SHAPES])
    args = ap.parse_args()

    info = card()
    ctx = Context(0)
    sms = ctx.info().sm_count
    side = torch.cuda.Stream()
    st = side.cuda_stream
    result = {"card": info, "sm_count": sms, "rounds": args.rounds, "hbm_bytes_per_s": HBM_BYTES_PER_S, "points": []}
    for name, S, N, M, D, ntaps, iters, split_form in SHAPES:
        if name not in args.shapes:
            continue
        h = signal.firwin(ntaps, 1.0 / M)
        nout = N * D
        freqs = [k / M if k < M // 2 else (k - M) / M for k in range(M)]
        with ChanSynth(ctx, S, h, M, D) as s:
            y = torch.randn(S * M * N * 2, dtype=torch.float32, device="cuda")
            x = torch.empty(S * nout * 2, dtype=torch.float32, device="cuda")
            dy, dx = y.data_ptr(), x.data_ptr()
            forms = {"synth": lambda: s.apply(dy, N, dx, st)}
            extra, scratch = [], None
            if split_form == "rows":
                fir, nco = Fir(ctx, S * M, h, D, 1), Nco(ctx, S * M, freqs * S)
                extra = [fir, nco]
                scratch = torch.empty(S * M * nout * 2, dtype=torch.float32, device="cuda")
                rows = torch.view_as_complex(scratch.view(S, M, nout, 2))
                xc = torch.view_as_complex(x.view(S, nout, 2))

                def split():
                    fir.apply(dy, N, scratch.data_ptr(), st)
                    nco.apply(scratch.data_ptr(), nout, st)
                    with torch.cuda.stream(side):
                        torch.sum(rows, dim=1, out=xc)
                forms["split"] = split
            elif split_form == "channels":
                assert S == 1  # channel k's row of y is then contiguous
                firs = [Fir(ctx, 1, h, D, 1) for _ in range(M)]
                ncos = [Nco(ctx, 1, f) for f in freqs]
                extra = firs + ncos
                scratch = torch.empty(nout * 2, dtype=torch.float32, device="cuda")

                def split():
                    with torch.cuda.stream(side):
                        x.zero_()
                        for k in range(M):
                            firs[k].apply(dy + 8 * k * N, N, scratch.data_ptr(), st)
                            ncos[k].apply(scratch.data_ptr(), nout, st)
                            x.add_(scratch)
                forms["split"] = split
            torch.cuda.synchronize()
            times = timed_pair(forms, side, iters, args.rounds)
            nbytes, fp32, hbm = bounds(S, N, M, D, ntaps, sms, info["max_sm_clock_mhz"])
            before = ctx.counter("launches")
            forms["synth"]()
            side.synchronize()
            us = statistics.median(times["synth"])
            point = {"shape": name, "streams": S, "frames_in": N, "channels": M, "up": D, "taps": ntaps,
                     "outputs": nout, "us_per_call": us, "min_us": min(times["synth"]), "max_us": max(times["synth"]),
                     "launches_per_call": ctx.counter("launches") - before, "bytes": nbytes,
                     "fp32_bound_us": fp32, "hbm_bound_us": hbm, "bound": "hbm" if hbm >= fp32 else "fp32",
                     "achieved_over_bound": us / max(hbm, fp32)}
            point["profiled_kernel_us"] = kernel_breakdown(forms["synth"], side, 5)
            if split_form:
                t = times["split"]
                point["split"] = {"form": split_form, "us_per_call": statistics.median(t), "min_us": min(t),
                                  "max_us": max(t), "bytes": split_bytes(S, N, M, D, ntaps)}
                point["split"]["hbm_bound_us"] = point["split"]["bytes"] / HBM_BYTES_PER_S * 1e6
                point["split_over_synth"] = point["split"]["us_per_call"] / us
            result["points"].append(point)
            print(json.dumps(point), flush=True)
            side.synchronize()
            for obj in extra:
                obj.close()
            del x, y, scratch
            torch.cuda.empty_cache()
    ctx.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
