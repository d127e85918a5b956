#!/usr/bin/env python
"""The FIR halves with an oscillator fused in (Bank.read_ddc, Bank.write_duc) against the split
forms they replace and against the FIR halves without the oscillator, on twin banks, filters and
oscillators, alternating the forms in the same rounds; and the standalone Nco.apply at 2^27 frames
against a device-to-device copy of the same block.

    RX-A  65 536 streams x 256 frames, 64 taps, down 4, synthetic capture
    RX-B  the same with ingested capture
    RX-C  4 096 streams x 256 frames, 64 taps, down 4, synthetic capture
    TX-A  65 536 streams x 256 frames from 64-frame blocks, 64 taps, up 4
    TX-B  65 536 streams x 255 frames from 170-frame blocks, 96 taps, up 3 down 2
    NCO   1 x 2^27 frames (1 GiB) mixed in place

    rx fused  read_ddc(N, F, out)          rx split  read(cf32), N.apply(cf32, period), F.apply(cf32, period, out)
                                           rx fir    read_fir(F, out): the same call without the mixer
    tx fused  write_duc(G, N, in, nin)     tx split  G.apply(in, nin, cf32), N.apply(cf32, period), write(cf32)
                                           tx fir    write_fir(G, in, nin)
    (writes untimed)

For each: the median over rounds of the CUDA-event time per call (each round times back-to-back
warmed calls of each form in turn; every call keeps the filter's phase, so every call does the same
work), the bytes each form must move through HBM computed from the shapes (bench_fir_bank.py's
count, plus the oscillator's phases and increments, plus for the split form the full-rate block
read and written once more by Nco.apply), and a torch.profiler run of its own splitting each call
by kernel.  Every shape but RX-C moves more than the 126 MB of L2 per call.  NCO reports GB/s as
bytes read plus bytes written over time, beside a torch device-to-device copy of the same block in
the same rounds and the copy ceiling recorded in profiles/r02_bank_and_converter_limits.json.  The
card's name, power limit and maximum SM clock are read in the same run.

    python tools/bench_ddc.py --out bench_ddc.json
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

import numpy as np  # noqa: E402
import torch  # noqa: E402
from scipy import signal  # noqa: E402

from bench_fir_bank import kernel_breakdown, timed_pair, traffic  # noqa: E402
from bench_iir import HBM_BYTES_PER_S, card  # noqa: E402
from sxxcvr_b200 import Bank, Context, Fir, Nco  # noqa: E402

SHAPES = [  # name, side, streams, period, taps, up, down, capture, calls per round
    ("RX-A", "rx", 65536, 256, 64, 1, 4, "synthetic", 20),
    ("RX-B", "rx", 65536, 256, 64, 1, 4, "ingested", 20),
    ("RX-C", "rx", 4096, 256, 64, 1, 4, "synthetic", 200),
    ("TX-A", "tx", 65536, 256, 64, 4, 1, None, 20),
    ("TX-B", "tx", 65536, 255, 96, 3, 2, None, 20),
]
NCO_FRAMES = 1 << 27
COPY_CEILING = ("profiles/r02_bank_and_converter_limits.json", "3_converters_and_bank_with_plan", "memcpy_d2d_1GiB")


def recorded_copy_ceiling():
    path, part, kernel = COPY_CEILING
    runs = json.loads((ROOT / path).read_text())["passes"][part]
    return next(r["gbs"] for r in runs if r["kernel"] == kernel)


def bank_points(ctx, info, side, rounds, names):
    st = side.cuda_stream
    points = []
    for name, kind, S, P, ntaps, up, down, capture, iters in SHAPES:
        if name not in names:
            continue
        h = signal.firwin(ntaps, 0.8 / max(up, down))
        hp = -(-ntaps // up)
        nin = P if kind == "rx" else P * down // up
        freqs = np.linspace(-0.45, 0.45, S)
        with Bank(ctx, S, P) as fb, Bank(ctx, S, P) as sb, Bank(ctx, S, P) as rb, Fir(ctx, S, h, up, down) as ff, \
                Fir(ctx, S, h, up, down) as sf, Fir(ctx, S, h, up, down) as rf, Nco(ctx, S, freqs) as fn, \
                Nco(ctx, S, freqs) as sn:
            nout = ff.output_frames(nin)
            full = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
            if kind == "rx":
                chan = torch.zeros(S * nout * 2, dtype=torch.float32, device="cuda")
                if capture == "ingested":
                    i2s = torch.randint(-2**31, 2**31 - 1, (S * P * 2,), dtype=torch.int32, device="cuda")
                    for b in (fb, sb, rb):
                        b.ingest(0, S, i2s.data_ptr())
                dc, df = chan.data_ptr(), full.data_ptr()

                def split():
                    sb.read(df, st)
                    sn.apply(df, P, st)
                    sf.apply(df, P, dc, st)
                forms = {"fused": lambda: fb.read_ddc(fn, ff, dc, st), "split": split,
                         "fir": lambda: rb.read_fir(rf, dc, st)}
            else:
                chan = torch.randn(S * nin * 2, dtype=torch.float32, device="cuda")
                dc, df = chan.data_ptr(), full.data_ptr()

                def split():
                    sf.apply(dc, nin, df, st)
                    sn.apply(df, P, st)
                    sb.write(df, 0, None, 0, st)
                forms = {"fused": lambda: fb.write_duc(ff, fn, dc, nin, 0, None, 0, st), "split": split,
                         "fir": lambda: rb.write_fir(rf, dc, nin, 0, None, 0, st)}
            torch.cuda.synchronize()  # the calls run on another stream
            times = timed_pair(forms, side, iters, rounds)
            fir_bytes, fir_split_bytes = traffic(kind, S, P, nin, nout, hp)
            state = 4 * S * 3  # phases read and written, increments read
            nbytes = {"fused": fir_bytes + state, "split": fir_split_bytes + 2 * 8 * S * P + state, "fir": fir_bytes}
            point = {"shape": name, "side": kind, "streams": S, "period": P, "taps": ntaps, "up": up, "down": down,
                     "capture": capture, "frames_in": nin, "frames_out": nout}
            for k in forms:
                before = ctx.counter("launches")
                forms[k]()
                side.synchronize()
                us = statistics.median(times[k])
                hbm = nbytes[k] / HBM_BYTES_PER_S * 1e6
                point[k] = {"us_per_call": us, "min_us": min(times[k]), "max_us": max(times[k]),
                            "launches_per_call": ctx.counter("launches") - before, "bytes": nbytes[k],
                            "hbm_bound_us": hbm, "achieved_over_hbm_bound": us / hbm}
            for k in forms:
                point[k]["profiled_kernel_us"] = kernel_breakdown(forms[k], side, 5)
            point["fused_over_split"] = point["fused"]["us_per_call"] / point["split"]["us_per_call"]
            point["fused_over_fir"] = point["fused"]["us_per_call"] / point["fir"]["us_per_call"]
            points.append(point)
            print(json.dumps(point), flush=True)
            del full, chan
            torch.cuda.empty_cache()
    return points


def nco_point(ctx, side, rounds):
    st = side.cuda_stream
    n = NCO_FRAMES
    x = torch.randn(2 * n, dtype=torch.float32, device="cuda")
    y = torch.empty_like(x)
    with Nco(ctx, 1, [0.123456]) as N:
        def copy():
            with torch.cuda.stream(side):
                y.copy_(x)
        forms = {"nco_apply": lambda: N.apply(x.data_ptr(), n, st), "copy": copy}
        torch.cuda.synchronize()
        times = timed_pair(forms, side, 20, rounds)
        moved = 2 * 8 * n  # read and written
        ceiling = recorded_copy_ceiling()
        point = {"shape": "NCO", "frames": n, "bytes_moved": moved, "recorded_copy_ceiling_gbs": ceiling,
                 "recorded_copy_ceiling": "/".join(COPY_CEILING)}
        for k in forms:
            us = statistics.median(times[k])
            point[k] = {"us_per_call": us, "min_us": min(times[k]), "max_us": max(times[k]), "gbs": moved / us / 1e3}
        point["nco_apply"]["profiled_kernel_us"] = kernel_breakdown(forms["nco_apply"], side, 5)
        point["nco_over_recorded_ceiling"] = point["nco_apply"]["gbs"] / ceiling
        point["nco_over_copy_same_run"] = point["nco_apply"]["gbs"] / point["copy"]["gbs"]
        print(json.dumps(point), flush=True)
    del x, y
    torch.cuda.empty_cache()
    return point


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="bench_ddc.json", help="where the JSON result goes")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--shapes", nargs="*", default=[s[0] for s in SHAPES] + ["NCO"])
    args = ap.parse_args()

    info = card()
    ctx = Context(0)
    side = torch.cuda.Stream()
    result = {"card": info, "sm_count": ctx.info().sm_count, "rounds": args.rounds, "hbm_bytes_per_s": HBM_BYTES_PER_S,
              "points": bank_points(ctx, info, side, args.rounds, args.shapes)}
    if "NCO" in args.shapes:
        result["points"].append(nco_point(ctx, side, args.rounds))
    ctx.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
