#!/usr/bin/env python
"""The bank's halves with a FIR filter fused in (Bank.read_fir, Bank.write_fir) against the split
forms they replace, on twin banks and twin filters, alternating fused and split in the same rounds.

    RX-A  65 536 streams x 256 frames, 64 taps, down 4, synthetic capture
    RX-B  the same with ingested capture
    RX-C  4 096 streams x 256 frames, 64 taps, down 4, synthetic capture
    TX-A  65 536 streams x 256 frames from 64-frame blocks, 64 taps, up 4
    TX-B  65 536 streams x 255 frames from 170-frame blocks, 96 taps, up 3 down 2

    rx fused  read_fir(F, out)                       rx split  read(cf32), F.apply(cf32, period, out)
    tx fused  write_fir(G, in, nin, untimed)         tx split  G.apply(in, nin, cf32), write(cf32, untimed)

For each: the median over rounds of the CUDA-event time per call (each round times back-to-back
warmed calls of the fused form, then of the split form; every call keeps the phase, so every call
does the same work), and beside it, computed from the shapes,
    bytes       what each form must move through HBM: the capture slot (written, or read when
                ingested), the channel-rate block, the history read and written, and for the split
                form the full-rate CF32 block written and read back; the TX side in reverse, with
                the playback ring written
    HBM bound   bytes / 7.7 TB/s (the B200's data-sheet bandwidth)
    FP32 bound  4 FP32 instructions (2 FMUL, 2 FADD: no FFMA) per polyphase tap and output frame /
                (SMs x 128 lanes x the card's maximum SM clock)
and a torch.profiler run of its own splitting each form's call by kernel.  Every shape but RX-C
moves more than the 126 MB of L2 per call.  The card's name, power limit and maximum SM clock are
read in the same run.

    python tools/bench_fir_bank.py --out bench_fir_bank.json
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
from sxxcvr_b200 import Bank, Context, Fir  # noqa: E402

FP32_PER_TAP_OUTPUT = 4
SHAPES = [  # name, side, streams, period, taps, up, down, capture, calls per round
    ("RX-A", "rx", 65536, 256, 64, 1, 4, "synthetic", 20),
    ("RX-B", "rx", 65536, 256, 64, 1, 4, "ingested", 20),
    ("RX-C", "rx", 4096, 256, 64, 1, 4, "synthetic", 200),
    ("TX-A", "tx", 65536, 256, 64, 4, 1, None, 20),
    ("TX-B", "tx", 65536, 255, 96, 3, 2, None, 20),
]


def traffic(side, S, P, nin, nout, hp):
    """Bytes through HBM per call, (fused, split), 8-byte frames: the capture slot (written when
    synthetic, read when ingested) or the ring slice is one full-rate pass; the split form adds the
    full-rate CF32 block written and read back."""
    hist = 2 * 8 * S * (hp - 1)
    full = 8 * S * P
    chan = 8 * S * (nout if side == "rx" else nin)
    return full + chan + hist, 3 * full + chan + hist


def timed_pair(fns, side, iters, rounds):
    """{name: [us per call per round]}, the forms alternating within each round."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for fn in fns.values():
        for _ in range(3):
            fn()
    side.synchronize()
    times = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            ev[0].record(side)
            for _ in range(iters):
                fn()
            ev[1].record(side)
            ev[1].synchronize()
            times[k].append(ev[0].elapsed_time(ev[1]) * 1e3 / iters)
    return times


def kernel_breakdown(fn, side, calls):
    """Device time per call by kernel name, from torch.profiler."""
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
        name = ev.key.split("<")[0].split("(")[0].replace("void ", "").replace("sx::", "")
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = ev.cuda_time_total
        out[name] = out.get(name, 0.0) + us / calls
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="bench_fir_bank.json", help="where the JSON result goes")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--shapes", nargs="*", default=[s[0] for s in SHAPES])
    args = ap.parse_args()

    info = card()
    ctx = Context(0)
    sms = ctx.info().sm_count
    side = torch.cuda.Stream()
    st = side.cuda_stream
    result = {"card": info, "sm_count": sms, "rounds": args.rounds, "hbm_bytes_per_s": HBM_BYTES_PER_S,
              "fp32_per_tap_output": FP32_PER_TAP_OUTPUT, "points": []}
    for name, kind, S, P, ntaps, up, down, capture, iters in SHAPES:
        if name not in args.shapes:
            continue
        h = signal.firwin(ntaps, 0.8 / max(up, down))
        hp = -(-ntaps // up)
        nin = P if kind == "rx" else P * down // up
        with Bank(ctx, S, P) as fb, Bank(ctx, S, P) as sb, Fir(ctx, S, h, up, down) as ff, \
                Fir(ctx, S, h, up, down) as sf:
            nout = ff.output_frames(nin)
            full = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
            if kind == "rx":
                chan = torch.zeros(S * nout * 2, dtype=torch.float32, device="cuda")
                if capture == "ingested":
                    i2s = torch.randint(-2**31, 2**31 - 1, (S * P * 2,), dtype=torch.int32, device="cuda")
                    fb.ingest(0, S, i2s.data_ptr())
                    sb.ingest(0, S, i2s.data_ptr())
                dc, df = chan.data_ptr(), full.data_ptr()

                def split():
                    sb.read(df, st)
                    sf.apply(df, P, dc, st)
                forms = {"fused": lambda: fb.read_fir(ff, dc, st), "split": split}
            else:
                chan = torch.randn(S * nin * 2, dtype=torch.float32, device="cuda")
                dc, df = chan.data_ptr(), full.data_ptr()

                def split():
                    sf.apply(dc, nin, df, st)
                    sb.write(df, 0, None, 0, st)
                forms = {"fused": lambda: fb.write_fir(ff, dc, nin, 0, None, 0, st), "split": split}
            torch.cuda.synchronize()  # the calls run on another stream
            times = timed_pair(forms, side, iters, args.rounds)
            fused_bytes, split_bytes = traffic(kind, S, P, nin, nout, hp)
            fp32 = FP32_PER_TAP_OUTPUT * hp * S * nout / (sms * FP32_LANES_PER_SM * info["max_sm_clock_mhz"] * 1e6) * 1e6
            point = {"shape": name, "side": kind, "streams": S, "period": P, "taps": ntaps, "up": up, "down": down,
                     "capture": capture, "frames_in": nin, "frames_out": nout, "fp32_bound_us": fp32}
            for k, nbytes in (("fused", fused_bytes), ("split", split_bytes)):
                before = ctx.counter("launches")
                forms[k]()
                side.synchronize()
                hbm = nbytes / HBM_BYTES_PER_S * 1e6
                us = statistics.median(times[k])
                point[k] = {"us_per_call": us, "min_us": min(times[k]), "max_us": max(times[k]),
                            "launches_per_call": ctx.counter("launches") - before, "bytes": nbytes,
                            "hbm_bound_us": hbm, "bound": "hbm" if hbm >= fp32 else "fp32",
                            "achieved_over_bound": us / max(hbm, fp32)}
            for k in forms:
                point[k]["profiled_kernel_us"] = kernel_breakdown(forms[k], side, 5)
            point["fused_over_split"] = point["fused"]["us_per_call"] / point["split"]["us_per_call"]
            result["points"].append(point)
            print(json.dumps(point), flush=True)
            del full, chan
            torch.cuda.empty_cache()
    ctx.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
