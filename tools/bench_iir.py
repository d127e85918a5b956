#!/usr/bin/env python
"""The repeater iteration with its channel filters, against the plain iteration and the split form.

For S streams x 256 frames and two 4-section filters, times per iteration, with CUDA events over
back-to-back warmed iterations on one bank:
    plain     Bank.repeat                                    (no filters)
    filtered  Bank.repeat_filtered(pre, post)                (one plan kernel + one data kernel)
    split     read, pre.apply, post.apply, write(HAS_TIME)   (what a caller without the fused path runs)
and the separate halves with one filter (pre), on a bank that is only read and one that is only
written (every burst of the latter lands at its last read's timestamp + 768 frames, which for a
bank never read is the same place of the ring each time):
    rx_filtered  Bank.read_filtered(pre)                     (one plan kernel + one data kernel)
    rx_split     read, pre.apply
    tx_filtered  Bank.write_filtered(pre, HAS_TIME)          (the caller's block left as it was)
    tx_split     pre.apply in place, write(HAS_TIME)
The seven modes alternate round by round and the median round is reported.  Beside each time,
the least time the shapes allow:
    HBM bound   algorithmic bytes / 7.7 TB/s (the B200's data-sheet bandwidth): 24 B/frame for the
                plain and the filtered iteration (capture slot, CF32 block, ring), 64 B/frame for the
                split form (read 16, two applies 16 each, write 16), 16 B/frame for a fused half
                (capture slot and CF32 block; CF32 block and ring) and 32 for a split one, plus each
                filter's state read and written once per iteration (16 B per section and stream each way)
    FP32 bound  9 FP32 instructions per section, component and frame (un-contracted transposed
                direct form II) / (SMs x 128 lanes x the card's maximum SM clock)
and achieved / max(bounds).  At 65536 x 256 the iteration writes 402 MB, above the 126 MB of L2;
at 4096 x 256 it is 25 MB and the split form's re-reads may come from L2.
The card's name, power limit and maximum SM clock are read in the same run.

    python tools/bench_iir.py --out bench_iir.json
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402
from scipy import signal  # noqa: E402

from sxxcvr_b200 import Bank, Context, Iir  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
FP32_LANES_PER_SM = 128
FLOPS_PER_SECTION_SAMPLE = 9
HAS_TIME = 4


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", "0"], capture_output=True, text=True)
    if q.returncode != 0:
        raise RuntimeError("nvidia-smi could not be queried: " + q.stderr)
    name, power, clock = [x.strip() for x in q.stdout.strip().split("\n")[0].split(",")]
    return {"name": name, "power_limit_w": float(power), "max_sm_clock_mhz": float(clock)}


def bounds(S, P, nsections, bytes_per_frame, sms, clock_mhz):
    hbm = (bytes_per_frame * S * P + 2 * 16 * nsections * S) / HBM_BYTES_PER_S
    fp32 = FLOPS_PER_SECTION_SAMPLE * nsections * 2 * S * P / (sms * FP32_LANES_PER_SM * clock_mhz * 1e6)
    return hbm * 1e6, fp32 * 1e6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="bench_iir.json", help="where the JSON result goes")
    ap.add_argument("--streams", type=int, nargs="*", default=[64, 4096, 65536])
    ap.add_argument("--period", type=int, default=256)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()

    info = card()
    ctx = Context(0)
    sms = ctx.info().sm_count
    side = torch.cuda.Stream()
    st = side.cuda_stream
    P = args.period
    lat = int(round(768 * 1e9 / 75000.0))
    sos_pre = signal.butter(8, 0.25, output="sos")
    sos_post = signal.cheby1(8, 1.0, 0.3, output="sos")
    nsec = sos_pre.shape[0] + sos_post.shape[0]
    nsec_half = sos_pre.shape[0]
    result = {"card": info, "sm_count": sms, "period": P, "iters_per_round": args.iters, "rounds": args.rounds,
              "filters": {"pre": "butter(8, 0.25), 4 sections", "post": "cheby1(8, 1 dB, 0.3), 4 sections",
                          "halves": "pre only"},
              "hbm_bytes_per_s": HBM_BYTES_PER_S, "points": []}
    for S in args.streams:
        with Bank(ctx, S, P, 75000.0, 1.0e-6, 7) as bank, Iir(ctx, S, sos_pre) as pre, Iir(ctx, S, sos_post) as post, \
                Bank(ctx, S, P, 75000.0, 1.0e-6, 7) as rx_bank, Bank(ctx, S, P, 75000.0, 1.0e-6, 7) as tx_bank:
            cf = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
            d = cf.data_ptr()

            def split():
                bank.read(d, st)
                pre.apply(d, P, st)
                post.apply(d, P, st)
                bank.write(d, HAS_TIME, None, lat, st)

            def rx_split():
                rx_bank.read(d, st)
                pre.apply(d, P, st)

            def tx_split():
                pre.apply(d, P, st)
                tx_bank.write(d, HAS_TIME, None, lat, st)

            modes = {
                "plain": lambda: bank.repeat(d, lat, st),
                "filtered": lambda: bank.repeat_filtered(d, pre, post, lat, st),
                "split": split,
                "rx_filtered": lambda: rx_bank.read_filtered(d, pre, st),
                "rx_split": rx_split,
                "tx_filtered": lambda: tx_bank.write_filtered(d, pre, HAS_TIME, None, lat, st),
                "tx_split": tx_split,
            }
            times = {m: [] for m in modes}
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for fn in modes.values():
                for _ in range(20):
                    fn()
            side.synchronize()
            for _ in range(args.rounds):
                for m, fn in modes.items():
                    a.record(side)
                    for _ in range(args.iters):
                        fn()
                    b.record(side)
                    b.synchronize()
                    times[m].append(a.elapsed_time(b) * 1e3 / args.iters)
            for m, bpf, ns in (("plain", 24, 0), ("filtered", 24, nsec), ("split", 64, nsec),
                               ("rx_filtered", 16, nsec_half), ("rx_split", 32, nsec_half),
                               ("tx_filtered", 16, nsec_half), ("tx_split", 32, nsec_half)):
                us = statistics.median(times[m])
                hbm, fp32 = bounds(S, P, ns, bpf, sms, info["max_sm_clock_mhz"])
                point = {"streams": S, "mode": m, "us_per_iteration": us, "min_us": min(times[m]), "max_us": max(times[m]),
                         "hbm_bound_us": hbm, "fp32_bound_us": fp32, "bound": "hbm" if hbm >= fp32 else "fp32",
                         "achieved_over_bound": us / max(hbm, fp32)}
                result["points"].append(point)
                print(json.dumps(point), flush=True)
            del cf
    ctx.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
