#!/usr/bin/env python
"""BASELINE config 4 as one launch: sxgpu_bank_repeat against sxgpu_bank_read + sxgpu_bank_write.

For S streams x 256 frames, times one repeater iteration (read 256, timed write of the same
block at +768 frames) for the two-call form and for every schedule of the one-launch form
(option bank_repeat_variant), per launch and replayed from a CUDA graph,
and checks after every point that the constant-latency property still holds.

    python tools/sweep_bank_repeat.py --out gpurun_out/sweep_bank_repeat.json
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

from sxxcvr_b200 import Bank, Context  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="gpurun_out/sweep_bank_repeat.json")
    ap.add_argument("--streams", type=int, nargs="*", default=[64, 1024, 4096, 8192, 16384, 65536])
    ap.add_argument("--iters", type=int, default=200)
    args = ap.parse_args()

    ctx = Context(0)
    side = torch.cuda.Stream()
    torch.cuda.set_stream(side)
    st = side.cuda_stream
    lat = 10_240_000
    P = 256
    out = {"period": P, "iters": args.iters, "points": []}

    def timed(fn):
        """(sustained ms per call over `iters` back-to-back calls, median of 20 isolated calls)"""
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(side)
        for _ in range(args.iters):
            fn()
        b.record(side)
        torch.cuda.synchronize()
        sustained = a.elapsed_time(b) / args.iters
        lone = []
        for _ in range(20):
            a.record(side)
            fn()
            b.record(side)
            torch.cuda.synchronize()
            lone.append(a.elapsed_time(b))
        return sustained, statistics.median(lone)

    for S in args.streams:
        cf = torch.empty(S * P * 2, dtype=torch.float32, device="cuda")
        schedules = [("read+write", None, 0)]
        for variant in (0, 1, 2, 4, 100):
            schedules.append(("repeat", variant, 0))
        for name, variant, ctas in schedules:
            if variant is not None:
                ctx.set_option("bank_repeat_variant", variant)
            with Bank(ctx, S, P, 75000.0, 0.0, 1) as bank:
                if name == "repeat":
                    it = lambda: bank.repeat(cf.data_ptr(), lat, st)  # noqa: E731
                else:
                    def it():
                        bank.read(cf.data_ptr(), st)
                        bank.write(cf.data_ptr(), 4, None, lat, st)
                ms, lone = timed(it)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=side):
                    it()
                gms, glone = timed(g.replay)
                _, rxp, txp = bank.positions(st)
                ok = bool(((txp - rxp) == 768).all())
            rec = {"streams": S, "schedule": name, "bank_repeat_variant": variant, "ctas_per_sm": ctas,
                   "us_per_iteration": ms * 1e3, "us_lone": lone * 1e3,
                   "graph_us_per_iteration": gms * 1e3, "graph_us_lone": glone * 1e3,
                   "msps_rx_plus_tx": 2 * S * P / ms / 1e3, "graph_msps_rx_plus_tx": 2 * S * P / gms / 1e3,
                   "gbs_of_40B_per_frame": 40 * S * P / ms / 1e6,
                   "hbm_gbs_written_24B_per_frame": (24 * S * P / ms / 1e6) if name == "repeat" else None, "constant_latency_holds": ok}
            out["points"].append(rec)
            print(f"S={S:6d} {name:10s} variant={variant}: {ms*1e3:8.1f} us "
                  f"({rec['msps_rx_plus_tx']:9.0f} Msps)  graph {gms*1e3:8.1f} us  latency ok={ok}", flush=True)
        del cf
    ctx.set_option("bank_repeat_variant", 0)
    ctx.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
