#!/usr/bin/env python
"""Hardware-scheduled CTAs ("direct": one tile per CTA) against the persistent schedules, through
the library's own entry points on one B200 (run under gpurun; results -> gpurun_out/<tag>.json).

  convert     RX / TX CF32 at 2^17 .. 2^29 frames: variant 4 (direct) vs 3 (bulk-async) vs 1 (vector, persistent)
  ext         CS16 / S16 extensions (12 B/frame) at 2^27 frames: 4 vs 3
  loopback    fused RX->TX: 2 (direct) vs 3 (bulk-async) vs 1 (vector, persistent), with and without the CF32 block
  batched     1 GiB as N blocks per launch: 2 (direct) vs 3 (bulk-async tiles) vs 1 (slices)
  bank        one repeater iteration: 600 / 604 (plan + data kernels) vs 100, per launch and from a CUDA graph,
              synthetic and ingested capture, S in {1024 .. 65536}
"""
import argparse
import json
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from sxxcvr_b200 import Bank, Context  # noqa: E402
from sxxcvr_b200.capi import Block  # noqa: E402

PEAK = 6553.0
try:
    PEAK = float(json.loads((ROOT / "MEASURED_PEAKS.json").read_text())["hbm_gbs"])
except Exception:
    pass


def timed(fn, side, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(side)
    for _ in range(reps):
        fn()
    b.record(side)
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps * 1e-3


def sweep_convert(ctx, side, out):
    st = side.cuda_stream
    rows = []
    nmax = 1 << 29
    src = torch.empty(2 * nmax, dtype=torch.int32, device="cuda")
    ctx.synth_frames(src.data_ptr(), 0, nmax, 1, st)
    cf = torch.empty(2 * nmax, dtype=torch.float32, device="cuda")
    for log2n in (17, 19, 21, 23, 25, 27, 29):
        n = 1 << log2n
        row = {"frames": n}
        reps = 200 if log2n <= 21 else 20 if log2n <= 27 else 6
        for v in (4, 3, 1):
            ctx.set_option("rx_variant", v)
            ctx.set_option("tx_variant", v)
            sec = timed(lambda: ctx.convert_rx_buffer(src.data_ptr(), 0, cf.data_ptr(), 0, n, st), side, reps)
            row[f"rx_v{v}_gbs"] = round(16 * n / sec / 1e9, 1)
            sec = timed(lambda: ctx.convert_tx_buffer(cf.data_ptr(), 0, src.data_ptr(), 0, n, 1e-6, st), side, reps)
            row[f"tx_v{v}_gbs"] = round(16 * n / sec / 1e9, 1)
            ctx.synth_frames(src.data_ptr(), 0, n, 1, st)
        rows.append(row)
        print(json.dumps(row), flush=True)
    ctx.set_option("rx_variant", 0)
    ctx.set_option("tx_variant", 0)
    out["convert"] = rows
    del src, cf


def sweep_ext(ctx, side, out):
    st = side.cuda_stream
    n = 1 << 27
    wide = torch.empty(2 * n, dtype=torch.int32, device="cuda")
    narrow = torch.empty(2 * n, dtype=torch.int16, device="cuda")
    ctx.synth_frames(wide.data_ptr(), 0, n, 1, st)
    ops = {
        "rx_cs16": lambda: ctx.convert_rx_buffer_cs16(wide.data_ptr(), 0, narrow.data_ptr(), 0, n, st),
        "tx_cs16": lambda: ctx.convert_tx_buffer_cs16(narrow.data_ptr(), 0, wide.data_ptr(), 0, n, 1e-6, st),
        "rx_s16": lambda: ctx.convert_rx_buffer_s16(narrow.data_ptr(), 0, wide.data_ptr(), 0, n, st),
        "tx_s16": lambda: ctx.convert_tx_buffer_s16(wide.data_ptr(), 0, narrow.data_ptr(), 0, n, 1e-6, st),
    }
    for fn in ops.values():
        timed(fn, side, 5)
    rows = []
    for v in (4, 3):
        ctx.set_option("rx_variant", v)
        ctx.set_option("tx_variant", v)
        row = {"variant": v}
        for name, fn in ops.items():
            sec = timed(fn, side, 10)
            row[name + "_gbs"] = round(12 * n / sec / 1e9, 1)
            row[name + "_frac"] = round(12 * n / sec / 1e9 / PEAK, 3)
        rows.append(row)
        print(json.dumps(row), flush=True)
    ctx.set_option("rx_variant", 0)
    ctx.set_option("tx_variant", 0)
    out["extensions_12B_per_frame"] = rows


def sweep_loopback(ctx, side, out):
    st = side.cuda_stream
    rows = []
    for log2n in (21, 24, 27):
        n = 1 << log2n
        src = torch.empty(2 * n, dtype=torch.int32, device="cuda")
        ctx.synth_frames(src.data_ptr(), 0, n, 1, st)
        mid = torch.empty(2 * n, dtype=torch.float32, device="cuda")
        dst = torch.empty(2 * n, dtype=torch.int32, device="cuda")
        row = {"frames": n}
        for v in (2, 3, 1):
            ctx.set_option("loopback_variant", v)
            sec = timed(lambda: ctx.convert_loopback(src.data_ptr(), mid.data_ptr(), dst.data_ptr(), n, 1e-6, st), side, 20)
            row[f"v{v}_24B_gbs"] = round(24 * n / sec / 1e9, 1)
            sec = timed(lambda: ctx.convert_loopback(src.data_ptr(), None, dst.data_ptr(), n, 1e-6, st), side, 20)
            row[f"v{v}_16B_gbs"] = round(16 * n / sec / 1e9, 1)
        ctx.set_option("loopback_variant", 0)
        rows.append(row)
        print(json.dumps(row), flush=True)
    out["loopback"] = rows


def sweep_batched(ctx, side, out):
    st = side.cuda_stream
    total = 1 << 27
    src = torch.empty(2 * total, dtype=torch.int32, device="cuda")
    ctx.synth_frames(src.data_ptr(), 0, total, 1, st)
    cf = torch.empty(2 * total, dtype=torch.float32, device="cuda")
    dst = torch.empty(2 * total, dtype=torch.int32, device="cuda")
    rows = []
    for log2n in (17, 19, 21, 23, 25, 27):
        n = 1 << log2n
        nb = total // n
        rx_blocks = [Block(src.data_ptr() + 8 * n * b, cf.data_ptr() + 8 * n * b, n, 0.0, 0) for b in range(nb)]
        tx_blocks = [Block(cf.data_ptr() + 8 * n * b, dst.data_ptr() + 8 * n * b, n, 1e-6, 0) for b in range(nb)]
        d_rx = torch.from_numpy(np.frombuffer(bytes((Block * nb)(*rx_blocks)), dtype=np.uint8).copy()).cuda()
        d_tx = torch.from_numpy(np.frombuffer(bytes((Block * nb)(*tx_blocks)), dtype=np.uint8).copy()).cuda()
        row = {"shape": f"{nb} x {8 * n >> 20} MiB", "blocks": nb, "frames_per_block": n}
        for v in (2, 3, 1):
            ctx.set_option("batch_variant", v)
            for direction, d_list in (("rx", d_rx), ("tx", d_tx)):
                sec = timed(lambda: ctx.convert_batch(direction, d_list.data_ptr(), on_device=True, max_length=n,
                                                      stream=st, nblocks=nb), side, 10)
                row[f"{direction}_v{v}_gbs"] = round(16 * total / sec / 1e9, 1)
            if v == 2:
                sec = timed(lambda: ctx.convert_batch("rx", rx_blocks, stream=st), side, 5)
                row["rx_v2_host_list_gbs"] = round(16 * total / sec / 1e9, 1)
        ctx.set_option("batch_variant", 0)
        row["rx_v2_frac"] = round(row["rx_v2_gbs"] / PEAK, 3)
        row["tx_v2_frac"] = round(row["tx_v2_gbs"] / PEAK, 3)
        rows.append(row)
        print(json.dumps(row), flush=True)
    out["batched"] = rows


def sweep_bank(ctx, side, out):
    st = side.cuda_stream
    P, rate = 256, 75000.0
    lat = int(round(768 * 1e9 / rate))
    rows = []
    for S in (1024, 4096, 16384, 65536):
        cf = torch.empty(S * P * 2, dtype=torch.float32, device="cuda")
        row = {"streams": S}
        for variant in (0, 600, 604, 100, 201 if S <= 4096 else 2):
            ctx.set_option("bank_repeat_variant", variant)
            with Bank(ctx, S, P, rate, 0.0, 7) as bank:
                sec = timed(lambda: bank.repeat(cf.data_ptr(), lat, st), side, 200, warm=5)
                g = torch.cuda.CUDAGraph()
                torch.cuda.synchronize()
                with torch.cuda.graph(g, stream=side):
                    bank.repeat(cf.data_ptr(), lat, st)
                gsec = timed(g.replay, side, 200, warm=3)
                _, rxp, txp = bank.positions(st)
                assert ((txp - rxp) == 768).all()
            row[f"v{variant}_us"] = round(sec * 1e6, 2)
            row[f"v{variant}_graph_us"] = round(gsec * 1e6, 2)
        for variant in (0, 600, 604, 100):
            ctx.set_option("bank_repeat_variant", variant)
            with Bank(ctx, S, P, rate, 0.0, 7) as bank:
                bank.ingest(0, 0, None, st)
                sec = timed(lambda: bank.repeat(cf.data_ptr(), lat, st), side, 200, warm=5)
            row[f"external_v{variant}_us"] = round(sec * 1e6, 2)
        ctx.set_option("bank_repeat_variant", 0)
        row["v600_graph_write_gbs"] = round(24 * S * P / (row["v600_graph_us"] * 1e-6) / 1e9, 1)
        row["v604_graph_write_gbs"] = round(24 * S * P / (row["v604_graph_us"] * 1e-6) / 1e9, 1)
        row["external_v600_hbm_gbs"] = round(24 * S * P / (row["external_v600_us"] * 1e-6) / 1e9, 1)
        # the two-call form (read, then write) beside it
        with Bank(ctx, S, P, rate, 0.0, 7) as bank:
            def two():
                bank.read(cf.data_ptr(), st)
                bank.write(cf.data_ptr(), 4, None, lat, st)
            row["two_calls_us"] = round(timed(two, side, 200, warm=5) * 1e6, 2)
        rows.append(row)
        print(json.dumps(row), flush=True)
    out["bank_repeat"] = rows


def sweep_warp(ctx, side, out):
    """Warp-per-stream kernels (the bank's separate read / write calls, batches of period-sized
    blocks): persistent grid of 8 CTAs per SM against one CTA per eight streams."""
    st = side.cuda_stream
    P, rate = 256, 75000.0
    lat = int(round(768 * 1e9 / rate))
    rows = []
    for S in (4096, 16384, 65536):
        cf = torch.empty(S * P * 2, dtype=torch.float32, device="cuda")
        src = torch.empty(S * P * 2, dtype=torch.int32, device="cuda")
        ctx.synth_frames(src.data_ptr(), 0, S * P, 1, st)
        blocks = [Block(src.data_ptr() + 8 * P * b, cf.data_ptr() + 8 * P * b, P, 0.0, 0) for b in range(S)]
        d_list = torch.from_numpy(np.frombuffer(bytes((Block * S)(*blocks)), dtype=np.uint8).copy()).cuda()
        row = {"streams": S}
        for cap in (8, 4, 0):
            ctx.set_option("warp_ctas_per_sm", cap)
            with Bank(ctx, S, P, rate, 0.0, 7) as bank:
                def two():
                    bank.read(cf.data_ptr(), st)
                    bank.write(cf.data_ptr(), 4, None, lat, st)
                row[f"two_calls_cap{cap}_us"] = round(timed(two, side, 200, warm=5) * 1e6, 2)
            sec = timed(lambda: ctx.convert_batch("rx", d_list.data_ptr(), on_device=True, max_length=P, stream=st, nblocks=S),
                        side, 200, warm=5)
            row[f"batch_rx_cap{cap}_us"] = round(sec * 1e6, 2)
            row[f"batch_rx_cap{cap}_gbs"] = round(16 * S * P / sec / 1e9, 1)
        ctx.set_option("warp_ctas_per_sm", 0)
        rows.append(row)
        print(json.dumps(row), flush=True)
    out["warp_per_stream"] = rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="convert,ext,loopback,batched,bank")
    ap.add_argument("--tag", default="sweep_direct")
    args = ap.parse_args()
    only = set(args.only.split(","))
    out = {"peak_gbs": PEAK}
    ctx = Context(0)
    side = torch.cuda.Stream()
    torch.cuda.set_stream(side)
    for name, fn in (("convert", sweep_convert), ("ext", sweep_ext), ("loopback", sweep_loopback),
                     ("batched", sweep_batched), ("bank", sweep_bank), ("warp", sweep_warp)):
        if name in only:
            fn(ctx, side, out)
            torch.cuda.empty_cache()
    ctx.close()
    (ROOT / "gpurun_out").mkdir(exist_ok=True)
    (ROOT / "gpurun_out" / f"{args.tag}.json").write_text(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
