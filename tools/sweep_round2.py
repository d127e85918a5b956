#!/usr/bin/env python
"""Round-2 measurements on one B200 (run under gpurun; results -> gpurun_out/r02_sweep.json).

  batched     1 GiB of RX (and TX) work as N blocks per launch, N x size in {1024 x 1 MiB ...
              16 x 64 MiB}, bulk-async tile walker against the round-1 slice kernel, and the single
              large block beside them
  loopback    fused RX->TX, bulk-async against vector accesses, with and without the CF32 block
  bank        one repeater iteration per launch: every schedule at S in {64 .. 65536}
  host        sxgpu_convert_rx_buffer_host: frames per call x caller memory x first-chunk size
  small       period-sized synchronous calls: completion by flag / stream sync / resident kernel
  duplex      an RX thread and a TX thread on one context (one lane per direction)
"""
import argparse
import ctypes
import json
import sys
import threading
import time
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


def sweep_batched(ctx, side, out):
    st = side.cuda_stream
    total = 1 << 27                      # frames: 1 GiB in, 1 GiB out
    src = torch.empty(2 * total, dtype=torch.int32, device="cuda")
    ctx.synth_frames(src.data_ptr(), 0, total, 1, st)
    cf = torch.empty(2 * total, dtype=torch.float32, device="cuda")
    dst = torch.empty(2 * total, dtype=torch.int32, device="cuda")
    rows = []
    sec = timed(lambda: ctx.convert_rx_buffer(src.data_ptr(), 0, cf.data_ptr(), 0, total, st), side, 20)
    rows.append({"shape": "1 x 1 GiB (single-block kernel)", "rx_gbs": 16 * total / sec / 1e9})
    sec = timed(lambda: ctx.convert_tx_buffer(cf.data_ptr(), 0, dst.data_ptr(), 0, total, 1e-6, st), side, 20)
    rows[-1]["tx_gbs"] = 16 * total / sec / 1e9
    ctx.set_option("bulk_contiguous", 1)     # what does one contiguous tile range per CTA cost by itself?
    sec = timed(lambda: ctx.convert_rx_buffer(src.data_ptr(), 0, cf.data_ptr(), 0, total, st), side, 20)
    rows[-1]["rx_contiguous_ranges_gbs"] = 16 * total / sec / 1e9
    sec = timed(lambda: ctx.convert_tx_buffer(cf.data_ptr(), 0, dst.data_ptr(), 0, total, 1e-6, st), side, 20)
    rows[-1]["tx_contiguous_ranges_gbs"] = 16 * total / sec / 1e9
    ctx.set_option("bulk_contiguous", 0)
    print(json.dumps(rows[-1]), flush=True)
    for log2n in (17, 19, 21, 23, 25):
        n = 1 << log2n
        nb = total // n
        rx_blocks = [Block(src.data_ptr() + 8 * n * b, cf.data_ptr() + 8 * n * b, n, 0.0, 0) for b in range(nb)]
        tx_blocks = [Block(cf.data_ptr() + 8 * n * b, dst.data_ptr() + 8 * n * b, n, 1e-6, 0) for b in range(nb)]
        arr_rx = (Block * nb)(*rx_blocks)
        arr_tx = (Block * nb)(*tx_blocks)
        d_rx = torch.from_numpy(np.frombuffer(bytes(arr_rx), dtype=np.uint8).copy()).cuda()
        d_tx = torch.from_numpy(np.frombuffer(bytes(arr_tx), dtype=np.uint8).copy()).cuda()
        row = {"shape": f"{nb} x {8 * n >> 20} MiB", "blocks": nb, "frames_per_block": n}
        for variant, name in ((0, "bulk"), (1, "slices")):
            ctx.set_option("batch_variant", variant)
            for direction, d_list in (("rx", d_rx), ("tx", d_tx)):
                sec = timed(lambda: ctx.convert_batch(direction, d_list.data_ptr(), on_device=True, max_length=n,
                                                      stream=st, nblocks=nb), side, 10)
                row[f"{direction}_{name}_gbs"] = 16 * total / sec / 1e9
                row[f"{direction}_{name}_frac"] = 16 * total / sec / 1e9 / PEAK
            if variant == 0:     # host-resident descriptor list: staging copy inside the call
                sec = timed(lambda: ctx.convert_batch("rx", rx_blocks, stream=st), side, 5)
                row["rx_bulk_host_list_gbs"] = 16 * total / sec / 1e9
        ctx.set_option("batch_variant", 0)
        rows.append(row)
        print(json.dumps(row), flush=True)
    out["batched"] = rows


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
        for variant, name in ((0, "bulk"), (1, "vector")):
            ctx.set_option("loopback_variant", variant)
            sec = timed(lambda: ctx.convert_loopback(src.data_ptr(), mid.data_ptr(), dst.data_ptr(), n, 1e-6, st), side, 20)
            row[f"{name}_24B_gbs"] = 24 * n / sec / 1e9
            sec = timed(lambda: ctx.convert_loopback(src.data_ptr(), None, dst.data_ptr(), n, 1e-6, st), side, 20)
            row[f"{name}_16B_gbs"] = 16 * n / sec / 1e9
        ctx.set_option("loopback_variant", 0)
        for tile, stages in ((2048, 4), (1024, 6)):
            ctx.set_option("bulk_tile", tile)
            ctx.set_option("bulk_stages", stages)
            for cps in (0, 1):
                ctx.set_option("ctas_per_sm", cps)
                sec = timed(lambda: ctx.convert_loopback(src.data_ptr(), mid.data_ptr(), dst.data_ptr(), n, 1e-6, st), side, 20)
                row[f"bulk_{tile}x{stages}_cps{cps}_24B_gbs"] = round(24 * n / sec / 1e9, 1)
        ctx.set_option("bulk_tile", 0)
        ctx.set_option("bulk_stages", 0)
        ctx.set_option("ctas_per_sm", 0)
        rows.append(row)
        print(json.dumps(row), flush=True)
    out["loopback"] = rows


def sweep_bank(ctx, side, out):
    st = side.cuda_stream
    P, rate = 256, 75000.0
    lat = int(round(768 * 1e9 / rate))
    rows = []
    for S in (4096, 16384, 65536):
        cf = torch.empty(S * P * 2, dtype=torch.float32, device="cuda")
        row = {"streams": S}
        for variant in (2, 100, 600):
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
        # frames from outside (sxgpu_bank_ingest): the capture slots are read, not synthesised
        for variant in (100, 202, 604):
            ctx.set_option("bank_repeat_variant", variant)
            with Bank(ctx, S, P, rate, 0.0, 7) as bank:
                bank.ingest(0, 0, None, st)
                sec = timed(lambda: bank.repeat(cf.data_ptr(), lat, st), side, 200, warm=5)
            row[f"external_v{variant}_us"] = round(sec * 1e6, 2)
        ctx.set_option("bank_repeat_variant", 0)
        ext = min((row[k], k) for k in row if k.startswith("external_"))
        row["external_best"] = ext[1]
        row["external_best_hbm_gbs"] = 24 * S * P / (ext[0] * 1e-6) / 1e9
        best = min((row[k], k) for k in row if k.endswith("_graph_us"))
        row["best"] = best[1]
        row["best_write_gbs"] = 24 * S * P / (best[0] * 1e-6) / 1e9
        rows.append(row)
        print(json.dumps(row), flush=True)
    out["bank_repeat"] = rows


def sweep_extensions(ctx, side, out):
    """CS16 stream format and S16 I2S frames (extensions, 12 B/frame): bulk shapes per conversion."""
    st = side.cuda_stream
    n = 1 << 27
    wide = torch.empty(2 * n, dtype=torch.int32, device="cuda")      # 8 B/frame side
    narrow = torch.empty(2 * n, dtype=torch.int16, device="cuda")    # 4 B/frame side
    ctx.synth_frames(wide.data_ptr(), 0, n, 1, st)
    ops = {
        "rx_cs16": lambda: ctx.convert_rx_buffer_cs16(wide.data_ptr(), 0, narrow.data_ptr(), 0, n, st),
        "tx_cs16": lambda: ctx.convert_tx_buffer_cs16(narrow.data_ptr(), 0, wide.data_ptr(), 0, n, 1e-6, st),
        "rx_s16": lambda: ctx.convert_rx_buffer_s16(narrow.data_ptr(), 0, wide.data_ptr(), 0, n, st),
        "tx_s16": lambda: ctx.convert_tx_buffer_s16(wide.data_ptr(), 0, narrow.data_ptr(), 0, n, 1e-6, st),
    }
    rows = []
    for fn in ops.values():      # first touch of the buffers and clock ramp: not part of any row
        timed(fn, side, 5)
    for tile, stages in ((0, 0), (2048, 4), (2048, 6), (3072, 4), (4096, 3)):
        ctx.set_option("bulk_tile", tile)
        ctx.set_option("bulk_stages", stages)
        for cps in (0, 1):
            ctx.set_option("ctas_per_sm", cps)
            row = {"tile": tile or "default", "stages": stages or "default", "ctas_per_sm": cps or "occupancy"}
            for name, fn in ops.items():
                sec = timed(fn, side, 10)
                row[name + "_gbs"] = round(12 * n / sec / 1e9, 1)
                row[name + "_frac"] = round(12 * n / sec / 1e9 / PEAK, 3)
            rows.append(row)
            print(json.dumps(row), flush=True)
    ctx.set_option("bulk_tile", 0)
    ctx.set_option("bulk_stages", 0)
    ctx.set_option("ctas_per_sm", 0)
    out["extensions_12B_per_frame"] = rows


def pinned(ctx, nbytes, dtype):
    addr = ctx.malloc_host(nbytes)
    return addr, torch.frombuffer((ctypes.c_char * nbytes).from_address(addr), dtype=dtype)


def sweep_host(ctx, out):
    rows = []
    big = 1 << 26
    a_in, h_in = pinned(ctx, 8 * big, torch.int32)
    a_out, h_out = pinned(ctx, 8 * big, torch.float32)
    h_in.random_(-2**31, 2**31 - 1)
    p_in = np.random.default_rng(1).integers(-2**31, 2**31, size=2 * big, dtype=np.int64).astype(np.int32)
    p_out = np.ones(2 * big, np.float32)

    def rate(fn, n):
        fn()
        reps = max(2, min(50, int((1 << 27) // n)))
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        return 8 * n / ((time.perf_counter() - t0) / reps) / 1e9

    for log2n in (16, 18, 19, 20, 21, 22, 24, 26):
        n = 1 << log2n
        row = {"frames": n}
        row["pinned_auto_gbs"] = round(rate(lambda: ctx.convert_rx_buffer_host(a_in, 0, a_out, 0, n), n), 2)
        ctx.set_option("host_mode", 1)
        for pmode in (1, 2):
            ctx.set_option("pipeline_mode", pmode)
            for out_mode in (1, 2):
                ctx.set_option("host_out_mode", out_mode)
                for chunk in (1 << 15, 1 << 16, 1 << 17, 1 << 18, 1 << 19, 1 << 20, 1 << 22):
                    if chunk * 2 <= n or chunk == 1 << 15:
                        ctx.set_option("host_chunk_frames", chunk)
                        row[f"pinned_p{pmode}_out{out_mode}_chunk{chunk}_gbs"] = round(
                            rate(lambda: ctx.convert_rx_buffer_host(a_in, 0, a_out, 0, n), n), 2)
        ctx.set_option("host_chunk_min_frames", 1 << 14)
        ctx.set_option("host_chunk_frames", 1 << 18)
        ctx.set_option("host_out_mode", 1)
        row["pinned_p2_ramp16k_to_256k_gbs"] = round(rate(lambda: ctx.convert_rx_buffer_host(a_in, 0, a_out, 0, n), n), 2)
        ctx.set_option("host_chunk_min_frames", 0)
        ctx.set_option("host_chunk_frames", 0)
        ctx.set_option("pipeline_mode", 0)
        ctx.set_option("host_mode", 0)
        for nt in (0, 1):
            ctx.set_option("bounce_nt", nt)
            ctx.set_option("bounce_threads", 8)
            row[f"pageable_out_8thr_nt{nt}_gbs"] = round(
                rate(lambda: ctx.convert_rx_buffer_host(a_in, 0, p_out.ctypes.data, 0, n), n), 2)
            row[f"pageable_in_8thr_nt{nt}_gbs"] = round(
                rate(lambda: ctx.convert_rx_buffer_host(p_in.ctypes.data, 0, a_out, 0, n), n), 2)
            row[f"pageable_both_8thr_nt{nt}_gbs"] = round(
                rate(lambda: ctx.convert_rx_buffer_host(p_in.ctypes.data, 0, p_out.ctypes.data, 0, n), n), 2)
        ctx.set_option("bounce_nt", 1)
        for threads in (1, 4, 8):
            ctx.set_option("bounce_threads", threads)
            row[f"pageable_both_{threads}thr_gbs"] = round(
                rate(lambda: ctx.convert_rx_buffer_host(p_in.ctypes.data, 0, p_out.ctypes.data, 0, n), n), 2)
            row[f"pageable_out_{threads}thr_gbs"] = round(
                rate(lambda: ctx.convert_rx_buffer_host(a_in, 0, p_out.ctypes.data, 0, n), n), 2)
            row[f"pageable_in_{threads}thr_gbs"] = round(
                rate(lambda: ctx.convert_rx_buffer_host(p_in.ctypes.data, 0, a_out, 0, n), n), 2)
        ctx.set_option("bounce_threads", 0)
        rows.append(row)
        print(json.dumps(row), flush=True)
    out["host_path_gbs_each_way"] = rows

    # duplex: RX thread + TX thread on one context, pinned buffers, 2^24 frames per call
    n = 1 << 24
    a_f, h_f = pinned(ctx, 8 * n, torch.float32)
    a_i, h_i = pinned(ctx, 8 * n, torch.int32)
    h_f.uniform_(-0.9, 0.9)
    res = {}

    def loop(fn, name, reps=8):
        fn()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        res[name] = 8 * n / ((time.perf_counter() - t0) / reps) / 1e9

    loop(lambda: ctx.convert_rx_buffer_host(a_in, 0, a_out, 0, n), "rx_alone")
    loop(lambda: ctx.convert_tx_buffer_host(a_f, 0, a_i, 0, n, 1e-6), "tx_alone")
    ts = [threading.Thread(target=loop, args=(lambda: ctx.convert_rx_buffer_host(a_in, 0, a_out, 0, n), "rx_duplex")),
          threading.Thread(target=loop, args=(lambda: ctx.convert_tx_buffer_host(a_f, 0, a_i, 0, n, 1e-6), "tx_duplex"))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    out["duplex_gbs_each_way_per_direction"] = {k: round(v, 2) for k, v in res.items()}
    print(json.dumps(out["duplex_gbs_each_way_per_direction"]), flush=True)

    # small calls through the C ABI (ctypes adds ~1.5 us per call on top of the native figure)
    small = {}
    for label, setup in (("flag", lambda: ctx.set_option("small_mode", 2)),
                         ("stream_sync", lambda: ctx.set_option("small_mode", 1)),
                         ("resident", lambda: ctx.set_option("resident_max_frames", 4096))):
        setup()
        for nf in (256, 1024, 4096, 16384, 65536):
            if label == "resident" and nf > 4096:
                continue
            for _ in range(10):
                ctx.convert_rx_buffer_host(a_in, 0, a_out, 0, nf)
            reps = 2000
            t0 = time.perf_counter()
            for _ in range(reps):
                ctx.convert_rx_buffer_host(a_in, 0, a_out, 0, nf)
            small[f"rx_{nf}_{label}_us"] = round((time.perf_counter() - t0) / reps * 1e6, 2)
        ctx.set_option("small_mode", 0)
        ctx.set_option("resident_max_frames", 0)
    out["small_calls_c_abi_via_ctypes"] = small
    print(json.dumps(small), flush=True)
    del h_in, h_out, h_f, h_i
    for a in (a_in, a_out, a_f, a_i):
        ctx.free_host(a)


def sweep_plugin(out):
    """Native read+write pair loops through the plugin, product against reference."""
    sys.path.insert(0, str(ROOT))
    import bench
    from sxxcvr_b200 import plugin
    product = plugin.Harness()
    ref = bench.reference_harness()
    rows = []
    ctx = Context(0)
    for n, iters in ((256, 5000), (1024, 3000), (4096, 2000), (65536, 200), (1 << 20, 20), (1 << 24, 4)):
        row = {"frames_per_call": n}

        def pair_us(h, kind, extra=""):
            s = bench.PluginStreams(h, n, 1, kind, extra, ctx)
            try:
                return round(s.run(iters, 3) * 1e6, 2)
            finally:
                s.close()

        row["reference_us"] = pair_us(ref, "pageable") if ref else None
        row["product_us"] = pair_us(product, "pageable", ", gpu=0")
        row["product_flag_us"] = pair_us(product, "pageable", ", gpu=0, lowlatency=0, sxgpu.small_mode=2")
        row["product_pinned_us"] = pair_us(product, "pinned", ", gpu=0")
        row["product_pin1_us"] = pair_us(product, "pin", ", gpu=0")
        if n <= 4096:
            row["product_lowlatency0_us"] = pair_us(product, "pageable", ", gpu=0, lowlatency=0")
            row["product_lowlatency1_us"] = pair_us(product, "pageable", ", gpu=0, lowlatency=1")
            row["product_lowlatency1_pinned_us"] = pair_us(product, "pinned", ", gpu=0, lowlatency=1")
        rows.append(row)
        print(json.dumps(row), flush=True)
    ctx.close()
    out["plugin_pairs"] = rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="batched,loopback,bank,host,plugin")
    ap.add_argument("--tag", default="r02_sweep")
    args = ap.parse_args()
    which = set(args.only.split(","))
    out = {"peak_gbs": PEAK}
    ctx = Context(0)
    side = torch.cuda.Stream()
    torch.cuda.set_stream(side)
    if "batched" in which:
        sweep_batched(ctx, side, out)
    if "loopback" in which:
        sweep_loopback(ctx, side, out)
    if "bank" in which:
        sweep_bank(ctx, side, out)
    if "ext" in which:
        sweep_extensions(ctx, side, out)
    if "host" in which:
        sweep_host(ctx, out)
    ctx.close()
    if "plugin" in which:
        sweep_plugin(out)
    Path(ROOT / "gpurun_out").mkdir(exist_ok=True)
    (ROOT / "gpurun_out" / (args.tag + ".json")).write_text(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
