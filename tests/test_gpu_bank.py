"""-m gpu: the HBM-resident stream bank (sxgpu_bank_*) against S independent driver=sx devices.

BASELINE config 4: S streams x (readStream 256 -> identity DSP -> writeStream 256 with HAS_TIME at
rx.timeNs + latency).  The comparator is the unmodified reference driver when oracle/_ref is
present, else the product's own host-side device (itself held to the reference's golden traces in
test_gpu_stream.py).  Everything an application could observe must agree: return codes, flags,
timestamps, CF32 sample bits, and the I2S words left in each stream's playback ring."""
import numpy as np
import pytest

import sxstream
import sxtest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

HAS_TIME = sxstream.HAS_TIME


def comparator():
    from sxxcvr_b200 import _build
    if sxstream.REF_LIB.exists():
        return sxstream.Harness(sxstream.REF_LIB), "reference"
    _build.build_soapy_module()
    return sxstream.Harness(sxstream.PRODUCT_LIB), "product-device"


# (advance_before, write_mode, offset_ns): write_mode in {"rx+", "untimed", "none"}
def script(rate):
    lat = int(round(768 * 1e9 / rate))
    s = [(0, "rx+", lat)] * 6
    s += [(70000, "rx+", lat)]                  # RX overrun; the TX side is now late as well
    s += [(0, "rx+", lat)] * 3
    s += [(0, "rx+", -1_000_000_000)]           # a burst timed a second in the past: dropped whole
    s += [(0, "rx+", lat)] * 2
    s += [(100000, "untimed", 0)]               # untimed write after a stall: underrun forward
    s += [(0, "untimed", 0)] * 2
    s += [(0, "rx+", int(2.5e9))]               # further ahead than the ring: forward-and-wait
    s += [(0, "none", 0), (0, "rx+", lat), (5, "rx+", lat)]
    return s


@pytest.mark.parametrize("nstreams,period,rate,threshold", [
    (3, 256, 75000.0, "0"),            # linear_repeater.py settings
    (5, 1000, 300000.0, "0.001"),      # ring of 65000 frames: not a power of two, odd wrap points
    (2, 4096, 32.0e6 / 1536, "0.5"),   # non-integer rate
    (4, 3, 600000.0, "0"),             # odd ring (65535), tiny blocks: frame-wide accesses only
])
def test_bank_matches_independent_devices(ctx, nstreams, period, rate, threshold):
    from sxxcvr_b200 import Bank
    h, kind = comparator()
    clock_arg = ", clock=32e6" if abs(rate * 1536 - 32.0e6) < 1 else ""
    steps = script(rate)
    thr2 = float(np.float32(float(threshold)) * np.float32(float(threshold)))

    # ---- comparator: S separate devices driven one call at a time -------------------------------
    devs = []
    for s in range(nstreams):
        d = h.device("driver=sx" + clock_arg)
        d.set_rate(rate)
        h.lib.sx_alsa_set_capture_seed(d.cap, sxtest.SEED + s)
        rx = d.setup(sxstream.RX, args=f"period={period}")
        tx = d.setup(sxstream.TX, args=f"threshold={threshold}, period={period}")
        assert d.activate(rx) == 0 and d.activate(tx) == 0
        devs.append((d, rx, tx))
    want = []
    for adv, mode, off in steps:
        row = []
        for d, rx, tx in devs:
            if adv:
                d.advance(adv)
            r, fl, t, buf = d.read(rx, period)
            w = None
            if mode == "rx+":
                w = d.write(tx, buf, period, HAS_TIME, t + off)
            elif mode == "untimed":
                w = d.write(tx, buf, period)
            row.append((r, fl, t, buf.copy(), w, d.pointers()))
        want.append(row)

    # ---- the bank: every stream per launch ------------------------------------------------------
    with Bank(ctx, nstreams, period, rate, thr2, sxtest.SEED) as bank:
        assert bank.ring == 65536 // period * period
        cf = torch.empty(nstreams * period * 2, dtype=torch.float32, device="cuda")
        for i, (adv, mode, off) in enumerate(steps):
            if adv:
                bank.advance(adv)
            bank.read(cf.data_ptr())
            ret, fl, t = bank.last_read()
            got_cf = cf.cpu().numpy().reshape(nstreams, 2 * period)
            if mode == "rx+":
                bank.write(cf.data_ptr(), HAS_TIME, None, off)
            elif mode == "untimed":
                bank.write(cf.data_ptr(), 0, None, 0)
            wret = bank.last_write() if mode != "none" else None
            clock, rxp, txp = bank.positions()
            for s in range(nstreams):
                r_, fl_, t_, buf_, w_, ptrs = want[i][s]
                assert (int(ret[s]), int(fl[s]), int(t[s])) == (r_, fl_, t_), (kind, i, s)
                assert np.array_equal(got_cf[s].view(np.uint32), buf_.view(np.uint32)), (kind, i, s)
                if w_ is not None:
                    assert int(wret[s]) == w_, (kind, i, s)
                # stub pointers: [capture hw, capture appl, playback hw, playback appl]
                assert (int(clock[s]), int(rxp[s]), int(clock[s]), int(txp[s])) == tuple(ptrs), (kind, i, s)

        # ---- what is left in the playback rings --------------------------------------------------
        clock, rxp, txp = bank.positions()
        for s, (d, rx, tx) in enumerate(devs):
            end = int(txp[s])
            start = max(0, end - bank.ring)
            n = end - start
            ring = bank.playback(s, start, n)
            ref = d.sink(start, n)
            assert np.array_equal(ring, ref), (kind, s, int(np.flatnonzero(ring != ref)[0]))
            assert np.count_nonzero(ref) > 0
    for d, _, _ in devs:
        d.close()


def test_bank_constant_latency_at_every_rate(ctx):
    """SURVEY.md Appendix C: at every legal rate the TX block lands exactly 768 frames after the
    RX block it answers, for every stream, forever."""
    from sxxcvr_b200 import Bank
    for rate in sxtest.RATES:
        lat = int(round(768 * 1e9 / rate))
        with Bank(ctx, 64, 256, rate, 0.0, 1) as bank:
            cf = torch.empty(64 * 512, dtype=torch.float32, device="cuda")
            for k in range(20):
                bank.read(cf.data_ptr())
                bank.write(cf.data_ptr(), HAS_TIME, None, lat)
                _, rxp, txp = bank.positions()
                assert (rxp == 256 * (k + 1)).all() and (txp == 256 * k + 768 + 256).all(), (rate, k)


@pytest.mark.parametrize("S", [4096, 16384])       # planned inside the data kernels / by plan kernels
def test_bank_large_and_values_against_oracle(ctx, oracle, S):
    from sxxcvr_b200 import Bank
    P = 256
    with Bank(ctx, S, P, 75000.0, 0.0, 77) as bank:
        cf = torch.empty(S * P * 2, dtype=torch.float32, device="cuda")
        for _ in range(3):
            bank.read(cf.data_ptr())
            bank.write(cf.data_ptr(), HAS_TIME, None, 10_240_000)
        got = cf.cpu().numpy().reshape(S, 2 * P)
        for s in (0, 1, 2047, S - 1):
            frames = sxtest.synth_frames(oracle, 2 * P, P, seed=77 + s)
            want_cf = sxtest.oracle_rx(oracle, frames)
            assert np.array_equal(got[s].view(np.uint32), want_cf.view(np.uint32))
            ring = bank.playback(s, 2 * P + 768, P)
            assert np.array_equal(ring, sxtest.oracle_tx(oracle, want_cf, 0.0))
            assert not bank.playback(s, 0, 768).any()          # silence before the first burst
        ret, fl, t = bank.last_read()
        assert (ret == P).all() and (fl == HAS_TIME).all() and (t == 6_826_667).all()


def test_asynchronous_entry_points_can_be_captured_into_a_cuda_graph(ctx, oracle):
    """The async entry points only enqueue work on the caller's stream, so a launch-bound inner
    loop (a converter call, a whole bank iteration) can be captured once and replayed."""
    from sxxcvr_b200 import Bank
    side = torch.cuda.Stream()
    st = side.cuda_stream
    n = 4096
    words = sxtest.rx_uniform(n, seed=8)
    src = torch.from_numpy(words).cuda()
    mid = torch.zeros(2 * n, dtype=torch.float32, device="cuda")
    dst = torch.zeros(2 * n, dtype=torch.int32, device="cuda")
    S, P = 64, 256
    with Bank(ctx, S, P, 75000.0, 0.0, 5) as bank:
        cf = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        with torch.cuda.stream(side):
            # warm up outside the capture (first-use work such as the occupancy query happens here)
            ctx.convert_rx_buffer(src.data_ptr(), 0, mid.data_ptr(), 0, n, st)
            ctx.convert_tx_buffer(mid.data_ptr(), 0, dst.data_ptr(), 0, n, 0.0, st)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            ctx.convert_rx_buffer(src.data_ptr(), 0, mid.data_ptr(), 0, n, st)
            ctx.convert_tx_buffer(mid.data_ptr(), 0, dst.data_ptr(), 0, n, 0.0, st)
            bank.read(cf.data_ptr(), st)
            bank.write(cf.data_ptr(), HAS_TIME, None, 10_240_000, st)
        mid.zero_(), dst.zero_()
        torch.cuda.synchronize()
        for _ in range(5):
            g.replay()
        torch.cuda.synchronize()
        want_mid = sxtest.oracle_rx(oracle, words)
        assert np.array_equal(mid.cpu().numpy().view(np.uint32), want_mid.view(np.uint32))
        assert np.array_equal(dst.cpu().numpy(), sxtest.oracle_tx(oracle, want_mid, 0.0))
        # nothing ran during capture; five replays = five bank iterations
        _, rxp, txp = bank.positions()
        assert (rxp == 5 * P).all() and (txp == 4 * P + 768 + P).all()
        got = cf.cpu().numpy().reshape(S, 2 * P)
        for s_ in (0, 63):
            want = sxtest.oracle_rx(oracle, sxtest.synth_frames(oracle, 4 * P, P, seed=5 + s_))
            assert np.array_equal(got[s_].view(np.uint32), want.view(np.uint32))


def test_context_refuses_to_die_before_its_banks():
    from sxxcvr_b200 import Bank, Context
    c = Context(0)
    bank = Bank(c, 4, 256, 75000.0, 0.0, 1)
    assert c.lib.sxgpu_destroy(c.handle) == -1          # SXGPU_ERR_INVALID, context still alive
    assert b"banks first" in c.lib.sxgpu_last_error(c.handle)
    bank.close()
    c.close()


def snapshot(bank, cf, nstreams):
    """Everything an application could observe of a bank: results, counters, CF32 block, rings."""
    ret, fl, t = bank.last_read()
    clock, rxp, txp = bank.positions()
    rings = []
    for s in range(nstreams):
        end = int(txp[s])
        start = max(0, end - bank.ring)
        rings.append((start, bank.playback(s, start, end - start)))
    return {"read": (ret.copy(), fl.copy(), t.copy()), "write": bank.last_write().copy(),
            "positions": (clock.copy(), rxp.copy(), txp.copy()), "cf": cf.cpu().numpy().view(np.uint32).copy(),
            "rings": rings}


def assert_same(a, b, where):
    for key in ("read", "positions"):
        for x, y in zip(a[key], b[key]):
            assert np.array_equal(x, y), (where, key)
    assert np.array_equal(a["write"], b["write"]), (where, "write")
    assert np.array_equal(a["cf"], b["cf"]), (where, "cf")
    for s, ((sa, ra), (sb, rb)) in enumerate(zip(a["rings"], b["rings"])):
        assert sa == sb and np.array_equal(ra, rb), (where, "ring", s)


@pytest.mark.parametrize("nstreams,period,rate,thr2", [
    (3, 256, 75000.0, 0.0),
    (37, 256, 75000.0, 1.0e-6),      # one whole group of 32 streams and a ragged one
    (5, 1000, 300000.0, 1.0e-6),     # ring of 65000 frames: blocks straddle the wrap at odd offsets
    (70, 3, 600000.0, 0.0),          # odd ring, tiny blocks: frame-wide accesses only
    (2, 4096, 32.0e6 / 1536, 0.25),
])
@pytest.mark.parametrize("variant", [0, 1, 2, 4, 100, 201, 202, 204, 600, 604])
def test_repeat_is_read_then_write(ctx, nstreams, period, rate, thr2, variant):
    """sxgpu_bank_repeat against the two calls it fuses, through overruns, late (discarded)
    bursts, far-ahead bursts (forward-and-wait with silence) and interleaved separate calls."""
    from sxxcvr_b200 import Bank
    lat = int(round(768 * 1e9 / rate))
    steps = [(0, lat)] * 5 + [(70000, lat)] + [(0, lat)] * 3 + [(0, -1_000_000_000)] + [(0, lat)] * 2
    steps += [(0, int(2.5e9)), (0, lat), (5, lat), (100000, lat), (0, lat)]
    if variant >= 200 and period % 2:
        pytest.skip("the register schedules need an even period")
    if variant >= 600 and period < 4:
        pytest.skip("the plan + data schedules need a period of at least four frames")
    ctx.set_option("bank_repeat_variant", variant)
    with Bank(ctx, nstreams, period, rate, thr2, sxtest.SEED) as two_calls, \
            Bank(ctx, nstreams, period, rate, thr2, sxtest.SEED) as fused:
        cf_a = torch.zeros(nstreams * period * 2, dtype=torch.float32, device="cuda")
        cf_b = torch.zeros_like(cf_a)
        for i, (adv, off) in enumerate(steps):
            if adv:
                two_calls.advance(adv)
                fused.advance(adv)
            two_calls.read(cf_a.data_ptr())
            two_calls.write(cf_a.data_ptr(), HAS_TIME, None, off)
            fused.repeat(cf_b.data_ptr(), off)
            assert_same(snapshot(two_calls, cf_a, nstreams), snapshot(fused, cf_b, nstreams), i)
            if i == 7:   # separate calls in between leave the fused path where it should be
                for bank, cf in ((two_calls, cf_a), (fused, cf_b)):
                    bank.read(cf.data_ptr())
                    bank.write(cf.data_ptr(), 0, None, 0)
        assert snapshot(fused, cf_b, nstreams)["rings"][0][1].any()
    ctx.set_option("bank_repeat_variant", 0)


@pytest.mark.parametrize("variant", [0, 1, 2, 4, 100, 201, 202, 204, 600, 604])
def test_repeat_large_bank_against_oracle(ctx, oracle, variant):
    from sxxcvr_b200 import Bank
    S, P = 16384 + 5, 256
    ctx.set_option("bank_repeat_variant", variant)
    with Bank(ctx, S, P, 75000.0, 0.0, 77) as bank:
        cf = torch.empty(S * P * 2, dtype=torch.float32, device="cuda")
        for _ in range(3):
            bank.repeat(cf.data_ptr(), 10_240_000)
        got = cf.cpu().numpy().reshape(S, 2 * P)
        for s in (0, 31, 32, 2047, S - 6, S - 1):
            frames = sxtest.synth_frames(oracle, 2 * P, P, seed=77 + s)
            want_cf = sxtest.oracle_rx(oracle, frames)
            assert np.array_equal(got[s].view(np.uint32), want_cf.view(np.uint32))
            assert np.array_equal(bank.playback(s, 2 * P + 768, P), sxtest.oracle_tx(oracle, want_cf, 0.0))
            assert not bank.playback(s, 0, 768).any()
        ret, fl, t = bank.last_read()
        assert (ret == P).all() and (fl == HAS_TIME).all() and (t == 6_826_667).all()
        _, rxp, txp = bank.positions()
        assert (rxp == 3 * P).all() and (txp == 2 * P + 768 + P).all()
    ctx.set_option("bank_repeat_variant", 0)


def test_far_future_timestamp_costs_nothing(ctx):
    """A timed write a million seconds ahead: the forward-and-wait loop of SoapySX.cpp:1043-1073
    would turn 3e8 times; the bank takes it in closed form and lands where the loop would."""
    from sxxcvr_b200 import Bank
    import time
    S, P, rate = 8, 256, 75000.0
    with Bank(ctx, S, P, rate, 0.0, 3) as bank:
        cf = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        bank.read(cf.data_ptr())
        far = int(1.0e15)                                   # nanoseconds: 7.5e10 frames ahead
        t0 = time.perf_counter()
        bank.write(cf.data_ptr(), HAS_TIME, None, far)
        clock, rxp, txp = bank.positions()
        assert time.perf_counter() - t0 < 5.0
        target = 7.5e10
        assert (np.abs(txp - P - target) < 2).all()          # the block sits at the requested counter value
        assert (clock == txp - bank.ring).all()             # the clock ran until the block fitted the ring


@pytest.mark.parametrize("variant", [0, 4, 100, 202, 600, 604])
def test_ingested_frames_replace_the_synthetic_capture(ctx, oracle, variant):
    """sxgpu_bank_ingest / sxgpu_bank_drain: frames handed in from outside go through the same
    bookkeeping and come out of the rings converted; values against the oracle."""
    from sxxcvr_b200 import Bank
    S, P, rate = 70, 256, 75000.0
    lat = int(round(768 * 1e9 / rate))
    rng = np.random.default_rng(5)
    ctx.set_option("bank_repeat_variant", variant)
    with Bank(ctx, S, P, rate, 1.0e-6, 9) as bank:
        cf = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        out = torch.zeros(S * P * 2, dtype=torch.int32, device="cuda")
        for it in range(4):
            frames = rng.integers(-2**31, 2**31, size=S * P * 2, dtype=np.int64).astype(np.int32)
            if it % 2 == 0:       # pageable host source, whole bank
                bank.ingest(0, S, frames.ctypes.data)
            else:                 # device source, in two parts
                d = torch.from_numpy(frames).cuda()
                bank.ingest(0, 32, d.data_ptr())
                bank.ingest(32, S - 32, d.data_ptr() + 32 * P * 8)
            if it < 2:
                bank.repeat(cf.data_ptr(), lat)
            else:
                bank.read(cf.data_ptr())
                bank.write(cf.data_ptr(), HAS_TIME, None, lat)
            bank.drain(0, S, P, out.data_ptr())
            ctx.stream_sync()
            want_cf = sxtest.oracle_rx(oracle, frames)
            assert np.array_equal(cf.cpu().numpy().view(np.uint32), want_cf.view(np.uint32)), it
            assert np.array_equal(out.cpu().numpy(), sxtest.oracle_tx(oracle, want_cf, 1.0e-6)), it
            _, rxp, txp = bank.positions()
            assert (rxp == P * (it + 1)).all() and (txp == P * it + 768 + P).all()
        # drain into pinned host memory: the kernel writes across PCIe itself
        addr = ctx.malloc_host(S * P * 8)
        try:
            bank.drain(3, 5, P, addr)
            ctx.stream_sync()
            import ctypes
            host = np.frombuffer((ctypes.c_char * (5 * P * 8)).from_address(addr), dtype=np.int32)
            assert np.array_equal(host, out.cpu().numpy()[3 * P * 2: 8 * P * 2])
        finally:
            ctx.free_host(addr)
    ctx.set_option("bank_repeat_variant", 0)


@pytest.mark.parametrize("latency_frames", [769, 770, 1023, 1])
@pytest.mark.parametrize("variant", [2, 100, 202, 600, 604])
def test_repeat_with_blocks_that_straddle_ring_slices(ctx, variant, latency_frames):
    """Write positions that are not multiples of the period (odd, and even but inside a slice of
    the time-major ring): every schedule against the two calls it fuses."""
    from sxxcvr_b200 import Bank
    S, P, rate = 37, 256, 75000.0
    lat = int(round(latency_frames * 1e9 / rate))
    ctx.set_option("bank_repeat_variant", variant)
    with Bank(ctx, S, P, rate, 1.0e-6, 11) as two_calls, Bank(ctx, S, P, rate, 1.0e-6, 11) as fused:
        cf_a = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        cf_b = torch.zeros_like(cf_a)
        for i in range(300):                       # more than one lap of the 65536-frame ring
            two_calls.read(cf_a.data_ptr())
            two_calls.write(cf_a.data_ptr(), HAS_TIME, None, lat)
            fused.repeat(cf_b.data_ptr(), lat)
            if i in (0, 1, 5, 255, 256, 257, 299):
                assert_same(snapshot(two_calls, cf_a, S), snapshot(fused, cf_b, S), i)
        _, rxp, txp = fused.positions()
        if latency_frames >= P:
            assert (txp - rxp == latency_frames).all()
        else:                       # a block timed before the end of its own read is late: dropped whole, every time
            assert (txp == 0).all() and (rxp == 300 * P).all()
    ctx.set_option("bank_repeat_variant", 0)


@pytest.mark.parametrize("cap", [0, 8])
def test_large_bank_default_schedules_and_grid_options(ctx, oracle, cap):
    """A large bank's default schedules -- decisions by one kernel, samples by the next, launched as
    its programmatic dependent -- for the fused iteration and for the separate read / write calls,
    against the warp-per-stream kernels (bank_split_variant = 1; persistent grid with cap 8, one
    CTA per eight streams with cap 0)."""
    from sxxcvr_b200 import Bank
    S, P, rate = 32768 + 37, 64, 75000.0
    lat = int(round(768 * 1e9 / rate))
    ctx.set_option("warp_ctas_per_sm", cap)
    ctx.set_option("bank_repeat_variant", 0)
    try:
        with Bank(ctx, S, P, rate, 1.0e-6, 5) as ref, Bank(ctx, S, P, rate, 1.0e-6, 5) as split, \
                Bank(ctx, S, P, rate, 1.0e-6, 5) as fused:
            cf = [torch.zeros(S * P * 2, dtype=torch.float32, device="cuda") for _ in range(3)]
            for it, adv in enumerate((0, 0, 70000, 0, 13, 0)):   # an overrun and a clock jump on the way
                if adv:
                    for bank in (ref, split, fused):
                        bank.advance(adv)
                ctx.set_option("bank_split_variant", 1)
                ref.read(cf[0].data_ptr())
                ref.write(cf[0].data_ptr(), HAS_TIME, None, lat)
                ctx.set_option("bank_split_variant", 0)
                split.read(cf[1].data_ptr())
                split.write(cf[1].data_ptr(), HAS_TIME, None, lat)
                fused.repeat(cf[2].data_ptr(), lat)
                _, _, txp = ref.positions()
                for other, c in ((split, cf[1]), (fused, cf[2])):
                    assert torch.equal(cf[0].view(torch.int32), c.view(torch.int32)), it
                    for x, y in zip(ref.positions(), other.positions()):
                        assert np.array_equal(x, y), it
                    for x, y in zip(ref.last_read(), other.last_read()):
                        assert np.array_equal(x, y), it
                    assert np.array_equal(ref.last_write(), other.last_write()), it
                    for s in (0, 1, 31, 32, 4095, 32767, 32768, S - 1):
                        end = int(txp[s])
                        start = max(0, end - 4 * P)
                        assert np.array_equal(ref.playback(s, start, end - start), other.playback(s, start, end - start)), (it, s)
            frames = sxtest.synth_frames(oracle, int(fused.positions()[1][S - 1]) - P, P, seed=5 + S - 1)
            assert np.array_equal(cf[2].view(torch.int32).cpu().numpy().reshape(S, 2 * P)[S - 1].view(np.uint32),
                                  sxtest.oracle_rx(oracle, frames).view(np.uint32))
            # the separate calls with an untimed write and with per-stream timestamps, ingested capture
            t_ns = torch.full((S,), lat, dtype=torch.int64, device="cuda") + torch.arange(S, device="cuda") % 3 * 1_000_000
            for flags, times in ((0, None), (HAS_TIME, t_ns.data_ptr())):
                for variant, bank, c in ((1, ref, cf[0]), (0, split, cf[1])):
                    ctx.set_option("bank_split_variant", variant)
                    bank.ingest(0, 0, None)
                    bank.read(c.data_ptr())
                    bank.write(c.data_ptr(), flags, times, 0)
                assert torch.equal(cf[0].view(torch.int32), cf[1].view(torch.int32))
                for x, y in zip(ref.positions(), split.positions()):
                    assert np.array_equal(x, y)
                assert np.array_equal(ref.last_write(), split.last_write())
                _, _, txp = ref.positions()
                for s in (0, 1, 2, 4095, S - 1):
                    end = int(txp[s])
                    start = max(0, end - 4 * P)
                    assert np.array_equal(ref.playback(s, start, end - start), split.playback(s, start, end - start)), s
    finally:
        ctx.set_option("warp_ctas_per_sm", 0)
        ctx.set_option("bank_split_variant", 0)
