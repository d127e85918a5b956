"""-m gpu: the bank's separate read and write calls with a channel filter fused in
(sxgpu_bank_read_filtered, sxgpu_bank_write_filtered) against the numpy restatement in
tests/sxiir.py and against twin banks that run the same sequence unfused: read then
Iir.apply, or a copy of the block filtered by Iir.apply then write.  Everything bit for bit."""
import numpy as np
import pytest

import sxiir
import sxtest
from test_gpu_iir import as_blocks, design, latency_ns, random_state, same_bits

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

HAS_TIME = 1 << 2
RATE = 75000.0


def ticks_ns(ticks):
    return np.round(np.asarray(ticks, np.float64) * 1e9 / RATE).astype(np.int64)


def assert_same_bank(a, b, S, P, st, where):
    """Positions, results and the rings of twin banks: the last two periods of every stream, and
    stream by stream the whole lap the ring still holds, forwarded-over silence included."""
    for x, y in zip(a.positions(st), b.positions(st)):
        assert np.array_equal(x, y), where
    assert all(np.array_equal(x, y) for x, y in zip(a.last_read(st), b.last_read(st))), where
    assert np.array_equal(a.last_write(st), b.last_write(st)), where
    out_a = torch.zeros(S * 2 * P * 2, dtype=torch.int32, device="cuda")
    out_b = torch.zeros_like(out_a)
    a.drain(0, S, 2 * P, out_a.data_ptr(), st)
    b.drain(0, S, 2 * P, out_b.data_ptr(), st)
    a.ctx.stream_sync(st)
    assert np.array_equal(out_a.cpu().numpy(), out_b.cpu().numpy()), where
    _, _, txp = a.positions(st)
    for s in sorted({0, 1, 2, 3, S // 2, S - 1}):
        end = int(txp[s])
        start = max(0, end - a.ring)
        assert np.array_equal(a.playback(s, start, end - start, st), b.playback(s, start, end - start, st)), (where, s)


# A partial CTA, a tail tile shorter than 32 frames, and both sides of bank_is_large.
@pytest.mark.parametrize("S,P", [(1, 2), (5, 34), (63, 256), (2100, 256), (32768 + 3, 64), (65536, 256)])
@pytest.mark.parametrize("nsections", [1, 4, 8])
def test_read_filtered_matches_the_restatement(ctx, oracle, S, P, nsections):
    from sxxcvr_b200 import Bank, Iir
    rng = np.random.default_rng(S * 10 + nsections)
    sos = design(nsections, nsections % 2)
    side = torch.cuda.Stream()
    st = side.cuda_stream
    with Bank(ctx, S, P, RATE, 1.0e-6, 43) as bank, Bank(ctx, S, P, RATE, 1.0e-6, 43) as plain, Iir(ctx, S, sos) as F:
        z = random_state(rng, nsections, S)
        F.set_state(z, st)
        cf = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        cf_plain = torch.zeros_like(cf)
        for it in range(3):
            with torch.cuda.stream(side):
                bank.read_filtered(cf.data_ptr(), F, st)
                plain.read(cf_plain.data_ptr(), st)
            side.synchronize()
            frames = np.concatenate([sxtest.synth_frames(oracle, it * P, P, seed=43 + s) for s in range(S)])
            rx = sxtest.oracle_rx(oracle, frames).view(np.complex64).reshape(S, P)
            want, z = sxiir.sosfilt(sos, rx, z)
            assert same_bits(as_blocks(cf, S, P), want), it
            for a, b in zip(bank.positions(st), plain.positions(st)):
                assert np.array_equal(a, b), it
            assert all(np.array_equal(a, b) for a, b in zip(bank.last_read(st), plain.last_read(st))), it
        assert same_bits(F.state(st), z)


@pytest.mark.parametrize("S,P", [(2100, 256), (32768 + 3, 64)])
@pytest.mark.parametrize("capture", ["synthetic", "ingested"])
def test_read_filtered_equals_read_then_apply(ctx, oracle, S, P, capture):
    from sxxcvr_b200 import Bank, Iir
    rng = np.random.default_rng(7)
    sos = design(3, 1)
    side = torch.cuda.Stream()
    st = side.cuda_stream
    with Bank(ctx, S, P, RATE, 1.0e-6, 5) as fused, Bank(ctx, S, P, RATE, 1.0e-6, 5) as split, \
            Iir(ctx, S, sos) as F1, Iir(ctx, S, sos) as F2:
        z = random_state(rng, 3, S)
        F1.set_state(z, st)
        F2.set_state(z, st)
        cf1 = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        cf2 = torch.zeros_like(cf1)
        for it in range(3):
            with torch.cuda.stream(side):
                if capture == "ingested":
                    frames = torch.from_numpy(rng.integers(-2**31, 2**31, S * P * 2, dtype=np.int64).astype(np.int32)).cuda()
                    fused.ingest(0, S, frames.data_ptr(), st)
                    split.ingest(0, S, frames.data_ptr(), st)
                if it == 1:
                    fused.advance(70000, st)  # an overrun on the way
                    split.advance(70000, st)
                fused.read_filtered(cf1.data_ptr(), F1, st)
                split.read(cf2.data_ptr(), st)
                F2.apply(cf2.data_ptr(), P, st)
            side.synchronize()
            assert same_bits(cf1.cpu().numpy(), cf2.cpu().numpy()), it
            for a, b in zip(fused.positions(st), split.positions(st)):
                assert np.array_equal(a, b), it
            assert all(np.array_equal(a, b) for a, b in zip(fused.last_read(st), split.last_read(st))), it
            assert same_bits(F1.state(st), F2.state(st)), it
        assert not same_bits(F1.state(st), z)
        # The capture slots: switched to ingested capture with nothing handed in, a plain read
        # converts what the last read left in them.
        for bank, cf in ((fused, cf1), (split, cf2)):
            with torch.cuda.stream(side):
                bank.ingest(0, 0, None, st)
                bank.read(cf.data_ptr(), st)
        side.synchronize()
        assert same_bits(cf1.cpu().numpy(), cf2.cpu().numpy())
        if capture == "synthetic":
            first = int(split.positions(st)[1][0]) - 2 * P  # the filtered read's first frame
            rx = as_blocks(cf1, S, P)
            for s in (0, S - 1):
                frames = sxtest.synth_frames(oracle, first, P, seed=5 + s)
                assert same_bits(rx[s], sxtest.oracle_rx(oracle, frames)), s


def write_times(case, S, P, clock, txp):
    """Per-stream timestamps for write_filtered's cases (None: the call takes none)."""
    if case == "mixed":
        kind = np.arange(S) % 4
        ticks = np.where(kind == 0, txp,                      # on time: right after what is queued
                np.where(kind == 1, clock - 3 * P,           # late: before what is playing now (dropped)
                np.where(kind == 2, txp + 3 * P,             # ahead: forwarded over, the gap silenced
                         txp + 37)))                          # ahead by a part of a period: straddles two slices
        return ticks_ns(ticks)
    if case == "late":
        return ticks_ns(clock - 1)
    return None


@pytest.mark.parametrize("S,P", [(37, 256), (32768 + 3, 64)])
@pytest.mark.parametrize("case", ["mixed", "offset", "untimed", "late"])
def test_write_filtered_equals_apply_then_write(ctx, S, P, case):
    """write_filtered(F) against a copy of the block filtered by F.apply and then written, on a
    twin bank with a twin filter.  `offset`: HAS_TIME with no timestamps, 769 frames after a plain
    read (blocks straddle); `untimed`: flags 0 through an underrun; `late`: every write dropped."""
    from sxxcvr_b200 import Bank, Iir
    rng = np.random.default_rng(S + P)
    sos = design(4, 0)
    lat = latency_ns(769)
    side = torch.cuda.Stream()
    st = side.cuda_stream
    with Bank(ctx, S, P, RATE, 1.0e-6, 9) as fused, Bank(ctx, S, P, RATE, 1.0e-6, 9) as split, \
            Iir(ctx, S, sos) as F1, Iir(ctx, S, sos) as F2:
        z = random_state(rng, 4, S)
        F1.set_state(z, st)
        F2.set_state(z, st)
        if case == "late":
            fused.advance(4 * P, st)
            split.advance(4 * P, st)
        cf_rx = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        for it in range(3):
            x = (0.5 * rng.standard_normal(S * P * 2)).astype(np.float32)
            cf = torch.from_numpy(x).cuda()
            clock, _, txp = fused.positions(st)
            times = write_times(case, S, P, clock, txp)
            d_times = torch.from_numpy(times).cuda() if times is not None else None
            flags = 0 if case == "untimed" else HAS_TIME
            with torch.cuda.stream(side):
                if case == "offset":
                    fused.read(cf_rx.data_ptr(), st)
                    split.read(cf_rx.data_ptr(), st)
                if case == "untimed" and it == 1:
                    fused.advance(5 * P + 3, st)  # the clock overtakes what was queued: an underrun
                    split.advance(5 * P + 3, st)
                t_ptr = d_times.data_ptr() if d_times is not None else None
                fused.write_filtered(cf.data_ptr(), F1, flags, t_ptr, lat, st)
                copy = cf.clone()
                F2.apply(copy.data_ptr(), P, st)
                split.write(copy.data_ptr(), flags, t_ptr, lat, st)
            side.synchronize()
            assert same_bits(cf.cpu().numpy(), x), it  # the caller's block is left as it was
            assert same_bits(F1.state(st), F2.state(st)), it
            assert_same_bank(fused, split, S, P, st, it)
        clock, _, txp = fused.positions(st)
        if case == "late":
            assert (txp == 0).all()                      # nothing was written ...
            out = torch.ones(S * P * 2, dtype=torch.int32, device="cuda")
            fused.drain(0, S, P, out.data_ptr(), st)
            side.synchronize()
            assert not out.any()
            assert not same_bits(F1.state(st), z)        # ... and the filter advanced all the same
        elif case == "mixed":
            kind = np.arange(S) % 4
            assert (txp[kind == 1] == 0).all() and (txp[kind != 1] > 0).all() and (txp[kind == 3] % P != 0).all()
        else:
            assert (txp > 0).all()


@pytest.mark.parametrize("S,P", [(2100, 256), (32768 + 3, 64)])
@pytest.mark.parametrize("latency_frames", [768, 769])
def test_halves_compose_to_the_filtered_iteration(ctx, S, P, latency_frames):
    """read_filtered(F), then write_filtered(G, HAS_TIME, NULL, offset) equals
    repeat_filtered(F, G, offset) on a twin bank with twin filters."""
    from sxxcvr_b200 import Bank, Iir
    rng = np.random.default_rng(latency_frames)
    sos_f, sos_g = design(4, 0), design(4, 1)
    lat = latency_ns(latency_frames)
    side = torch.cuda.Stream()
    st = side.cuda_stream
    with Bank(ctx, S, P, RATE, 1.0e-6, 3) as halves, Bank(ctx, S, P, RATE, 1.0e-6, 3) as whole, \
            Iir(ctx, S, sos_f) as F1, Iir(ctx, S, sos_g) as G1, Iir(ctx, S, sos_f) as F2, Iir(ctx, S, sos_g) as G2:
        zf, zg = random_state(rng, 4, S), random_state(rng, 4, S)
        for f, z in ((F1, zf), (F2, zf), (G1, zg), (G2, zg)):
            f.set_state(z, st)
        cf1 = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        cf2 = torch.zeros_like(cf1)
        for it in range(3):
            with torch.cuda.stream(side):
                halves.read_filtered(cf1.data_ptr(), F1, st)
                halves.write_filtered(cf1.data_ptr(), G1, HAS_TIME, None, lat, st)
                whole.repeat_filtered(cf2.data_ptr(), F2, G2, lat, st)
            side.synchronize()
            assert_same_bank(halves, whole, S, P, st, it)
            assert same_bits(F1.state(st), F2.state(st)) and same_bits(G1.state(st), G2.state(st)), it
        _, rxp, txp = halves.positions(st)
        assert (txp - rxp == latency_frames).all()


@pytest.mark.parametrize("S,P", [(37, 256), (32768 + 3, 64)])
def test_no_filter_is_the_plain_call(ctx, S, P):
    from sxxcvr_b200 import Bank
    lat = latency_ns(769)
    side = torch.cuda.Stream()
    st = side.cuda_stream
    with Bank(ctx, S, P, RATE, 1.0e-6, 21) as a, Bank(ctx, S, P, RATE, 1.0e-6, 21) as b:
        cf_a = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        cf_b = torch.zeros_like(cf_a)
        for it in range(3):
            with torch.cuda.stream(side):
                a.read_filtered(cf_a.data_ptr(), None, st)
                b.read(cf_b.data_ptr(), st)
                a.write_filtered(cf_a.data_ptr(), None, HAS_TIME, None, lat, st)
                b.write(cf_b.data_ptr(), HAS_TIME, None, lat, st)
            side.synchronize()
            assert same_bits(cf_a.cpu().numpy(), cf_b.cpu().numpy()), it
            assert_same_bank(a, b, S, P, st, it)


def test_invalid_arguments_are_refused(ctx):
    from sxxcvr_b200 import Bank, Context, Iir
    from sxxcvr_b200.capi import ERR_INVALID, SxGpuError
    good = design(2)

    def refused(fn):
        with pytest.raises(SxGpuError) as e:
            fn()
        assert e.value.code == ERR_INVALID

    S, P = 5, 256
    cf = torch.zeros(S * P * 2 + 8, dtype=torch.float32, device="cuda")
    d = cf.data_ptr()
    c2 = Context(0)
    try:
        with Bank(ctx, S, P) as bank, Bank(ctx, S, 255) as odd, Iir(ctx, S, good) as F, \
                Iir(ctx, S + 1, good) as other, Iir(c2, S, good) as foreign:
            for f in (F, None):
                refused(lambda: odd.read_filtered(d, f))
                refused(lambda: odd.write_filtered(d, f))
                refused(lambda: bank.read_filtered(d + 8, f))
                refused(lambda: bank.write_filtered(d + 8, f))
                refused(lambda: bank.read_filtered(0, f))
                refused(lambda: bank.write_filtered(0, f))
            for f in (other, foreign):
                refused(lambda: bank.read_filtered(d, f))
                refused(lambda: bank.write_filtered(d, f))
            # and the same calls with good arguments run, two launches each
            launches, frx, ftx = ctx.counter("launches"), ctx.counter("frames_rx"), ctx.counter("frames_tx")
            bank.read_filtered(d, F)
            bank.write_filtered(d, F, HAS_TIME, None, latency_ns(768))
            ctx.stream_sync()
            assert ctx.counter("launches") - launches == 4
            assert ctx.counter("frames_rx") - frx == S * P and ctx.counter("frames_tx") - ftx == S * P
            assert (bank.positions()[2] == 768 + P).all()
    finally:
        c2.close()
