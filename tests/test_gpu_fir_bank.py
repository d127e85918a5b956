"""-m gpu: the bank's separate read and write calls with a FIR filter or resampler fused in
(sxgpu_bank_read_fir, sxgpu_bank_write_fir) against the numpy restatement in tests/sxfir.py and
against twin banks and twin filters that run the same sequence unfused: read then Fir.apply, or
Fir.apply into a scratch block then write.  Everything bit for bit."""
import numpy as np
import pytest

import sxfir
import sxtest
from test_gpu_fir import FACTORS, design, same_bits
from test_gpu_iir import latency_ns
from test_gpu_iir_halves import HAS_TIME, RATE, assert_same_bank, write_times

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def out_buffer(S, n):
    return torch.zeros(max(2, 2 * S * n), dtype=torch.float32, device="cuda")


def as_frames(t, S, n):
    return t[:2 * S * n].cpu().numpy().view(np.complex64).reshape(S, n)


def same_state(f, g, st):
    (h1, p1), (h2, p2) = f.state(st), g.state(st)
    return p1 == p2 and same_bits(h1, h2)


def synth_rx(oracle, S, first, P, seed):
    frames = np.concatenate([sxtest.synth_frames(oracle, first, P, seed=seed + s) for s in range(S)])
    return sxtest.oracle_rx(oracle, frames).view(np.complex64).reshape(S, P)


# A partial CTA, and both sides of bank_is_large.
@pytest.mark.parametrize("S,P", [(1, 2), (5, 34), (63, 256), (2100, 256), (32768 + 3, 64), (65536, 256)])
@pytest.mark.parametrize("ntaps,up,down", FACTORS)
def test_read_fir_matches_the_restatement(ctx, oracle, S, P, ntaps, up, down):
    from sxxcvr_b200 import Bank, Fir
    h = design(ntaps, up, down)
    ref = sxfir.Stream(h, up, down, S)
    side = torch.cuda.Stream()
    st = side.cuda_stream
    with Bank(ctx, S, P, RATE, 1.0e-6, 43) as bank, Bank(ctx, S, P, RATE, 1.0e-6, 43) as plain, \
            Fir(ctx, S, h, up, down) as F:
        out = out_buffer(S, -(-P * up // down))
        cf_plain = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        for it in range(3):
            want_n = sxfir.output_frames(ref.fed, P, up, down)
            with torch.cuda.stream(side):
                n = bank.read_fir(F, out.data_ptr(), st)
                plain.read(cf_plain.data_ptr(), st)
            side.synchronize()
            assert n == want_n, it
            assert same_bits(as_frames(out, S, n), ref.feed(synth_rx(oracle, S, it * P, P, 43))), it
            hist, phase = F.state(st)
            assert phase == ref.phase and same_bits(hist, ref.hist), it
            for a, b in zip(bank.positions(st), plain.positions(st)):
                assert np.array_equal(a, b), it
            assert all(np.array_equal(a, b) for a, b in zip(bank.last_read(st), plain.last_read(st))), it


# A history longer than the period (4 096 taps at P = 64), calls that emit nothing (P = 2, down 8:
# 1, 0, 0, 0 frames), and one tap (hp = 1: no history).
@pytest.mark.parametrize("S,P,ntaps,up,down", [(2100, 256, 64, 1, 4), (32768 + 3, 64, 96, 3, 2), (37, 64, 4096, 1, 1),
                                               (5, 2, 64, 1, 8), (37, 256, 1, 1, 1)])
@pytest.mark.parametrize("capture", ["synthetic", "ingested"])
def test_read_fir_equals_read_then_apply(ctx, oracle, S, P, ntaps, up, down, capture):
    from sxxcvr_b200 import Bank, Fir
    rng = np.random.default_rng(S + P + ntaps)
    h = design(ntaps, up, down) if ntaps > 1 else np.array([0.7])
    side = torch.cuda.Stream()
    st = side.cuda_stream
    nmax = -(-P * up // down)
    with Bank(ctx, S, P, RATE, 1.0e-6, 5) as fused, Bank(ctx, S, P, RATE, 1.0e-6, 5) as split, \
            Fir(ctx, S, h, up, down) as F1, Fir(ctx, S, h, up, down) as F2:
        out1, out2 = out_buffer(S, nmax), out_buffer(S, nmax)
        cf = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        counts = []
        for it in range(4):
            with torch.cuda.stream(side):
                if capture == "ingested":
                    frames = torch.from_numpy(rng.integers(-2**31, 2**31, S * P * 2, dtype=np.int64).astype(np.int32)).cuda()
                    fused.ingest(0, S, frames.data_ptr(), st)
                    split.ingest(0, S, frames.data_ptr(), st)
                if it == 1:
                    fused.advance(70000, st)  # an overrun on the way
                    split.advance(70000, st)
                n1 = fused.read_fir(F1, out1.data_ptr(), st)
                split.read(cf.data_ptr(), st)
                n2 = F2.apply(cf.data_ptr(), P, out2.data_ptr(), st)
            side.synchronize()
            assert n1 == n2, it
            counts.append(n1)
            assert same_bits(as_frames(out1, S, n1), as_frames(out2, S, n2)), it
            for a, b in zip(fused.positions(st), split.positions(st)):
                assert np.array_equal(a, b), it
            assert all(np.array_equal(a, b) for a, b in zip(fused.last_read(st), split.last_read(st))), it
            assert same_state(F1, F2, st), it
        if down == 8:
            assert counts == [1, 0, 0, 0]
        # The capture slots: switched to ingested capture with nothing handed in, a plain read
        # converts what the last read left in them.
        cf1 = torch.zeros_like(cf)
        with torch.cuda.stream(side):
            fused.ingest(0, 0, None, st)
            split.ingest(0, 0, None, st)
            fused.read(cf1.data_ptr(), st)
            split.read(cf.data_ptr(), st)
        side.synchronize()
        assert same_bits(cf1.cpu().numpy(), cf.cpu().numpy())
        if capture == "synthetic":
            first = int(split.positions(st)[1][0]) - 2 * P  # the fused read's first frame
            rx = cf1.cpu().numpy().view(np.complex64).reshape(S, P)
            for s in (0, S - 1):
                assert same_bits(rx[s], synth_rx(oracle, 1, first, P, 5 + s)[0]), s


# ↑4 at P = 256 on both sides of bank_is_large, ↑3 ↓2 at P = 66 and at an odd P = 255, and 1/1.
WRITE_FILTERS = [(37, 256, 64, 4, 1), (32768 + 3, 256, 64, 4, 1), (37, 66, 96, 3, 2), (37, 255, 96, 3, 2),
                 (37, 64, 31, 1, 1)]


@pytest.mark.parametrize("S,P,ntaps,up,down", WRITE_FILTERS)
@pytest.mark.parametrize("case", ["mixed", "offset", "untimed", "late"])
def test_write_fir_equals_apply_then_write(ctx, S, P, ntaps, up, down, case):
    """write_fir(F) against F.apply into a scratch block and then write, on a twin bank with a twin
    filter.  `offset`: HAS_TIME with no timestamps, 769 frames after a plain read (blocks
    straddle); `untimed`: flags 0 through an underrun; `late`: every write dropped."""
    from sxxcvr_b200 import Bank, Fir
    rng = np.random.default_rng(S + P + up)
    h = design(ntaps, up, down)
    nin = P * down // up
    lat = latency_ns(769)
    side = torch.cuda.Stream()
    st = side.cuda_stream
    with Bank(ctx, S, P, RATE, 1.0e-6, 9) as fused, Bank(ctx, S, P, RATE, 1.0e-6, 9) as split, \
            Fir(ctx, S, h, up, down) as F1, Fir(ctx, S, h, up, down) as F2:
        assert F1.output_frames(nin) == P
        if case == "late":
            fused.advance(4 * P, st)
            split.advance(4 * P, st)
        cf_rx = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        tmp = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        for it in range(3):
            x = (0.5 * rng.standard_normal(S * nin * 2)).astype(np.float32)
            d_in = torch.from_numpy(x).cuda()
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
                fused.write_fir(F1, d_in.data_ptr(), nin, flags, t_ptr, lat, st)
                assert F2.apply(d_in.data_ptr(), nin, tmp.data_ptr(), st) == P
                split.write(tmp.data_ptr(), flags, t_ptr, lat, st)
            side.synchronize()
            assert same_bits(d_in.cpu().numpy(), x), it  # the caller's block is left as it was
            assert same_state(F1, F2, st), it
            assert_same_bank(fused, split, S, P, st, it)
        clock, _, txp = fused.positions(st)
        if case == "late":
            assert (txp == 0).all()                      # nothing was written ...
            out = torch.ones(S * P * 2, dtype=torch.int32, device="cuda")
            fused.drain(0, S, P, out.data_ptr(), st)
            side.synchronize()
            assert not out.any()
            assert F1.state(st)[0].any()                 # ... and the filter advanced all the same
        elif case == "mixed":
            kind = np.arange(S) % 4
            assert (txp[kind == 1] == 0).all() and (txp[kind != 1] > 0).all() and (txp[kind == 3] % P != 0).all()
        else:
            assert (txp > 0).all()


@pytest.mark.parametrize("S,P", [(2100, 256), (32768 + 3, 64)])
@pytest.mark.parametrize("latency_frames", [768, 769])
def test_halves_compose_around_channel_rate_dsp(ctx, S, P, latency_frames):
    """read_fir(F ↓4), then write_fir(G ↑4, HAS_TIME, NULL, offset) equals read, F.apply, G.apply,
    write on a twin bank with twin filters."""
    from sxxcvr_b200 import Bank, Fir
    f_taps, g_taps = design(64, 1, 4), design(48, 4, 1)
    lat = latency_ns(latency_frames)
    C = P // 4
    side = torch.cuda.Stream()
    st = side.cuda_stream
    with Bank(ctx, S, P, RATE, 1.0e-6, 3) as halves, Bank(ctx, S, P, RATE, 1.0e-6, 3) as whole, \
            Fir(ctx, S, f_taps, 1, 4) as F1, Fir(ctx, S, g_taps, 4, 1) as G1, \
            Fir(ctx, S, f_taps, 1, 4) as F2, Fir(ctx, S, g_taps, 4, 1) as G2:
        chan1, chan2 = out_buffer(S, C), out_buffer(S, C)
        cf = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        up = torch.zeros_like(cf)
        for it in range(3):
            with torch.cuda.stream(side):
                assert halves.read_fir(F1, chan1.data_ptr(), st) == C
                halves.write_fir(G1, chan1.data_ptr(), C, HAS_TIME, None, lat, st)
                whole.read(cf.data_ptr(), st)
                F2.apply(cf.data_ptr(), P, chan2.data_ptr(), st)
                G2.apply(chan2.data_ptr(), C, up.data_ptr(), st)
                whole.write(up.data_ptr(), HAS_TIME, None, lat, st)
            side.synchronize()
            assert same_bits(chan1.cpu().numpy(), chan2.cpu().numpy()), it
            assert same_state(F1, F2, st) and same_state(G1, G2, st), it
            assert_same_bank(halves, whole, S, P, st, it)
        _, rxp, txp = halves.positions(st)
        assert (txp - rxp == latency_frames).all()


@pytest.mark.parametrize("ntaps,capture,want", [(64, "synthetic", 3), (64, "ingested", 3), (1, "synthetic", 3),
                                                (1, "ingested", 2)])
def test_launch_counts(ctx, ntaps, capture, want):
    """plan + data kernel + the tail kernel when hp > 1 or the capture is synthetic; with nothing
    emitted (P = 2, ↓8, second call) the data kernel is left out.  The write: plan + data kernel +
    fir_history_kernel when hp > 1."""
    from sxxcvr_b200 import Bank, Fir
    S = 5
    h = design(ntaps, 1, 8) if ntaps > 1 else np.array([0.7])
    out = out_buffer(S, 256)
    i2s = torch.zeros(S * 256 * 2, dtype=torch.int32, device="cuda")

    def count(fn):
        before, rx, tx = ctx.counter("launches"), ctx.counter("frames_rx"), ctx.counter("frames_tx")
        fn()
        ctx.stream_sync()
        return ctx.counter("launches") - before, ctx.counter("frames_rx") - rx, ctx.counter("frames_tx") - tx

    with Bank(ctx, S, 256) as bank, Bank(ctx, S, 2) as tiny, Fir(ctx, S, h, 1, 8) as F, Fir(ctx, S, h, 1, 8) as Ft, \
            Fir(ctx, S, h, 8, 1) as G:
        if capture == "ingested":
            bank.ingest(0, S, i2s.data_ptr())
            tiny.ingest(0, S, i2s.data_ptr())
        assert count(lambda: bank.read_fir(F, out.data_ptr())) == (want, S * 256, 0)
        assert count(lambda: tiny.read_fir(Ft, out.data_ptr())) == (want, S * 2, 0)  # one frame
        assert Ft.output_frames(2) == 0
        assert count(lambda: tiny.read_fir(Ft, out.data_ptr())) == (want - 1, S * 2, 0)  # none
        assert count(lambda: bank.write_fir(G, out.data_ptr(), 32, HAS_TIME, None, latency_ns(768))) == \
            (3 if ntaps > 1 else 2, 0, S * 256)


def test_graph_replay_equals_direct_calls(ctx):
    """A captured read_fir(↓4) and write_fir(↑4) (period and nin multiples of down) replayed three
    times equal the direct calls on twins."""
    from sxxcvr_b200 import Bank, Fir
    S, P, C = 16, 256, 64
    f_taps, g_taps = design(64, 1, 4), design(48, 4, 1)
    lat = latency_ns(768)
    chan1, chan2 = out_buffer(S, C), out_buffer(S, C)
    with Bank(ctx, S, P, RATE, 1.0e-6, 77) as a, Bank(ctx, S, P, RATE, 1.0e-6, 77) as b, \
            Fir(ctx, S, f_taps, 1, 4) as F1, Fir(ctx, S, g_taps, 4, 1) as G1, \
            Fir(ctx, S, f_taps, 1, 4) as F2, Fir(ctx, S, g_taps, 4, 1) as G2:
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        before = ctx.counter("launches")
        with torch.cuda.graph(g, stream=side):
            st = torch.cuda.current_stream().cuda_stream
            a.read_fir(F1, chan1.data_ptr(), st)
            a.write_fir(G1, chan1.data_ptr(), C, HAS_TIME, None, lat, st)
        assert ctx.counter("launches") - before == 6
        for it in range(3):
            g.replay()
            b.read_fir(F2, chan2.data_ptr())
            b.write_fir(G2, chan2.data_ptr(), C, HAS_TIME, None, lat)
            torch.cuda.synchronize()
            ctx.stream_sync()
            assert same_bits(chan1.cpu().numpy(), chan2.cpu().numpy()), it
            assert same_state(F1, F2, None) and same_state(G1, G2, None), it
            assert_same_bank(a, b, S, P, None, it)


def test_invalid_arguments_are_refused(ctx):
    """Every refusal a bank that fits in memory can reach.  Two of the listed ones cannot be: the
    read's nstreams * nout * 8-byte overflow (nout <= 65 536 * 256 frames, nstreams < 2^32) and a
    data kernel of more than 2^31 - 1 CTAs (at most 512 per stream, so over 4 million streams of
    65 536-frame periods, a bank of more than 2 TB)."""
    from sxxcvr_b200 import Bank, Context, Fir
    from sxxcvr_b200.capi import ERR_INVALID, SxGpuError
    S, P = 5, 256
    buf = torch.zeros(S * P * 2 + 8, dtype=torch.float32, device="cuda")
    d = buf.data_ptr()
    c2 = Context(0)
    try:
        with Bank(ctx, S, P) as bank, Fir(ctx, S, design(64, 1, 3), 1, 3) as F, Fir(ctx, S, design(48, 4, 1), 4, 1) as G, \
                Fir(ctx, S + 1, design(64, 1, 3), 1, 3) as other, Fir(c2, S, design(64, 1, 3), 1, 3) as foreign:
            G.set_state(None, 0)
            F.set_state(None, 1)  # a phase a refused call must leave as it is
            launches, positions = ctx.counter("launches"), bank.positions()

            def refused(fn):
                with pytest.raises(SxGpuError) as e:
                    fn()
                assert e.value.code == ERR_INVALID
                assert ctx.counter("launches") == launches and F.state()[1] == 1 and G.state()[1] == 0
                assert all(np.array_equal(x, y) for x, y in zip(bank.positions(), positions))

            for f in (None, other, foreign):
                refused(lambda: bank.read_fir(f, d))
                refused(lambda: bank.write_fir(f, d, 64))
            refused(lambda: bank.read_fir(F, 0))
            refused(lambda: bank.read_fir(F, d + 4))
            refused(lambda: bank.write_fir(G, 0, 64))
            refused(lambda: bank.write_fir(G, d + 4, 64))
            refused(lambda: bank.write_fir(G, d, 1 << 62))  # 5 x 2^62 x 8 bytes overflows
            refused(lambda: bank.write_fir(G, d, 63))       # 252 frames, not one period
            refused(lambda: bank.write_fir(G, d, 65))
            refused(lambda: bank.write_fir(G, d, 0))
            # and the same calls with good arguments run
            frx, ftx = ctx.counter("frames_rx"), ctx.counter("frames_tx")
            assert F.output_frames(P) == 85 and bank.read_fir(F, d) == 85
            bank.write_fir(G, d, 64, HAS_TIME, None, latency_ns(768))
            ctx.stream_sync()
            assert ctx.counter("launches") - launches == 6
            assert ctx.counter("frames_rx") - frx == S * P and ctx.counter("frames_tx") - ftx == S * P
            assert F.state()[1] == (1 + P) % 3 and (bank.positions()[2] == 768 + P).all()
    finally:
        c2.close()
