"""-m gpu: the per-stream oscillators (sxgpu_nco_*) and the FIR halves with an oscillator fused in
(sxgpu_bank_read_ddc, sxgpu_bank_write_duc) against the numpy restatement in tests/sxnco.py and
against twin banks, filters and oscillators that run the same sequence unfused: read, Nco.apply,
Fir.apply; or Fir.apply, Nco.apply, write.  Everything bit for bit, plus one check of the physics
that a shared mistake of kernel and restatement could not pass."""
import numpy as np
import pytest

import sxfir
import sxnco
from test_gpu_fir import design, same_bits
from test_gpu_fir_bank import as_frames, out_buffer, same_state, synth_rx
from test_gpu_iir import latency_ns
from test_gpu_iir_halves import HAS_TIME, RATE, assert_same_bank, write_times

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

CHUNK = 1 << 22


def cf(rng, S, n):
    return rng.standard_normal((S, 2 * n), dtype=np.float32).view(np.complex64)


def ref_stream(S, freqs, phases):
    r = sxnco.Stream(S, freqs)
    r.phase = np.asarray(phases, np.uint32).copy()
    return r


def want_apply(ref, x):
    """ref.feed(x) in pieces of CHUNK frames (any split equals one call, test_nco_oracle.py)."""
    return np.concatenate([ref.feed(x[:, i:i + CHUNK]) for i in range(0, x.shape[1], CHUNK)], axis=1)


def same_nco(a, b, st):
    (p1, i1), (p2, i2) = a.state(st), b.state(st)
    return np.array_equal(p1, p2) and np.array_equal(i1, i2)


@pytest.mark.parametrize("S,n", [(1, 1), (3, 517), (64, 256), (4096, 1237), (65536, 256), (1, 1 << 27)])
def test_apply_matches_the_restatement(ctx, S, n):
    from sxxcvr_b200 import Nco
    rng = np.random.default_rng(S + n)
    freqs = rng.uniform(-0.5, 0.5, S)
    freqs[0] = 0.5
    phases = rng.integers(0, 2**32, S, dtype=np.uint64).astype(np.uint32)
    ref = ref_stream(S, freqs, phases)
    with Nco(ctx, S, freqs) as N:
        ph, inc = N.state()
        assert not ph.any() and np.array_equal(inc, ref.inc)
        N.set_state(phases, None)
        for it in range(2):
            x = cf(rng, S, n)
            d = torch.from_numpy(x.view(np.float32).reshape(-1)).cuda()
            N.apply(d.data_ptr(), n)
            ctx.stream_sync()
            got = d.cpu().numpy().view(np.complex64).reshape(S, n)
            del d
            assert same_bits(got, want_apply(ref, x)), it
            ph, inc = N.state()
            assert np.array_equal(ph, ref.phase) and np.array_equal(inc, ref.inc), it


def test_retune_mid_sequence_and_state_round_trip(ctx):
    from sxxcvr_b200 import Nco
    S, n = 300, 777
    rng = np.random.default_rng(11)
    f1, f2 = rng.uniform(-0.5, 0.5, S), rng.uniform(-0.5, 0.5, S)
    ref = sxnco.Stream(S, f1)
    with Nco(ctx, S, f1) as N:
        for it, f in enumerate((None, f2, 0.125, f1)):
            if f is not None:
                N.set_frequencies(f)
                ref.retune(f)
            x = cf(rng, S, n)
            d = torch.from_numpy(x.view(np.float32).reshape(-1)).cuda()
            N.apply(d.data_ptr(), n)
            ctx.stream_sync()
            assert same_bits(d.cpu().numpy().view(np.complex64).reshape(S, n), ref.feed(x)), it
        ph, inc = N.state()
        assert np.array_equal(ph, ref.phase) and np.array_equal(inc, ref.inc)
        p2 = rng.integers(0, 2**32, S, dtype=np.uint64).astype(np.uint32)
        i2 = rng.integers(0, 2**32, S, dtype=np.uint64).astype(np.uint32)
        N.set_state(p2, None)
        assert np.array_equal(N.state()[0], p2) and np.array_equal(N.state()[1], inc)
        N.set_state(None, i2)
        assert np.array_equal(N.state()[0], p2) and np.array_equal(N.state()[1], i2)
        N.set_state(None, None)
        only = np.empty(S, np.uint32)
        ctx.check(ctx.lib.sxgpu_nco_get_state(N.handle, None, only.ctypes.data, None), "get_state")
        assert np.array_equal(only, i2)
        ctx.check(ctx.lib.sxgpu_nco_get_state(N.handle, only.ctypes.data, None, None), "get_state")
        assert np.array_equal(only, p2)


@pytest.mark.parametrize("S,P", [(5, 34), (63, 256), (65536, 256)])
def test_read_ddc_matches_the_restatement(ctx, oracle, S, P):
    from sxxcvr_b200 import Bank, Fir, Nco
    h = design(64, 1, 4)
    freqs = np.random.default_rng(S).uniform(-0.5, 0.5, S)
    fir, nco = sxfir.Stream(h, 1, 4, S), sxnco.Stream(S, freqs)
    side = torch.cuda.Stream()
    st = side.cuda_stream
    with Bank(ctx, S, P, RATE, 1.0e-6, 43) as bank, Fir(ctx, S, h, 1, 4) as F, Nco(ctx, S, freqs) as N:
        out = out_buffer(S, -(-P // 4))
        for it in range(3):
            want_n = sxfir.output_frames(fir.fed, P, 1, 4)
            with torch.cuda.stream(side):
                n = bank.read_ddc(N, F, out.data_ptr(), st)
            side.synchronize()
            assert n == want_n, it
            assert same_bits(as_frames(out, S, n), sxnco.ddc(nco, fir, synth_rx(oracle, S, it * P, P, 43))), it
            assert np.array_equal(N.state(st)[0], nco.phase), it


@pytest.mark.parametrize("S,P,ntaps,up,down", [(2100, 256, 64, 1, 4), (32768 + 3, 64, 96, 3, 2), (37, 64, 4096, 1, 1),
                                               (5, 2, 64, 1, 8), (37, 256, 1, 1, 1)])
@pytest.mark.parametrize("capture", ["synthetic", "ingested"])
def test_read_ddc_equals_read_then_apply(ctx, S, P, ntaps, up, down, capture):
    from sxxcvr_b200 import Bank, Fir, Nco
    rng = np.random.default_rng(S + P + ntaps)
    h = design(ntaps, up, down) if ntaps > 1 else np.array([0.7])
    freqs = rng.uniform(-0.5, 0.5, S)
    side = torch.cuda.Stream()
    st = side.cuda_stream
    nmax = -(-P * up // down)
    with Bank(ctx, S, P, RATE, 1.0e-6, 5) as fused, Bank(ctx, S, P, RATE, 1.0e-6, 5) as split, \
            Fir(ctx, S, h, up, down) as F1, Fir(ctx, S, h, up, down) as F2, Nco(ctx, S, freqs) as N1, \
            Nco(ctx, S, freqs) as N2:
        start = rng.integers(0, 2**32, S, dtype=np.uint64).astype(np.uint32)
        N1.set_state(start, None, st)
        N2.set_state(start, None, st)
        out1, out2 = out_buffer(S, nmax), out_buffer(S, nmax)
        cf32 = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
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
                n1 = fused.read_ddc(N1, F1, out1.data_ptr(), st)
                split.read(cf32.data_ptr(), st)
                N2.apply(cf32.data_ptr(), P, st)
                n2 = F2.apply(cf32.data_ptr(), P, out2.data_ptr(), st)
            side.synchronize()
            assert n1 == n2, it
            counts.append(n1)
            assert same_bits(as_frames(out1, S, n1), as_frames(out2, S, n2)), it
            for a, b in zip(fused.positions(st), split.positions(st)):
                assert np.array_equal(a, b), it
            assert all(np.array_equal(a, b) for a, b in zip(fused.last_read(st), split.last_read(st))), it
            assert same_state(F1, F2, st) and same_nco(N1, N2, st), it
        if down == 8:
            assert counts == [1, 0, 0, 0]
        # the capture slots, as a plain read in ingested mode with nothing handed in converts them
        cf1 = torch.zeros_like(cf32)
        with torch.cuda.stream(side):
            fused.ingest(0, 0, None, st)
            split.ingest(0, 0, None, st)
            fused.read(cf1.data_ptr(), st)
            split.read(cf32.data_ptr(), st)
        side.synchronize()
        assert same_bits(cf1.cpu().numpy(), cf32.cpu().numpy())


WRITE_FILTERS = [(37, 256, 64, 4, 1), (32768 + 3, 256, 64, 4, 1), (37, 66, 96, 3, 2), (37, 255, 96, 3, 2),
                 (37, 64, 31, 1, 1)]


@pytest.mark.parametrize("S,P,ntaps,up,down", WRITE_FILTERS)
@pytest.mark.parametrize("case", ["mixed", "offset", "untimed", "late"])
def test_write_duc_equals_apply_then_write(ctx, S, P, ntaps, up, down, case):
    """write_duc(F, N) against F.apply into a scratch block, N.apply on it, then write, on twins.
    `mixed`: on-time, late, forwarded-over and straddling streams; `offset`: HAS_TIME with no
    timestamps, 769 frames after a plain read; `untimed`: flags 0 through an underrun; `late`:
    every write dropped."""
    from sxxcvr_b200 import Bank, Fir, Nco
    rng = np.random.default_rng(S + P + up + 1)
    h = design(ntaps, up, down)
    nin = P * down // up
    freqs = rng.uniform(-0.5, 0.5, S)
    lat = latency_ns(769)
    side = torch.cuda.Stream()
    st = side.cuda_stream
    with Bank(ctx, S, P, RATE, 1.0e-6, 9) as fused, Bank(ctx, S, P, RATE, 1.0e-6, 9) as split, \
            Fir(ctx, S, h, up, down) as F1, Fir(ctx, S, h, up, down) as F2, Nco(ctx, S, freqs) as N1, \
            Nco(ctx, S, freqs) as N2:
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
                    fused.advance(5 * P + 3, st)
                    split.advance(5 * P + 3, st)
                t_ptr = d_times.data_ptr() if d_times is not None else None
                fused.write_duc(F1, N1, d_in.data_ptr(), nin, flags, t_ptr, lat, st)
                assert F2.apply(d_in.data_ptr(), nin, tmp.data_ptr(), st) == P
                N2.apply(tmp.data_ptr(), P, st)
                split.write(tmp.data_ptr(), flags, t_ptr, lat, st)
            side.synchronize()
            assert same_bits(d_in.cpu().numpy(), x), it
            assert same_state(F1, F2, st) and same_nco(N1, N2, st), it
            assert_same_bank(fused, split, S, P, st, it)
        clock, _, txp = fused.positions(st)
        if case == "late":
            assert (txp == 0).all()
            ph, inc = N1.state(st)
            assert np.array_equal(ph, (3 * P * inc.astype(np.uint64) % 2**32).astype(np.uint32))  # advanced all the same


@pytest.mark.parametrize("ntaps,capture", [(64, "synthetic"), (1, "ingested")])
def test_launch_counts(ctx, ntaps, capture):
    """read_ddc: plan + data kernel + the tail kernel, which always runs (also with one tap and
    ingested capture, where read_fir has none); with nothing emitted (P = 2, ↓8, second call) the
    data kernel is left out.  write_duc: always 3.  apply: 2."""
    from sxxcvr_b200 import Bank, Fir, Nco
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
            Fir(ctx, S, h, 8, 1) as G, Nco(ctx, S, 0.1) as N:
        if capture == "ingested":
            bank.ingest(0, S, i2s.data_ptr())
            tiny.ingest(0, S, i2s.data_ptr())
        assert count(lambda: bank.read_ddc(N, F, out.data_ptr())) == (3, S * 256, 0)
        assert count(lambda: tiny.read_ddc(N, Ft, out.data_ptr())) == (3, S * 2, 0)  # one frame
        assert count(lambda: tiny.read_ddc(N, Ft, out.data_ptr())) == (2, S * 2, 0)  # none
        assert count(lambda: bank.write_duc(G, N, out.data_ptr(), 32, HAS_TIME, None, latency_ns(768))) == (3, 0, S * 256)
        assert count(lambda: N.apply(out.data_ptr(), 7)) == (2, 0, 0)


def test_graph_replay_equals_direct_calls(ctx):
    """A captured read_ddc(↓4), write_duc(↑4) and apply of 1237 frames, replayed three times, equal
    the direct calls on twins: the phases live on the device and advance in every replay."""
    from sxxcvr_b200 import Bank, Fir, Nco
    S, P, C, M = 16, 256, 64, 1237
    f_taps, g_taps = design(64, 1, 4), design(48, 4, 1)
    rng = np.random.default_rng(8)
    fr, ft = rng.uniform(-0.5, 0.5, S), rng.uniform(-0.5, 0.5, S)
    lat = latency_ns(768)
    chan1, chan2 = out_buffer(S, C), out_buffer(S, C)
    x = torch.from_numpy(cf(rng, S, M).view(np.float32).reshape(-1)).cuda()
    y1, y2 = x.clone(), x.clone()
    with Bank(ctx, S, P, RATE, 1.0e-6, 77) as a, Bank(ctx, S, P, RATE, 1.0e-6, 77) as b, \
            Fir(ctx, S, f_taps, 1, 4) as F1, Fir(ctx, S, g_taps, 4, 1) as G1, \
            Fir(ctx, S, f_taps, 1, 4) as F2, Fir(ctx, S, g_taps, 4, 1) as G2, \
            Nco(ctx, S, fr) as R1, Nco(ctx, S, ft) as T1, Nco(ctx, S, fr) as R2, Nco(ctx, S, ft) as T2, \
            Nco(ctx, S, ft) as A1, Nco(ctx, S, ft) as A2:
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        before = ctx.counter("launches")
        with torch.cuda.graph(g, stream=side):
            st = torch.cuda.current_stream().cuda_stream
            a.read_ddc(R1, F1, chan1.data_ptr(), st)
            a.write_duc(G1, T1, chan1.data_ptr(), C, HAS_TIME, None, lat, st)
            A1.apply(y1.data_ptr(), M, st)
        assert ctx.counter("launches") - before == 8
        for it in range(3):
            g.replay()
            b.read_ddc(R2, F2, chan2.data_ptr())
            b.write_duc(G2, T2, chan2.data_ptr(), C, HAS_TIME, None, lat)
            A2.apply(y2.data_ptr(), M)
            torch.cuda.synchronize()
            ctx.stream_sync()
            assert same_bits(chan1.cpu().numpy(), chan2.cpu().numpy()), it
            assert same_bits(y1.cpu().numpy(), y2.cpu().numpy()), it
            assert same_state(F1, F2, None) and same_state(G1, G2, None), it
            assert same_nco(R1, R2, None) and same_nco(T1, T2, None) and same_nco(A1, A2, None), it
            assert_same_bank(a, b, S, P, None, it)
        assert A1.state()[0].any()


def test_a_tone_is_brought_to_dc_and_the_others_are_rejected(ctx):
    """One tone at +f0 ingested into every stream.  Stream 0, tuned to -f0, comes out of the low-pass
    ↓4 at DC with the tone's amplitude times the filter's DC gain; the others, tuned so that the
    tone lands in the stopband, are attenuated by the stopband.  Kernel and restatement could share
    a sign or scaling mistake; this would not pass it."""
    from sxxcvr_b200 import Bank, Fir, Nco
    S, P, amp, f0 = 4, 256, 0.5, 0.1
    tune = np.array([-f0, 0.2, -0.4, 0.15])   # the tone lands at 0, 0.3, -0.3 and 0.25 cycles per sample
    h = design(64, 1, 4)                      # passband to 0.1 cycles per sample, ↓4
    gain = float(np.sum(h.astype(np.float32), dtype=np.float64))
    with Bank(ctx, S, P) as bank, Fir(ctx, S, h, 1, 4) as F, Nco(ctx, S, tune) as N:
        out = out_buffer(S, P // 4)
        for it in range(4):
            k = np.arange(it * P, (it + 1) * P)
            tone = amp * np.exp(2j * np.pi * f0 * k)
            words = np.empty((S, P, 2), np.int32)
            words[:, :, 0] = np.round(tone.real * 2**31).astype(np.int64)
            words[:, :, 1] = np.round(tone.imag * 2**31).astype(np.int64)
            i2s = torch.from_numpy(words.reshape(-1)).cuda()
            bank.ingest(0, S, i2s.data_ptr())
            assert bank.read_ddc(N, F, out.data_ptr()) == P // 4
            ctx.stream_sync()
        y = as_frames(out, S, P // 4).astype(np.complex128)   # the last call: past the filter's start
        assert np.abs(y[0] - amp * gain).max() < 1e-4 * amp, y[0][:4]
        for s in range(1, S):
            assert np.abs(y[s]).max() < amp * 10 ** (-40 / 20), (s, np.abs(y[s]).max())


def test_invalid_arguments_are_refused(ctx):
    """Every refusal: of create, apply and set_frequencies, and of the two bank calls, each leaving
    the launch counter, the positions, the filters' phases and the oscillator's state as they were."""
    from sxxcvr_b200 import Bank, Context, Fir, Nco
    from sxxcvr_b200.capi import ERR_INVALID, SxGpuError
    S, P = 5, 256
    buf = torch.zeros(S * P * 2 + 8, dtype=torch.float32, device="cuda")
    d = buf.data_ptr()
    c2 = Context(0)
    try:
        for bad in ([0.6] * S, [np.nan] * S, [-np.inf] * S, [0.5000001] * S):
            with pytest.raises(SxGpuError) as e:
                Nco(ctx, S, bad)
            assert e.value.code == ERR_INVALID
        with pytest.raises(SxGpuError):
            Nco(ctx, 0)
        with pytest.raises(SxGpuError):
            Nco(ctx, 2**31)
        with Bank(ctx, S, P) as bank, Fir(ctx, S, design(64, 1, 3), 1, 3) as F, Fir(ctx, S, design(48, 4, 1), 4, 1) as G, \
                Nco(ctx, S, 0.1) as N, Nco(ctx, S + 1) as other, Nco(c2, S) as foreign, \
                Fir(ctx, S + 1, design(64, 1, 3), 1, 3) as other_fir:
            G.set_state(None, 0)
            F.set_state(None, 1)
            N.set_state(np.arange(S, dtype=np.uint32) * 1000, None)
            launches, positions, nstate = ctx.counter("launches"), bank.positions(), N.state()

            def refused(fn):
                with pytest.raises(SxGpuError) as e:
                    fn()
                assert e.value.code == ERR_INVALID
                ctx.stream_sync()
                assert ctx.counter("launches") == launches and F.state()[1] == 1 and G.state()[1] == 0
                assert all(np.array_equal(x, y) for x, y in zip(bank.positions(), positions))
                assert all(np.array_equal(x, y) for x, y in zip(N.state(), nstate))

            for n in (None, other, foreign):
                refused(lambda: bank.read_ddc(n, F, d))
                refused(lambda: bank.write_duc(G, n, d, 64))
            for f in (None, other_fir):
                refused(lambda: bank.read_ddc(N, f, d))
                refused(lambda: bank.write_duc(f, N, d, 64))
            refused(lambda: bank.read_ddc(N, F, 0))
            refused(lambda: bank.read_ddc(N, F, d + 4))
            refused(lambda: bank.write_duc(G, N, 0, 64))
            refused(lambda: bank.write_duc(G, N, d + 4, 64))
            refused(lambda: bank.write_duc(G, N, d, 1 << 62))
            refused(lambda: bank.write_duc(G, N, d, 63))
            refused(lambda: bank.write_duc(G, N, d, 0))
            refused(lambda: N.apply(d, 0))
            refused(lambda: N.apply(0, 8))
            refused(lambda: N.apply(d + 4, 8))
            refused(lambda: N.apply(d, 1 << 62))          # 5 x 2^62 x 8 bytes overflows
            refused(lambda: N.apply(d, (1 << 60) // S))   # fits in bytes, but more than 2^31 - 1 CTAs
            for bad in (0.6, np.nan, -np.inf):
                refused(lambda: N.set_frequencies(bad))
            # and the same calls with good arguments run
            assert bank.read_ddc(N, F, d) == 85
            bank.write_duc(G, N, d, 64, HAS_TIME, None, latency_ns(768))
            N.apply(d, 8)
            ctx.stream_sync()
            assert ctx.counter("launches") - launches == 8
            inc = nstate[1].astype(np.uint64)
            assert np.array_equal(N.state()[0], ((nstate[0] + (2 * P + 8) * inc) % 2**32).astype(np.uint32))
        with Nco(c2, S):  # a context refuses to go while an oscillator is alive
            assert c2.lib.sxgpu_destroy(c2.handle) == ERR_INVALID
    finally:
        c2.close()
