"""-m gpu: sxgpu_chan_synth_apply (ChanSynth.apply) against the numpy restatement in
tests/sxchansynth.py, bit for bit: outputs, history and phase, over shapes from one frame to the
bank's 65 536 streams and 2^22 frames per channel, over sequences of calls of varying length; the
state round trip and resuming on a second synthesizer, the launch count, a CUDA-graph replay, the
cross-check against Fir.apply + Nco.apply + a sum over the channels, Chan.apply followed by
ChanSynth.apply reconstructing the signal on the device, and the refusals."""
import numpy as np
import pytest

import sxchansynth
from test_gpu_fir import frames, same_bits, to_device

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
signal = pytest.importorskip("scipy.signal")

# (M, D, ntaps); (64, 1, 2048) has hp = 2048 > 1024
FACTORS = [(16, 16, 256), (16, 8, 256), (64, 32, 1024), (1024, 1024, 16384), (2, 1, 5), (8, 2, 31), (64, 1, 2048)]
SMALL = [(1, 1), (3, 517), (64, 48)]
LARGE = [((65536, 16), (16, 16, 256)), ((65536, 32), (16, 8, 256)), ((1, 1 << 22), (64, 32, 1024)),
         ((16, 1024), (1024, 1024, 16384)), ((1, 1 << 20), (2, 1, 5))]


def design(ntaps, m):
    return signal.firwin(ntaps, 1.0 / m) if ntaps > 1 else np.array([0.7])


def channel_frames(rng, nstreams, m, n):
    return frames(rng, nstreams * m, n).reshape(nstreams, m, n)


def run(ctx, s, y, stream=None):
    """One ChanSynth.apply of y (nstreams, M, nin) -> (nstreams, nin D) on the host, checking the launches."""
    nstreams, m, nin = y.shape
    d_in = to_device(y)
    d_out = torch.empty(2 * nstreams * nin * s.up, dtype=torch.float32, device="cuda")
    before = ctx.counter("launches")
    s.apply(d_in.data_ptr(), nin, d_out.data_ptr(), stream)
    ctx.stream_sync(stream)
    assert ctx.counter("launches") - before == 1 + (1 if s.hp > 1 else 0)
    return d_out.cpu().numpy().view(np.complex64).reshape(nstreams, nin * s.up)


def check_state(s, ref):
    hist, phase = s.state()
    assert phase == ref.phase
    assert same_bits(hist, ref.hist)


def check_calls(ctx, s, ref, rng, lengths, stream=None):
    for n in lengths:
        y = channel_frames(rng, ref.nstreams, ref.m, n)
        assert same_bits(run(ctx, s, y, stream), ref.feed(y)), n
        check_state(s, ref)


@pytest.mark.parametrize("m,d,ntaps", FACTORS)
@pytest.mark.parametrize("nstreams,nin", SMALL)
def test_apply_matches_the_restatement(ctx, nstreams, nin, m, d, ntaps):
    from sxxcvr_b200 import ChanSynth
    rng = np.random.default_rng(nstreams * 31 + nin + ntaps + m + d)
    h = design(ntaps, m)
    ref = sxchansynth.Stream(h, m, d, nstreams)
    with ChanSynth(ctx, nstreams, h, m, d) as s:
        # the block, then a short call that starts at another phase and reads the history
        check_calls(ctx, s, ref, rng, (nin, 7))


@pytest.mark.parametrize("shape,factors", LARGE, ids=[f"{s[0]}x{s[1]}-{f}" for s, f in LARGE])
def test_large_shapes(ctx, shape, factors):
    from sxxcvr_b200 import ChanSynth
    (nstreams, nin), (m, d, ntaps) = shape, factors
    rng = np.random.default_rng(nstreams + nin + m)
    h = design(ntaps, m)
    ref = sxchansynth.Stream(h, m, d, nstreams)
    with ChanSynth(ctx, nstreams, h, m, d) as s:
        # the block, then a short call that reads the history the block left
        check_calls(ctx, s, ref, rng, (nin, 7))


@pytest.mark.parametrize("m,d,ntaps", FACTORS + [(4, 4, 1), (2, 2, 64), (1024, 512, 3000)])
def test_sequences_of_calls(ctx, m, d, ntaps):
    """Calls of 1 frame, of fewer frames than the history, and of lengths that are not multiples of
    M / D, on a side stream."""
    from sxxcvr_b200 import ChanSynth
    rng = np.random.default_rng(ntaps + 1000 * m + d)
    h = design(ntaps, m)
    S = 3 if m < 1024 else 1
    ref = sxchansynth.Stream(h, m, d, S)
    side = torch.cuda.Stream()
    lengths = [1, 2, 5, 63, 65, 300, 1, 17] if m < 1024 else [1, 2, 5, 63, 65, 3]
    with ChanSynth(ctx, S, h, m, d) as s, torch.cuda.stream(side):
        check_calls(ctx, s, ref, rng, lengths, side.cuda_stream)


def test_state_round_trip_and_resume_on_a_second_synthesizer(ctx):
    from sxxcvr_b200 import ChanSynth
    rng = np.random.default_rng(9)
    m, d, ntaps, S = 16, 4, 200, 5
    h = design(ntaps, m)
    ref = sxchansynth.Stream(h, m, d, S)
    with ChanSynth(ctx, S, h, m, d) as s, ChanSynth(ctx, S, h, m, d) as g:
        y = channel_frames(rng, S, m, 103)
        run(ctx, s, y)
        ref.feed(y)
        hist, phase = s.state()
        assert phase == 103 % 4 and same_bits(hist, ref.hist)
        g.set_state(hist, phase)
        hist2, phase2 = g.state()
        assert phase2 == phase and same_bits(hist2, hist)
        y2 = channel_frames(rng, S, m, 41)
        want = ref.feed(y2)
        assert same_bits(run(ctx, g, y2), want) and same_bits(run(ctx, s, y2), want)
        # NULL history = zeros, phase 0: a fresh synthesizer
        s.set_state()
        fresh = sxchansynth.Stream(h, m, d, S)
        assert same_bits(run(ctx, s, y2), fresh.feed(y2))
        check_state(s, fresh)


def test_graph_replay_equals_direct_calls(ctx):
    """A call with nin a multiple of M / D keeps the phase, so its graph can be replayed."""
    from sxxcvr_b200 import ChanSynth
    rng = np.random.default_rng(11)
    S, N, m, d = 16, 256, 16, 4
    h = design(256, m)
    ys = [channel_frames(rng, S, m, N) for _ in range(3)]
    ref = sxchansynth.Stream(h, m, d, S)
    d_in = to_device(ys[0])
    d_out = torch.empty(2 * S * N * d, dtype=torch.float32, device="cuda")
    with ChanSynth(ctx, S, h, m, d) as s:
        s.set_state(None, 3)
        ref.set_state(None, 3)
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.graph(g, stream=side):
            s.apply(d_in.data_ptr(), N, d_out.data_ptr(), torch.cuda.current_stream().cuda_stream)
        s.set_state(None, 3)  # capture ran nothing; start both from the same state
        for y in ys:
            d_in.copy_(to_device(y))
            g.replay()
            torch.cuda.synchronize()
            got = d_out.cpu().numpy().view(np.complex64).reshape(S, -1)
            assert same_bits(got, ref.feed(y))
        check_state(s, ref)


@pytest.mark.parametrize("m,d,ntaps", [(16, 16, 256), (16, 8, 256), (8, 2, 31), (64, 32, 1024)])
def test_matches_the_interpolator_the_oscillator_and_a_sum(ctx, m, d, ntaps):
    """One Fir.apply(h, D, 1) over S M rows, one Nco.apply at +k/M per row, and a torch sum over the
    channels, over two calls."""
    from sxxcvr_b200 import ChanSynth, Fir, Nco
    rng = np.random.default_rng(m + ntaps)
    S, N = 4, 512
    h = design(ntaps, m)
    freqs = [k / m if k < m // 2 else (k - m) / m for k in range(m)]
    h32 = np.abs(h.astype(np.float32).astype(np.float64))
    scale = m * max(h32[t::d].sum() for t in range(d))
    with ChanSynth(ctx, S, h, m, d) as s, Nco(ctx, S * m, np.tile(freqs, S)) as nco, Fir(ctx, S * m, h, d, 1) as f:
        for n in (N, N + 5):
            y = channel_frames(rng, S, m, n)
            d_in = to_device(y)
            d_x = torch.empty(2 * S * n * d, dtype=torch.float32, device="cuda")
            s.apply(d_in.data_ptr(), n, d_x.data_ptr())
            d_up = torch.empty(2 * S * m * n * d, dtype=torch.float32, device="cuda")
            assert f.apply(d_in.data_ptr(), n, d_up.data_ptr()) == n * d
            nco.apply(d_up.data_ptr(), n * d)
            ctx.stream_sync()
            want = torch.view_as_complex(d_up.view(S, m, n * d, 2)).to(torch.complex128).sum(dim=1)
            got = d_x.cpu().numpy().view(np.complex64).reshape(S, -1).astype(np.complex128)
            assert np.abs(got - want.cpu().numpy()).max() < 1e-6 * scale * np.abs(y).max() * 2


def test_analysis_then_synthesis_on_the_device_reconstructs_the_signal(ctx):
    """Chan.apply -> ChanSynth.apply over several calls, the phases carried: x delayed by the two
    linear-phase delays, scaled by about 1 / D, at least 50 dB above the error."""
    from sxxcvr_b200 import Chan, ChanSynth
    rng = np.random.default_rng(5)
    m, d, na, ns, S = 16, 8, 257, 129, 8
    delay = (na - 1) // 2 + (ns - 1) // 2
    x = frames(rng, S, 12000)
    out = []
    with Chan(ctx, S, signal.firwin(na, 1.0 / m), m, d) as c, ChanSynth(ctx, S, signal.firwin(ns, 2.0 / m), m, d) as s:
        for a, b in ((0, 3000), (3000, 3001), (3001, 7777), (7777, 12000)):
            n = b - a
            nout = c.output_frames(n)
            d_in = to_device(x[:, a:b])
            d_ch = torch.empty(2 * S * m * max(nout, 1), dtype=torch.float32, device="cuda")
            assert c.apply(d_in.data_ptr(), n, d_ch.data_ptr()) == nout
            if nout:
                d_x = torch.empty(2 * S * nout * d, dtype=torch.float32, device="cuda")
                s.apply(d_ch.data_ptr(), nout, d_x.data_ptr())
                out.append(d_x)
            ctx.stream_sync()  # before d_in and d_ch go back to torch's allocator
    xr = np.concatenate([o.cpu().numpy().view(np.complex64).reshape(S, -1) for o in out], axis=1).astype(np.complex128)
    assert xr.shape == (S, 12000)  # every D-th input frame starts an output of the channelizer
    start = na + ns
    ref = x[:, start:12000 - delay].astype(np.complex128)
    got = xr[:, delay + start:]
    g = np.vdot(ref, got) / np.vdot(ref, ref)
    assert abs(g * d - 1) < 5e-3, g
    snr = 10 * np.log10(np.mean(np.abs(g * ref) ** 2) / np.mean(np.abs(got - g * ref) ** 2))
    assert snr > 50, snr


def test_invalid_arguments_are_refused(ctx):
    import ctypes as C

    from sxxcvr_b200 import ChanSynth, Context
    from sxxcvr_b200.capi import ERR_INVALID, SxGpuError

    def refused(fn):
        with pytest.raises(SxGpuError) as e:
            fn()
        assert e.value.code == ERR_INVALID

    h = design(64, 16)
    refused(lambda: ChanSynth(ctx, 0, h, 16))
    refused(lambda: ChanSynth(ctx, (1 << 27), h, 16))  # 2^31 rows
    refused(lambda: ChanSynth(ctx, 1, h, 1))
    refused(lambda: ChanSynth(ctx, 1, h, 12))
    refused(lambda: ChanSynth(ctx, 1, h, 2048))
    refused(lambda: ChanSynth(ctx, 1, h, 16, 0))
    refused(lambda: ChanSynth(ctx, 1, h, 16, 3))
    refused(lambda: ChanSynth(ctx, 1, h, 16, 32))
    refused(lambda: ChanSynth(ctx, 1, [], 16))
    refused(lambda: ChanSynth(ctx, 1, np.ones(513), 16))  # above 32 M
    refused(lambda: ChanSynth(ctx, 1, np.ones(16385), 1024))  # above SXGPU_CHAN_MAX_TAPS
    refused(lambda: ChanSynth(ctx, 1, np.array([1.0, np.nan]), 16))
    refused(lambda: ChanSynth(ctx, 1, np.array([np.inf]), 16))
    handle = C.c_void_p()
    assert ctx.lib.sxgpu_chan_synth_create(ctx.handle, 1, 16, 16, 4, None, C.byref(handle)) == ERR_INVALID  # NULL taps
    with ChanSynth(ctx, (1 << 27) - 1, [1.0], 16):  # the largest stream count is accepted, and allocates no history
        pass

    a = torch.zeros(2 * 10000, dtype=torch.float32, device="cuda")
    b = torch.zeros(2 * 4000, dtype=torch.float32, device="cuda")
    with ChanSynth(ctx, 4, h, 16, 8) as s:  # 4 streams x 16 channels x 100 frames -> 4 x 800 frames
        pa, pb = a.data_ptr(), b.data_ptr()
        refused(lambda: s.apply(None, 100, pb))
        refused(lambda: s.apply(pa, 100, None))
        refused(lambda: s.apply(pa + 4, 100, pb))
        refused(lambda: s.apply(pa, 100, pb + 4))
        refused(lambda: s.apply(pa, 0, pb))
        refused(lambda: s.apply(pa, 1 << 62, pb))  # the input, 64 x 2^62 x 8 bytes, overflows
        refused(lambda: s.apply(pa, 100, pa))  # in place
        refused(lambda: s.apply(pa, 100, pa + 8 * 6399))  # the output starts in the input's last frame
        refused(lambda: s.apply(pa + 8 * 3199, 100, pa))  # the input starts in the output's last frame
        refused(lambda: s.apply(pa + (1 << 62), 1 << 52, pa))  # 2^44 CTAs: more than a grid holds
        refused(lambda: s.set_state(None, 2))
        # nothing was launched and the phase did not move; a good call runs
        assert s.state()[1] == 0
        before = ctx.counter("launches")
        s.apply(pa, 101, pa + 8 * 6464)  # adjacent, not overlapping
        ctx.stream_sync()
        assert ctx.counter("launches") - before == 2
        assert s.state()[1] == 101 % 2

    # the context refuses to go while a synthesizer lives
    other = Context(0)
    s = ChanSynth(other, 2, h, 16)
    assert other.lib.sxgpu_destroy(other.handle) == ERR_INVALID
    s.close()
    other.close()
