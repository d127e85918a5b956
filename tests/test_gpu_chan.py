"""-m gpu: sxgpu_chan_apply (Chan.apply) against the numpy restatement in tests/sxchan.py, bit for
bit: outputs, history and phase, over shapes from one frame to 2^22 frames and the bank's
65 536 x 256, over sequences of calls of varying length; output counts, the state round trip and
resuming on a second channelizer, the launch count, a CUDA-graph replay, the output fed on to
Fir.apply as nstreams * M streams, the cross-check against Nco.apply + Fir.apply per channel, and
the refusals."""
import numpy as np
import pytest

import sxchan
import sxfir
from test_gpu_fir import frames, same_bits, to_device

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
signal = pytest.importorskip("scipy.signal")

FACTORS = [(16, 16, 256), (16, 8, 256), (64, 32, 1024), (1024, 1024, 16384), (2, 1, 5), (8, 2, 31)]
SMALL = [(1, 1), (3, 517), (64, 256)]
LARGE = [((65536, 256), (16, 16, 256)), ((65536, 256), (16, 8, 256)), ((1, 1 << 22), (64, 32, 1024)),
         ((1, 1 << 22), (2, 1, 5)), ((16, 1 << 16), (1024, 1024, 16384)), ((256, 4096), (8, 2, 31))]


def design(ntaps, m):
    return signal.firwin(ntaps, 1.0 / m)


def run(ctx, c, x, nout_expected, stream=None):
    """One Chan.apply of x (nstreams, nin) -> (nstreams, M, nout) on the host, checking the counts."""
    nstreams, nin = x.shape
    assert c.output_frames(nin) == nout_expected
    d_in = to_device(x)
    rows = nstreams * c.channels
    d_out = torch.empty(max(1, 2 * rows * nout_expected), dtype=torch.float32, device="cuda")
    before = ctx.counter("launches")
    nout = c.apply(d_in.data_ptr(), nin, d_out.data_ptr(), stream)
    ctx.stream_sync(stream)
    assert nout == nout_expected
    assert ctx.counter("launches") - before == (1 if nout else 0) + (1 if c.ntaps > 1 else 0)
    return d_out[:2 * rows * nout].cpu().numpy().view(np.complex64).reshape(nstreams, c.channels, nout)


def check_state(c, ref):
    hist, phase = c.state()
    assert phase == ref.phase
    assert same_bits(hist, ref.hist)


def check_calls(ctx, c, ref, rng, lengths, stream=None):
    for n in lengths:
        x = frames(rng, ref.nstreams, n)
        want_n = sxchan.output_frames(ref.fed, n, ref.down)
        assert same_bits(run(ctx, c, x, want_n, stream), ref.feed(x)), n
        check_state(c, ref)


@pytest.mark.parametrize("m,d,ntaps", FACTORS)
@pytest.mark.parametrize("nstreams,nin", SMALL)
def test_apply_matches_the_restatement(ctx, nstreams, nin, m, d, ntaps):
    from sxxcvr_b200 import Chan
    rng = np.random.default_rng(nstreams * 31 + nin + ntaps + m + d)
    h = design(ntaps, m)
    ref = sxchan.Stream(h, m, d, nstreams)
    with Chan(ctx, nstreams, h, m, d) as c:
        # the block, then a short call that starts mid-period and reads the history
        check_calls(ctx, c, ref, rng, (nin, 7))


@pytest.mark.parametrize("shape,factors", LARGE, ids=[f"{s[0]}x{s[1]}-{f}" for s, f in LARGE])
def test_large_shapes(ctx, shape, factors):
    from sxxcvr_b200 import Chan
    (nstreams, nin), (m, d, ntaps) = shape, factors
    rng = np.random.default_rng(nstreams + nin + m)
    h = design(ntaps, m)
    ref = sxchan.Stream(h, m, d, nstreams)
    with Chan(ctx, nstreams, h, m, d) as c:
        check_calls(ctx, c, ref, rng, (nin, nin))


@pytest.mark.parametrize("m,d,ntaps", FACTORS + [(4, 4, 1), (2, 2, 64), (1024, 512, 3000)])
def test_sequences_of_calls(ctx, m, d, ntaps):
    """Calls of 1 frame, of fewer frames than the history, and of lengths that are not multiples of
    D or M, on a side stream."""
    from sxxcvr_b200 import Chan
    rng = np.random.default_rng(ntaps + 1000 * m + d)
    h = design(ntaps, m) if ntaps > 1 else np.array([0.7])
    ref = sxchan.Stream(h, m, d, 3)
    side = torch.cuda.Stream()
    with Chan(ctx, 3, h, m, d) as c, torch.cuda.stream(side):
        check_calls(ctx, c, ref, rng, [1, 1, 2, 5, 63, 64, 65, 1, 300, 1000, 3, 2049, 17], side.cuda_stream)


def test_state_round_trip_and_resume_on_a_second_channelizer(ctx):
    from sxxcvr_b200 import Chan
    rng = np.random.default_rng(9)
    m, d, ntaps, S = 16, 8, 200, 5
    h = design(ntaps, m)
    ref = sxchan.Stream(h, m, d, S)
    with Chan(ctx, S, h, m, d) as c, Chan(ctx, S, h, m, d) as g:
        x = frames(rng, S, 333)
        run(ctx, c, x, sxchan.output_frames(0, 333, d))
        ref.feed(x)
        hist, phase = c.state()
        assert phase == 333 % 16 and same_bits(hist, ref.hist)
        g.set_state(hist, phase)
        hist2, phase2 = g.state()
        assert phase2 == phase and same_bits(hist2, hist)
        x2 = frames(rng, S, 101)
        want = ref.feed(x2)
        n = sxchan.output_frames(333, 101, d)
        assert same_bits(run(ctx, g, x2, n), want) and same_bits(run(ctx, c, x2, n), want)
        # NULL history = zeros, phase 0: a fresh channelizer
        c.set_state()
        fresh = sxchan.Stream(h, m, d, S)
        assert same_bits(run(ctx, c, x2, sxchan.output_frames(0, 101, d)), fresh.feed(x2))
        check_state(c, fresh)


def test_graph_replay_equals_direct_calls(ctx):
    """A call with nin a multiple of M keeps the phase, so its graph can be replayed."""
    from sxxcvr_b200 import Chan
    rng = np.random.default_rng(11)
    S, N, m, d = 16, 4096, 16, 8
    h = design(256, m)
    xs = [frames(rng, S, N) for _ in range(3)]
    ref = sxchan.Stream(h, m, d, S)
    d_in = to_device(xs[0])
    d_out = torch.empty(2 * S * m * (N // d), dtype=torch.float32, device="cuda")
    with Chan(ctx, S, h, m, d) as c:
        c.set_state(None, 3)
        ref.set_state(None, 3)
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.graph(g, stream=side):
            c.apply(d_in.data_ptr(), N, d_out.data_ptr(), torch.cuda.current_stream().cuda_stream)
        c.set_state(None, 3)  # capture ran nothing; start both from the same state
        for x in xs:
            d_in.copy_(to_device(x))
            g.replay()
            torch.cuda.synchronize()
            got = d_out.cpu().numpy().view(np.complex64).reshape(S, m, -1)
            assert same_bits(got, ref.feed(x))
        check_state(c, ref)


def test_output_feeds_a_fir_as_nstreams_times_m_streams(ctx):
    """The channels go on to a second decimation stage with no transpose: one Fir of S M streams."""
    from sxxcvr_b200 import Chan, Fir
    rng = np.random.default_rng(12)
    S, N, m, d = 8, 2048, 16, 8
    h, h2 = design(256, m), signal.firwin(31, 0.25)
    ref, ref2 = sxchan.Stream(h, m, d, S), sxfir.Stream(h2, 1, 4, S * m)
    with Chan(ctx, S, h, m, d) as c, Fir(ctx, S * m, h2, 1, 4) as f:
        for _ in range(2):
            x = frames(rng, S, N)
            nout = c.output_frames(N)
            d_mid = torch.empty(2 * S * m * nout, dtype=torch.float32, device="cuda")
            d_out = torch.empty(2 * S * m * nout // 4, dtype=torch.float32, device="cuda")
            d_in = to_device(x)
            assert c.apply(d_in.data_ptr(), N, d_mid.data_ptr()) == nout
            assert f.apply(d_mid.data_ptr(), nout, d_out.data_ptr()) == nout // 4
            ctx.stream_sync()
            want = ref2.feed(ref.feed(x).reshape(S * m, nout))
            assert same_bits(d_out.cpu().numpy().view(np.complex64).reshape(S * m, -1), want)


@pytest.mark.parametrize("m,d,ntaps", [(16, 16, 256), (8, 2, 31), (64, 32, 1024)])
def test_channels_match_the_oscillator_and_the_decimator(ctx, m, d, ntaps):
    """Channel k against Nco.apply at -k/M on a copy of the block, then Fir.apply(h, 1, D), over two calls."""
    from sxxcvr_b200 import Chan, Fir, Nco
    rng = np.random.default_rng(m + ntaps)
    S, N = 4, 4096
    h = design(ntaps, m)
    freqs = [(-k / m + 1.0) if -k / m < -0.5 else -k / m for k in range(m)]
    scale = np.abs(h.astype(np.float32)).sum()
    with Chan(ctx, S, h, m, d) as c, Nco(ctx, S * m, np.repeat(np.array(freqs)[None], S, 0).reshape(-1)) as nco, \
            Fir(ctx, S * m, h, 1, d) as f:
        for n in (N, N + 5):
            x = frames(rng, S, n)
            nout = c.output_frames(n)
            d_in = to_device(x)
            d_ch = torch.empty(2 * S * m * nout, dtype=torch.float32, device="cuda")
            c.apply(d_in.data_ptr(), n, d_ch.data_ptr())
            copies = to_device(np.repeat(x[:, None, :], m, axis=1).reshape(S * m, n))
            nco.apply(copies.data_ptr(), n)
            d_sp = torch.empty_like(d_ch)
            assert f.apply(copies.data_ptr(), n, d_sp.data_ptr()) == nout
            ctx.stream_sync()
            got = d_ch.cpu().numpy().view(np.complex64).astype(np.complex128)
            want = d_sp.cpu().numpy().view(np.complex64).astype(np.complex128)
            assert np.abs(got - want).max() < 1e-6 * scale * np.abs(x).max() * 2


def test_invalid_arguments_are_refused(ctx):
    import ctypes as C

    from sxxcvr_b200 import Chan, Context
    from sxxcvr_b200.capi import ERR_INVALID, SxGpuError

    def refused(fn):
        with pytest.raises(SxGpuError) as e:
            fn()
        assert e.value.code == ERR_INVALID

    h = design(64, 16)
    refused(lambda: Chan(ctx, 0, h, 16))
    refused(lambda: Chan(ctx, (1 << 27), h, 16))  # 2^31 rows: more than the other calls take
    refused(lambda: Chan(ctx, 1, h, 1))
    refused(lambda: Chan(ctx, 1, h, 12))
    refused(lambda: Chan(ctx, 1, h, 2048))
    refused(lambda: Chan(ctx, 1, h, 16, 0))
    refused(lambda: Chan(ctx, 1, h, 16, 3))
    refused(lambda: Chan(ctx, 1, h, 16, 32))
    refused(lambda: Chan(ctx, 1, [], 16))
    refused(lambda: Chan(ctx, 1, np.ones(513), 16))  # above 32 M
    refused(lambda: Chan(ctx, 1, np.ones(16385), 1024))  # above SXGPU_CHAN_MAX_TAPS
    refused(lambda: Chan(ctx, 1, np.array([1.0, np.nan]), 16))
    refused(lambda: Chan(ctx, 1, np.array([np.inf]), 16))
    handle = C.c_void_p()
    assert ctx.lib.sxgpu_chan_create(ctx.handle, 1, 16, 16, 4, None, C.byref(handle)) == ERR_INVALID  # NULL taps
    with Chan(ctx, (1 << 27) - 1, [1.0], 16) as big:  # the largest stream count is accepted, and allocates nothing
        assert big.output_frames(16) == 1

    a = torch.zeros(2 * 12000, dtype=torch.float32, device="cuda")
    b = torch.zeros(2 * 4000, dtype=torch.float32, device="cuda")
    with Chan(ctx, 4, h, 16, 8) as c:  # 4 streams x 16 channels x 125 outputs from 1000 frames
        pa, pb = a.data_ptr(), b.data_ptr()
        refused(lambda: c.apply(None, 1000, pb))
        refused(lambda: c.apply(pa, 1000, None))
        refused(lambda: c.apply(pa + 4, 1000, pb))
        refused(lambda: c.apply(pa, 1000, pb + 4))
        refused(lambda: c.apply(pa, 0, pb))
        refused(lambda: c.apply(pa, 1 << 62, pb))  # 4 x 2^62 x 8 bytes overflows
        refused(lambda: c.apply(pa, 1 << 58, pb))  # the output, 64 x 2^55 x 8 bytes, overflows
        refused(lambda: c.apply(pa, 1000, pa))  # in place
        refused(lambda: c.apply(pa, 1000, pa + 8 * 3999))  # the output starts in the input's last frame
        refused(lambda: c.apply(pa + 8 * 7999, 1000, pa))  # the input starts in the output's last frame
        refused(lambda: c.apply(pa + (1 << 62), 1 << 52, pa))  # 2^44 CTAs: more than a grid holds
        refused(lambda: c.set_state(None, 16))
        # nothing was launched and the phase did not move; a good call runs
        assert c.state()[1] == 0
        before = ctx.counter("launches")
        assert c.apply(pa, 1000, pa + 8 * 4000) == 125  # adjacent, not overlapping
        ctx.stream_sync()
        assert ctx.counter("launches") - before == 2
        assert c.state()[1] == 1000 % 16

    # the context refuses to go while a channelizer lives
    other = Context(0)
    c = Chan(other, 2, h, 16)
    assert other.lib.sxgpu_destroy(other.handle) == ERR_INVALID
    c.close()
    other.close()
