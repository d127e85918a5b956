"""-m gpu: sxgpu_fir_apply (Fir.apply) against the numpy restatement in tests/sxfir.py, bit for
bit: outputs, history and phase, over shapes from one frame to 2^22 frames and the bank's
65 536 x 256, over sequences of calls of varying length; output counts, the state round trip and
resuming on a second filter, the launch count, a CUDA-graph replay, the bank's read followed by
decimation, and the refusals."""
import numpy as np
import pytest

import sxfir

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
signal = pytest.importorskip("scipy.signal")

FACTORS = [(64, 1, 4), (96, 3, 2), (127, 1, 1), (255, 1, 8), (40, 5, 3)]
SHAPES = [(1, 1), (3, 517), (64, 256), (4096, 256), (1, 1 << 22), (4, 1 << 20)]


def design(ntaps, up, down):
    return signal.firwin(ntaps, 0.8 / max(up, down))


def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def frames(rng, nstreams, n):
    x = rng.standard_normal((nstreams, 2 * n), dtype=np.float32).view(np.complex64)
    if n >= 64:
        x[:, 10:20] = np.complex64(complex(-0.0, 0.0))
        x[:, 30:34] = np.float32(1e-42)  # subnormal
    return x


def to_device(x):
    return torch.from_numpy(np.ascontiguousarray(x).view(np.float32).reshape(-1).copy()).cuda()


def run(ctx, f, x, nout_expected, stream=None):
    """One Fir.apply of x (nstreams, nin) -> (nstreams, nout) on the host, checking the counts."""
    nstreams, nin = x.shape
    assert f.output_frames(nin) == nout_expected
    d_in = to_device(x)
    d_out = torch.empty(max(1, 2 * nstreams * nout_expected), dtype=torch.float32, device="cuda")
    before = ctx.counter("launches")
    nout = f.apply(d_in.data_ptr(), nin, d_out.data_ptr(), stream)
    ctx.stream_sync(stream)
    assert nout == nout_expected
    assert ctx.counter("launches") - before == (1 if nout else 0) + (1 if f.hp > 1 else 0)
    return d_out[:2 * nstreams * nout].cpu().numpy().view(np.complex64).reshape(nstreams, nout)


def check_state(f, ref):
    hist, phase = f.state()
    assert phase == ref.phase
    assert same_bits(hist, ref.hist)


@pytest.mark.parametrize("ntaps,up,down", FACTORS)
@pytest.mark.parametrize("nstreams,nin", SHAPES)
def test_apply_matches_the_restatement(ctx, nstreams, nin, ntaps, up, down):
    from sxxcvr_b200 import Fir
    rng = np.random.default_rng(nstreams * 31 + nin + ntaps + up + down)
    h = design(ntaps, up, down)
    ref = sxfir.Stream(h, up, down, nstreams)
    with Fir(ctx, nstreams, h, up, down) as f:
        # the block, then a short call that starts mid-period and reads the history
        for n in (nin, 7):
            x = frames(rng, nstreams, n)
            want_n = sxfir.output_frames(ref.fed, n, up, down)
            want = ref.feed(x)
            assert same_bits(run(ctx, f, x, want_n), want), n
            check_state(f, ref)


def test_bank_shape(ctx):
    """The bank's shape, 65 536 streams x 256 frames, decimated by 4 with 64 taps, twice."""
    from sxxcvr_b200 import Fir
    rng = np.random.default_rng(65536)
    h = design(64, 1, 4)
    ref = sxfir.Stream(h, 1, 4, 65536)
    with Fir(ctx, 65536, h, 1, 4) as f:
        for _ in range(2):
            x = frames(rng, 65536, 256)
            assert same_bits(run(ctx, f, x, 64), ref.feed(x))
        check_state(f, ref)


@pytest.mark.parametrize("ntaps,up,down", FACTORS + [(1, 1, 1), (2, 5, 1), (7, 7, 7), (300, 1, 256), (513, 256, 255)])
def test_sequences_of_calls(ctx, ntaps, up, down):
    """Calls of 1 frame, of fewer frames than the history, and long ones, on a side stream."""
    from sxxcvr_b200 import Fir
    rng = np.random.default_rng(ntaps + 1000 * up + down)
    h = design(ntaps, up, down) if ntaps > 1 else np.array([0.7])
    ref = sxfir.Stream(h, up, down, 3)
    side = torch.cuda.Stream()
    with Fir(ctx, 3, h, up, down) as f:
        for n in [1, 1, 2, 5, 63, 64, 65, 1, 300, 1000, 3, 2049, 17]:
            x = frames(rng, 3, n)
            want_n = sxfir.output_frames(ref.fed, n, up, down)
            with torch.cuda.stream(side):
                got = run(ctx, f, x, want_n, side.cuda_stream)
            assert same_bits(got, ref.feed(x)), n
            check_state(f, ref)


def test_state_round_trip_and_resume_on_a_second_filter(ctx):
    from sxxcvr_b200 import Fir
    rng = np.random.default_rng(9)
    up, down, ntaps, S = 3, 2, 96, 5
    h = design(ntaps, up, down)
    ref = sxfir.Stream(h, up, down, S)
    with Fir(ctx, S, h, up, down) as f, Fir(ctx, S, h, up, down) as g:
        x = frames(rng, S, 333)
        run(ctx, f, x, sxfir.output_frames(0, 333, up, down))
        ref.feed(x)
        hist, phase = f.state()
        assert phase == 1 and same_bits(hist, ref.hist)
        g.set_state(hist, phase)
        hist2, phase2 = g.state()
        assert phase2 == phase and same_bits(hist2, hist)
        x2 = frames(rng, S, 101)
        want = ref.feed(x2)
        n = sxfir.output_frames(333, 101, up, down)
        assert same_bits(run(ctx, g, x2, n), want) and same_bits(run(ctx, f, x2, n), want)
        # NULL history = zeros, phase 0: a fresh filter
        f.set_state()
        fresh = sxfir.Stream(h, up, down, S)
        assert same_bits(run(ctx, f, x2, sxfir.output_frames(0, 101, up, down)), fresh.feed(x2))
        hist3, phase3 = f.state()
        assert phase3 == fresh.phase and same_bits(hist3, fresh.hist)


def test_graph_replay_equals_direct_calls(ctx):
    """A call with nin a multiple of down keeps the phase, so its graph can be replayed."""
    from sxxcvr_b200 import Fir
    rng = np.random.default_rng(11)
    S, N, up, down = 16, 4096, 1, 4
    h = design(64, up, down)
    xs = [frames(rng, S, N) for _ in range(3)]
    ref = sxfir.Stream(h, up, down, S)
    d_in = to_device(xs[0])
    d_out = torch.empty(2 * S * N // 4, dtype=torch.float32, device="cuda")
    with Fir(ctx, S, h, up, down) as f:
        f.set_state(None, 2)
        ref.set_state(None, 2)
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.graph(g, stream=side):
            f.apply(d_in.data_ptr(), N, d_out.data_ptr(), torch.cuda.current_stream().cuda_stream)
        f.set_state(None, 2)  # capture ran nothing; start both from the same state
        for x in xs:
            d_in.copy_(to_device(x))
            g.replay()
            torch.cuda.synchronize()
            got = d_out.cpu().numpy().view(np.complex64).reshape(S, -1)
            assert same_bits(got, ref.feed(x))
        hist, phase = f.state()
        assert phase == 2 and same_bits(hist, ref.hist)


def test_bank_read_then_decimation(ctx):
    from sxxcvr_b200 import Bank, Fir
    S, P = 256, 256
    h = design(64, 1, 4)
    ref = sxfir.Stream(h, 1, 4, S)
    cf = torch.empty(2 * S * P, dtype=torch.float32, device="cuda")
    out = torch.empty(2 * S * P // 4, dtype=torch.float32, device="cuda")
    with Bank(ctx, S, P) as bank, Fir(ctx, S, h, 1, 4) as f:
        for _ in range(3):
            bank.read(cf.data_ptr())
            assert f.apply(cf.data_ptr(), P, out.data_ptr()) == P // 4
            ctx.stream_sync()
            block = cf.cpu().numpy().view(np.complex64).reshape(S, P)
            assert same_bits(out.cpu().numpy().view(np.complex64).reshape(S, -1), ref.feed(block))


def test_invalid_arguments_are_refused(ctx):
    import ctypes as C

    from sxxcvr_b200 import Context, Fir
    from sxxcvr_b200.capi import ERR_INVALID, SxGpuError

    def refused(fn):
        with pytest.raises(SxGpuError) as e:
            fn()
        assert e.value.code == ERR_INVALID

    h = design(64, 1, 4)
    refused(lambda: Fir(ctx, 0, h))
    refused(lambda: Fir(ctx, 1 << 31, h))  # one history CTA per stream: the grid holds 2^31 - 1
    refused(lambda: Fir(ctx, 1, []))
    refused(lambda: Fir(ctx, 1, np.ones(4097)))
    refused(lambda: Fir(ctx, 1, h, 0, 1))
    refused(lambda: Fir(ctx, 1, h, 1, 0))
    refused(lambda: Fir(ctx, 1, h, 257, 1))
    refused(lambda: Fir(ctx, 1, h, 1, 257))
    refused(lambda: Fir(ctx, 1, np.array([1.0, np.nan])))
    refused(lambda: Fir(ctx, 1, np.array([np.inf])))
    handle = C.c_void_p()
    assert ctx.lib.sxgpu_fir_create(ctx.handle, 1, 4, None, 1, 1, C.byref(handle)) == ERR_INVALID  # NULL taps

    a = torch.zeros(2 * 5000, dtype=torch.float32, device="cuda")
    b = torch.zeros(2 * 4000, dtype=torch.float32, device="cuda")
    with Fir(ctx, 4, h, 1, 4) as f:
        pa, pb = a.data_ptr(), b.data_ptr()
        refused(lambda: f.apply(None, 1000, pb))
        refused(lambda: f.apply(pa, 1000, None))
        refused(lambda: f.apply(pa + 4, 1000, pb))
        refused(lambda: f.apply(pa, 1000, pb + 4))
        refused(lambda: f.apply(pa, 0, pb))
        refused(lambda: f.apply(pa, 1 << 62, pb))  # 4 x 2^62 x 8 bytes overflows
        refused(lambda: f.apply(pa, 1000, pa))  # in place
        refused(lambda: f.apply(pa, 1000, pa + 8 * 3999))  # the output starts in the input's last frame
        refused(lambda: f.apply(pa + 8 * 999, 1000, pa))  # the input starts in the output's last frame
        refused(lambda: f.apply(pa + (1 << 62), 1 << 56, pa))  # 2^49 CTAs: more than a grid holds
        refused(lambda: f.set_state(None, 4))
        # nothing was launched and the phase did not move; a good call runs
        assert f.state()[1] == 0
        before = ctx.counter("launches")
        assert f.apply(pa, 1000, pa + 8 * 4000) == 250  # adjacent, not overlapping
        ctx.stream_sync()
        assert ctx.counter("launches") - before == 2

    # the context refuses to go while a filter lives
    other = Context(0)
    f = Fir(other, 2, h)
    assert other.lib.sxgpu_destroy(other.handle) == ERR_INVALID
    f.close()
    other.close()
