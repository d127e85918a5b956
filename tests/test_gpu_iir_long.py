"""-m gpu: sxgpu_iir_apply_long (Iir.apply_long) against the numpy restatement in
tests/sxiir_long.py, bit for bit: the filtered block and the final state, with and without an
initial state, followed by the sequential apply on the next block, a block of one chunk against
Iir.apply, the launch count, a CUDA graph replay, and the refusals."""
import numpy as np
import pytest

import sxiir
import sxiir_long
from test_gpu_iir import design, random_state, same_bits

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
signal = pytest.importorskip("scipy.signal")

CHAINS = {}


def chain(nsections):
    if nsections not in CHAINS:
        CHAINS[nsections] = sxiir_long.power_chain(design(nsections))
    return CHAINS[nsections]


def block(rng, nstreams, nframes):
    x = rng.standard_normal((nstreams, 2 * nframes), dtype=np.float32).view(np.complex64)
    x *= np.float32(0.3)
    return x


def to_device(x):
    return torch.from_numpy(x.view(np.float32).reshape(-1).copy()).cuda()


def from_device(t, nstreams, nframes):
    return t.cpu().numpy().view(np.complex64).reshape(nstreams, nframes)


def launches(nstreams, nframes):
    size = sxiir_long.chunk_len(nstreams, nframes)
    chunks = -(-nframes // size)
    if chunks == 1:
        return 1
    groups = -(-chunks // sxiir_long.GROUP)
    return 4 + (groups - 1).bit_length()  # pass 1, reduce, scan levels, fix-up, pass 3


SHAPES = [(1, 1), (1, 128), (1, 129), (3, 5 * 128 + 17), (1, 1 << 24), (16, 1 << 20)]


@pytest.mark.parametrize("nsections", [1, 4, 8])
@pytest.mark.parametrize("nstreams,nframes", SHAPES)
def test_apply_long_matches_the_restatement(ctx, nstreams, nframes, nsections):
    from sxxcvr_b200 import Iir
    rng = np.random.default_rng(nstreams * 7 + nframes + nsections)
    sos = design(nsections)
    side = torch.cuda.Stream()
    st = side.cuda_stream
    big = nframes >= 1 << 20
    with Iir(ctx, nstreams, sos) as f:
        for with_state in ([True] if big else [False, True]):
            z = random_state(rng, nsections, nstreams) if with_state else None
            f.set_state(z, st)
            x = block(rng, nstreams, nframes)
            cf = to_device(x)
            before = ctx.counter("launches")
            with torch.cuda.stream(side):
                f.apply_long(cf.data_ptr(), nframes, st)
            side.synchronize()
            assert ctx.counter("launches") - before == launches(nstreams, nframes)
            want, zf = sxiir_long.apply_long(sos, x, z, chain=chain(nsections))
            assert same_bits(from_device(cf, nstreams, nframes), want), with_state
            assert same_bits(f.state(st), zf), with_state
            del cf
            if big:
                continue
            # and the sequential filter carries on from the state it left
            x2 = block(rng, nstreams, 300)
            cf2 = to_device(x2)
            with torch.cuda.stream(side):
                f.apply(cf2.data_ptr(), 300, st)
            side.synchronize()
            want2, zf2 = sxiir.sosfilt(sos, x2, zf)
            assert same_bits(from_device(cf2, nstreams, 300), want2) and same_bits(f.state(st), zf2)


def test_one_chunk_equals_apply(ctx):
    from sxxcvr_b200 import Iir
    rng = np.random.default_rng(3)
    S, P = 5, 100
    sos = design(4, 1)
    z = random_state(rng, 4, S)
    x = block(rng, S, P)
    a, b = to_device(x), to_device(x)
    with Iir(ctx, S, sos) as f, Iir(ctx, S, sos) as g:
        f.set_state(z)
        g.set_state(z)
        f.apply(a.data_ptr(), P)
        g.apply_long(b.data_ptr(), P)
        ctx.stream_sync()
        assert same_bits(a.cpu().numpy(), b.cpu().numpy()) and same_bits(f.state(), g.state())


def test_graph_replay_equals_a_direct_call(ctx):
    from sxxcvr_b200 import Iir
    rng = np.random.default_rng(4)
    S, N = 2, 1 << 18
    sos = design(4)
    z = random_state(rng, 4, S)
    x = block(rng, S, N)
    graphed, direct = to_device(x), to_device(x)
    with Iir(ctx, S, sos) as f:
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.graph(g, stream=side):
            f.apply_long(graphed.data_ptr(), N, torch.cuda.current_stream().cuda_stream)
        f.set_state(z)
        g.replay()
        torch.cuda.synchronize()
        got_state = f.state()
        f.set_state(z)
        f.apply_long(direct.data_ptr(), N)
        ctx.stream_sync()
        assert same_bits(graphed.cpu().numpy(), direct.cpu().numpy()) and same_bits(got_state, f.state())
        want, zf = sxiir_long.apply_long(sos, x, z, chain=chain(4))
        assert same_bits(from_device(graphed, S, N), want) and same_bits(got_state, zf)


def test_invalid_arguments_are_refused(ctx):
    from sxxcvr_b200 import Iir
    from sxxcvr_b200.capi import ERR_INVALID, SxGpuError

    def refused(fn):
        with pytest.raises(SxGpuError) as e:
            fn()
        assert e.value.code == ERR_INVALID

    cf = torch.zeros(4 * 1000 * 2 + 8, dtype=torch.float32, device="cuda")
    with Iir(ctx, 4, design(2)) as f:
        refused(lambda: f.apply_long(None, 1000))
        refused(lambda: f.apply_long(cf.data_ptr() + 4, 1000))
        refused(lambda: f.apply_long(cf.data_ptr(), 0))
        refused(lambda: f.apply_long(cf.data_ptr(), 1 << 62))  # 4 x 2^62 x 8 bytes overflows
        refused(lambda: f.apply_long(cf.data_ptr(), 1 << 50))  # 2^42 chunks: more CTAs than a grid holds
        before = ctx.counter("launches")
        f.apply_long(cf.data_ptr(), 1000)  # and the same call with good arguments runs
        ctx.stream_sync()
        assert ctx.counter("launches") - before == launches(4, 1000)
