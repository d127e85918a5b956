"""-m gpu: the bank's stateful IIR filters (sxgpu_iir_*, sxgpu_bank_repeat_filtered, the filtered
hook path of include/sx_hook.cuh) against the numpy restatement in tests/sxiir.py, which
tests/test_iir_oracle.py holds to scipy.signal.sosfilt bit for bit.  Everything is compared bit for
bit except the hook example against scipy plus the script's literal numpy clipper, which carries
the clipper's stated tolerance (tests/test_gpu_hook.py) through the post filter."""
import ctypes as C

import numpy as np
import pytest

import sxiir
import sxtest
from test_gpu_hook import POST, PRE, clip_gain_exact, clip_gain_literal

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
signal = pytest.importorskip("scipy.signal")

HAS_TIME = 1 << 2
RATE = 75000.0


def latency_ns(frames):
    return int(round(frames * 1e9 / RATE))


def design(nsections, kind=0):
    """A stable design of exactly `nsections` sections."""
    if kind == 0:
        return signal.butter(2 * nsections, 0.25, output="sos")
    return signal.cheby1(2 * nsections, 1.0, 0.3, output="sos")


def random_state(rng, nsections, nstreams):
    z = rng.standard_normal((nsections, nstreams, 2)) + 1j * rng.standard_normal((nsections, nstreams, 2))
    return (0.05 * z).astype(np.complex64)


def as_blocks(t, S, P):
    return t.cpu().numpy().view(np.complex64).reshape(S, P)


def same_bits(a, b):
    return np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))


@pytest.fixture(scope="module")
def hooklib():
    from sxxcvr_b200 import _build
    lib = C.CDLL(str(_build.build_hook_example()))
    P = C.c_void_p
    lib.sx_example_repeat_filtered_clip_gain.argtypes = [P, P, P, P, C.c_longlong, C.c_float, C.c_float, P]
    lib.sx_example_repeat_filtered_clip_gain.restype = C.c_int
    return lib


# Every section count, stream count and period at least once; each case at most 2^22 frames.
@pytest.mark.parametrize("nsections,S,P", [(1, 1, 4096), (2, 5, 3), (4, 2100, 256), (8, 65536, 1), (8, 5, 64),
                                           (2, 65536, 64)])
def test_apply_matches_the_restatement(ctx, nsections, S, P):
    from sxxcvr_b200 import Iir
    rng = np.random.default_rng(nsections * 1000 + P)
    sos = design(nsections)
    side = torch.cuda.Stream()
    st = side.cuda_stream
    with Iir(ctx, S, sos) as f:
        z = random_state(rng, nsections, S)
        f.set_state(z, st)
        for it in range(3):
            x = (rng.standard_normal((S, P)) + 1j * rng.standard_normal((S, P))).astype(np.complex64)
            if it == 2:
                x[:, P // 2:] = 0
            cf = torch.from_numpy(x.view(np.float32).reshape(-1).copy()).cuda()
            with torch.cuda.stream(side):
                f.apply(cf.data_ptr(), P, st)
            side.synchronize()
            want, z = sxiir.sosfilt(sos, x, z)
            assert same_bits(as_blocks(cf, S, P), want), it
        assert same_bits(f.state(st), z)


def run_restatement(filters, x, states):
    for i, (sos, _) in enumerate(filters):
        x, states[i] = sxiir.sosfilt(sos, x, states[i])
    return x


@pytest.mark.parametrize("S,P", [(5, 256), (2100, 256), (32768 + 3, 64), (65536, 256)])
@pytest.mark.parametrize("stages", ["none", "pre", "post", "both"])
def test_repeat_filtered_matches_restatement_and_plain_iteration(ctx, oracle, S, P, stages):
    from sxxcvr_b200 import Bank, Iir
    rng = np.random.default_rng(S + P)
    lat = latency_ns(768)
    side = torch.cuda.Stream()
    st = side.cuda_stream
    sos_f, sos_g = design(4, 0), design(4, 1)
    with Bank(ctx, S, P, RATE, 1.0e-6, 43) as bank, Bank(ctx, S, P, RATE, 1.0e-6, 43) as plain, \
            Iir(ctx, S, sos_f) as F, Iir(ctx, S, sos_g) as G:
        pre = F if stages in ("pre", "both") else None
        post = G if stages in ("post", "both") else None
        filters, states = [], []
        for filt, sos in ((pre, sos_f), (post, sos_g)):
            if filt is not None:
                z = random_state(rng, 4, S)
                filt.set_state(z, st)
                filters.append((sos, filt))
                states.append(z)
        cf = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        cf_plain = torch.zeros_like(cf)
        out = torch.zeros(S * P * 2, dtype=torch.int32, device="cuda")
        out_plain = torch.zeros_like(out)
        for it in range(3):
            with torch.cuda.stream(side):
                bank.repeat_filtered(cf.data_ptr(), pre, post, lat, st)
                bank.drain(0, S, P, out.data_ptr(), st)
                plain.repeat(cf_plain.data_ptr(), lat, st)
                plain.drain(0, S, P, out_plain.data_ptr(), st)
            side.synchronize()
            rx = as_blocks(cf_plain, S, P)
            for s in (0, S // 2, S - 1):  # the plain iteration's block is the oracle's RX of the capture
                frames = sxtest.synth_frames(oracle, it * P, P, seed=43 + s)
                assert same_bits(rx[s], sxtest.oracle_rx(oracle, frames)), (it, s)
            want = run_restatement(filters, rx, states)
            got = as_blocks(cf, S, P)
            assert same_bits(got, want), (it, "filtered block")
            if not filters:
                assert same_bits(got, rx) and np.array_equal(out.cpu().numpy(), out_plain.cpu().numpy())
            assert np.array_equal(out.cpu().numpy(), sxtest.oracle_tx(oracle, want.view(np.float32).reshape(-1), 1.0e-6)), it
            for a, b in zip(bank.positions(st), plain.positions(st)):
                assert np.array_equal(a, b)
            assert all(np.array_equal(a, b) for a, b in zip(bank.last_read(st), plain.last_read(st)))
            assert np.array_equal(bank.last_write(st), plain.last_write(st))
        for (sos, filt), z in zip(filters, states):
            assert same_bits(filt.state(st), z)


@pytest.mark.parametrize("case", ["synthetic", "ingested", "late"])
def test_fused_equals_the_split_sequence(ctx, case):
    """repeat_filtered(F, G) against read, F.apply, G.apply, write(HAS_TIME, rx time + offset) on a
    twin bank with twin filters.  `synthetic` writes 769 frames after the read (blocks straddle two
    slices of the ring), `ingested` converts frames from outside, `late` writes one frame after the
    read's first frame, which is before the read ends: every write is dropped, the filters run."""
    from sxxcvr_b200 import Bank, Iir
    S, P = 2100, 256
    rng = np.random.default_rng(11)
    lat = latency_ns({"synthetic": 769, "ingested": 768, "late": 1}[case])
    side = torch.cuda.Stream()
    st = side.cuda_stream
    sos_f, sos_g = design(3, 0), design(5, 1)
    with Bank(ctx, S, P, RATE, 1.0e-6, 5) as fused, Bank(ctx, S, P, RATE, 1.0e-6, 5) as split, \
            Iir(ctx, S, sos_f) as F1, Iir(ctx, S, sos_g) as G1, Iir(ctx, S, sos_f) as F2, Iir(ctx, S, sos_g) as G2:
        zf, zg = random_state(rng, 3, S), random_state(rng, 5, S)
        for f, z in ((F1, zf), (F2, zf), (G1, zg), (G2, zg)):
            f.set_state(z, st)
        cf1 = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        cf2 = torch.zeros_like(cf1)
        out1 = torch.zeros(S * P * 2, dtype=torch.int32, device="cuda")
        out2 = torch.zeros_like(out1)
        for it in range(3):
            with torch.cuda.stream(side):
                if case == "ingested":
                    frames = torch.from_numpy(rng.integers(-2**31, 2**31, S * P * 2, dtype=np.int64).astype(np.int32)).cuda()
                    fused.ingest(0, S, frames.data_ptr(), st)
                    split.ingest(0, S, frames.data_ptr(), st)
                fused.repeat_filtered(cf1.data_ptr(), F1, G1, lat, st)
                split.read(cf2.data_ptr(), st)
                F2.apply(cf2.data_ptr(), P, st)
                G2.apply(cf2.data_ptr(), P, st)
                split.write(cf2.data_ptr(), HAS_TIME, None, lat, st)
                fused.drain(0, S, P, out1.data_ptr(), st)
                split.drain(0, S, P, out2.data_ptr(), st)
            side.synchronize()
            assert same_bits(cf1.cpu().numpy(), cf2.cpu().numpy()), it
            assert np.array_equal(out1.cpu().numpy(), out2.cpu().numpy()), it
            for a, b in zip(fused.positions(st), split.positions(st)):
                assert np.array_equal(a, b)
            assert all(np.array_equal(a, b) for a, b in zip(fused.last_read(st), split.last_read(st)))
            assert np.array_equal(fused.last_write(st), split.last_write(st))
            assert same_bits(F1.state(st), F2.state(st)) and same_bits(G1.state(st), G2.state(st))
        _, rxp, txp = fused.positions(st)
        if case == "late":
            assert (txp == 0).all()                       # nothing was written ...
            assert not same_bits(F1.state(st), zf)        # ... and the filters advanced all the same
        else:
            assert (txp > 0).all()


@pytest.mark.parametrize("S,P", [(5, 256), (32768 + 3, 64)])
def test_filtered_hook_example(ctx, hooklib, S, P):
    """examples/repeater_hook.cu: filter -> clip/gain -> filter in the fused iteration."""
    from sxxcvr_b200 import Bank, Iir
    lat = latency_ns(768)
    side = torch.cuda.Stream()
    st = side.cuda_stream
    sos_f, sos_g = design(4, 0), design(4, 1)
    with Bank(ctx, S, P, RATE, 1.0e-6, 41) as bank, Bank(ctx, S, P, RATE, 1.0e-6, 41) as plain, \
            Iir(ctx, S, sos_f) as F, Iir(ctx, S, sos_g) as G:
        zf = zg = None
        lf = lg = None
        cf = torch.zeros(S * P * 2, dtype=torch.float32, device="cuda")
        cf_plain = torch.zeros_like(cf)
        for it in range(3):
            with torch.cuda.stream(side):
                assert hooklib.sx_example_repeat_filtered_clip_gain(bank.handle, F.handle, G.handle, cf.data_ptr(), lat,
                                                                    PRE, POST, st) == 0
                plain.repeat(cf_plain.data_ptr(), lat, st)
            side.synchronize()
            rx = as_blocks(cf_plain, S, P)
            a, zf = sxiir.sosfilt(sos_f, rx, zf)
            b = clip_gain_exact(a.view(np.float32).reshape(-1)).view(np.complex64).reshape(S, P)
            want, zg = sxiir.sosfilt(sos_g, b, zg)
            got = as_blocks(cf, S, P)
            assert same_bits(got, want), it
            # scipy and the script's literal clipper: the clipper's few ulp (of at most 0.3) through the filter
            s32 = sxiir.sos32(sos_f)
            a2, lf = signal.sosfilt(s32, rx, axis=-1, zi=lf if lf is not None else np.zeros((4, S, 2), np.complex64))
            b2 = clip_gain_literal(a2.view(np.float32).reshape(-1)).view(np.complex64).reshape(S, P)
            lit, lg = signal.sosfilt(sxiir.sos32(sos_g), b2, axis=-1, zi=lg if lg is not None else np.zeros((4, S, 2), np.complex64))
            assert np.abs(got - lit).max() <= 1e-5, it


def test_invalid_arguments_are_refused(ctx):
    from sxxcvr_b200 import Bank, Context, Iir
    from sxxcvr_b200.capi import ERR_INVALID, SxGpuError
    good = design(2)

    def refused(fn):
        with pytest.raises(SxGpuError) as e:
            fn()
        assert e.value.code == ERR_INVALID

    bad_a0 = good.copy()
    bad_a0[1, 3] = 2.0
    nan = good.copy()
    nan[0, 1] = np.nan
    refused(lambda: Iir(ctx, 4, bad_a0))
    refused(lambda: Iir(ctx, 4, nan))
    refused(lambda: Iir(ctx, 4, np.zeros((0, 6))))
    refused(lambda: Iir(ctx, 4, np.tile(good[:1], (9, 1))))
    S, P = 5, 256
    cf = torch.zeros(S * P * 2 + 8, dtype=torch.float32, device="cuda")
    with Bank(ctx, S, P) as bank, Bank(ctx, S, 255) as odd, Iir(ctx, S, good) as F, Iir(ctx, S + 1, good) as other:
        refused(lambda: bank.repeat_filtered(cf.data_ptr(), other, None))
        refused(lambda: bank.repeat_filtered(cf.data_ptr(), None, other))
        refused(lambda: bank.repeat_filtered(cf.data_ptr(), F, F))
        refused(lambda: odd.repeat_filtered(cf.data_ptr(), F, None))
        refused(lambda: bank.repeat_filtered(cf.data_ptr() + 8, F, None))
        refused(lambda: F.apply(cf.data_ptr(), 0))
        refused(lambda: F.apply(cf.data_ptr(), 65537))
        refused(lambda: F.apply(cf.data_ptr() + 4, P))
        bank.repeat_filtered(cf.data_ptr(), F, None)  # and the same call with good arguments runs
        ctx.stream_sync()
    c2 = Context(0)
    f = Iir(c2, 4, good)
    assert c2.lib.sxgpu_destroy(c2.handle) == ERR_INVALID  # refused while the filter is alive
    f.close()
    c2.close()
