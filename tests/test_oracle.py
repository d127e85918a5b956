"""CPU tests of the checker itself: the plain-C oracle against the golden vectors generated from
the unmodified reference, against the reference live (when oracle/_ref was built), and against
the known answers recorded in SURVEY.md's appendices."""
import json

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

import sxtest

KAT = json.loads((sxtest.GOLDEN / "convert_kat.json").read_text())


def unhex(words, dtype):
    return np.array([int(w, 16) for w in words], dtype=np.uint32).view(dtype)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def test_rx_golden_vectors(oracle):
    words = unhex(KAT["rx"]["in"], np.int32)
    want = unhex(KAT["rx"]["out"], np.uint32)
    assert np.array_equal(bits(sxtest.oracle_rx(oracle, words)), want)


@pytest.mark.parametrize("case", KAT["tx"], ids=lambda c: f"{c['set']}-{c['thr2']}")
def test_tx_golden_vectors(oracle, case):
    f = unhex(case["in"], np.float32)
    thr2 = float(unhex([case["thr2"]], np.float32)[0])
    assert np.array_equal(bits(sxtest.oracle_tx(oracle, f, thr2)), unhex(case["out"], np.uint32))


def test_tx_arm_semantics_where_reference_is_undefined(oracle):
    arm = KAT["tx_arm_semantics"]
    thr2 = float(unhex([arm["thr2"]], np.float32)[0])
    for c in arm["cases"]:
        got = bits(sxtest.oracle_tx(oracle, unhex(c["in"], np.float32), thr2))
        assert [format(int(x), "08x") for x in got] == c["out"], c


def test_survey_rx_kats(oracle):
    kat = {0: 0x00000000, 1: 0x30000000, -1: 0xB0000000, 2**31 - 1: 0x3F800000, -2**31: 0xBF800000,
           0x7FFFFF80: 0x3F7FFFFF, 0x7FFFFFBF: 0x3F7FFFFF, 0x7FFFFFC0: 0x3F800000, 16777217: 0x3C000000,
           0x12345678: 0x3E11A2B4, 0x87654321 - 2**32: 0xBF71357A}
    words = np.array(list(kat) + [0], dtype=np.int64).astype(np.int32)
    assert [int(x) for x in bits(sxtest.oracle_rx(oracle, words))[:len(kat)]] == list(kat.values())


def test_survey_tx_kats(oracle):
    thr = sxtest.THR2_DEFAULT
    f = np.array([-1.0, -1.0, 0.99999994, -0.99999994, 0.3, -0.3, 1e-3, 0.0, 0.000707106781, 0.000707106781,
                  0.0, -0.0, -6.98e-10, 6.98e-10], np.float32)
    got = [int(x) for x in bits(sxtest.oracle_tx(oracle, f, thr))]
    assert got == [0x80000003, 0x80000000, 0x7FFFFF83, 0x80000080, 0x26666683, 0xD9999980, 0x0020C49B, 0,
                   0x00172BA4, 0x00172BA4, 0, 0, 0xFFFFFFFC, 0]
    got0 = [int(x) for x in bits(sxtest.oracle_tx(oracle, f[8:12], 0.0))]
    assert got0 == [0x00172BA7, 0x00172BA4, 3, 0]


def test_oracle_equals_reference_on_defined_domain(oracle, ref):
    words = np.concatenate([sxtest.rx_structured(), sxtest.rx_uniform(1 << 18)])
    assert np.array_equal(bits(sxtest.oracle_rx(oracle, words)), bits(sxtest.ref_rx(ref, words)))
    for f in (sxtest.tx_uniform(1 << 18), sxtest.tx_gaussian_defined(1 << 18),
              sxtest.tx_threshold_circle(1 << 18, sxtest.THR2_DEFAULT), sxtest.tx_threshold_circle(1 << 16, 0.25)):
        for thr2 in (sxtest.THR2_DEFAULT, 0.0, 0.25, 1e-12):
            assert np.array_equal(sxtest.oracle_tx(oracle, f, thr2), sxtest.ref_tx(ref, f, thr2))


def test_reference_x86_build_differs_only_in_its_undefined_domain(oracle, ref):
    """Documents the parity policy: on NaN / >= 1.0 the x86 build of the reference gives the
    cvttss2si 'integer indefinite' 0x80000000 (or a compile-time folded INT_MAX), the oracle gives
    the ARM answers.  Everywhere else they agree word for word."""
    f = sxtest.tx_specials()
    a = sxtest.oracle_tx(oracle, f, sxtest.THR2_DEFAULT).reshape(-1, 2)
    b = sxtest.ref_tx(ref, f, sxtest.THR2_DEFAULT).reshape(-1, 2)
    fin = f.reshape(-1, 2)
    undefined = np.isnan(fin) | (fin >= 1.0)
    assert np.array_equal(a[~undefined], b[~undefined])
    assert (a[undefined] != b[undefined]).any()
    one = np.array([1.0, 0.0], np.float32)       # SoapySX/test/test_timestamps.py:34 sends exactly this
    assert [int(x) for x in bits(sxtest.ref_tx(ref, one, 1e-6))] == [0x80000003, 0]       # x86: wraps negative
    assert [int(x) for x in bits(sxtest.oracle_tx(oracle, one, 1e-6))] == [0x7FFFFFFF, 0]  # ARM: saturates


@settings(max_examples=200, deadline=None)
@given(st.lists(st.integers(-2**31, 2**31 - 1), min_size=2, max_size=64).filter(lambda v: len(v) % 2 == 0))
def test_rx_properties(oracle, vals):
    w = np.array(vals, dtype=np.int64).astype(np.int32)
    out = sxtest.oracle_rx(oracle, w)
    assert (np.abs(out) <= 1.0).all()
    # exact: float32(x) * 2^-31 with round-to-nearest-even int->float
    assert np.array_equal(bits(out), bits((w.astype(np.float32) * np.float32(2.0**-31))))
    neg = np.where(w == -2**31, w, -w)           # odd symmetry except at INT32_MIN
    assert np.array_equal(sxtest.oracle_rx(oracle, neg)[w != -2**31], -out[w != -2**31])


@settings(max_examples=200, deadline=None)
@given(st.lists(st.floats(width=32, allow_nan=True, allow_infinity=True), min_size=2, max_size=64)
       .filter(lambda v: len(v) % 2 == 0), st.sampled_from([0.0, 1e-6, 0.25, 1.0]))
def test_tx_properties(oracle, vals, thr2):
    f = np.array(vals, np.float32)
    out = bits(sxtest.oracle_tx(oracle, f, thr2)).reshape(-1, 2)
    fin = f.reshape(-1, 2)
    assert ((out[:, 1] & 3) == 0).all()                       # Q low bits reserved 0 (SoapySX.cpp:128-131)
    assert np.isin(out[:, 0] & 3, (0, 3)).all()               # I low bits are both set or both clear
    with np.errstate(over="ignore", invalid="ignore"):
        mag2 = (fin[:, 0] * fin[:, 0]).astype(np.float32) + (fin[:, 1] * fin[:, 1]).astype(np.float32)
        on = mag2 >= np.float32(thr2)
    assert np.array_equal((out[:, 0] & 3) == 3, on)
    top = (out & 0xFFFFFFFC).view(np.int32).astype(np.int64)
    with np.errstate(invalid="ignore", over="ignore"):
        exact = np.trunc(np.clip(np.nan_to_num(fin.astype(np.float64), nan=0.0), -1.0, 1.0) * 2.0**31)
    exact = np.minimum(exact, 2.0**31 - 1)
    assert ((exact - top >= 0) & (exact - top < 4) | (exact < 0) & (top - exact <= 0) & (exact - top < 4)).all()


def numpy_tx(f: np.ndarray, thr2: float) -> np.ndarray:
    """A second, independent restatement of SoapySX.cpp:116-137 (ARM semantics where C++ is
    undefined), in numpy float32 arithmetic: every operation is a single IEEE single-precision
    operation, so nothing can be fused."""
    f = np.ascontiguousarray(f, np.float32)
    one, two31 = np.float32(1.0), np.float32(2147483648.0)
    with np.errstate(invalid="ignore", over="ignore"):
        c = np.where(one < f, one, f)                       # std::min(f, 1.0f): NaN stays
        c = np.where(c < -one, -one, c).astype(np.float32)  # std::max(., -1.0f)
        p = (c * two31).astype(np.float32)
        t = np.trunc(p.astype(np.float64))
        v = np.where(np.isnan(p), 0.0, np.clip(t, -2.0**31, 2.0**31 - 1)).astype(np.int64)
        v = (v & 0xFFFFFFFC).astype(np.uint32)
        pairs = f.reshape(-1, 2)
        mag2 = ((pairs[:, 0] * pairs[:, 0]).astype(np.float32) + (pairs[:, 1] * pairs[:, 1]).astype(np.float32)).astype(np.float32)
        on = mag2 >= np.float32(thr2)
    out = v.reshape(-1, 2).copy()
    out[on, 0] |= 3
    return out.ravel()


@pytest.mark.parametrize("thr2", [sxtest.THR2_DEFAULT, 0.0, 0.25, 2.0, float("nan")])
def test_oracle_agrees_with_an_independent_numpy_restatement(oracle, thr2):
    sets = [sxtest.tx_uniform(1 << 16), sxtest.tx_gaussian_defined(1 << 16), sxtest.tx_specials(),
            sxtest.tx_threshold_circle(1 << 16, sxtest.THR2_DEFAULT), sxtest.tx_threshold_circle(1 << 14, 0.25)]
    rng = np.random.default_rng(3)
    sets.append(rng.integers(0, 2**32, size=1 << 17, dtype=np.uint64).astype(np.uint32).view(np.float32))  # any bit pattern
    for f in sets:
        assert np.array_equal(bits(sxtest.oracle_tx(oracle, f, thr2)), numpy_tx(f, thr2))


def test_rx_then_tx_is_not_identity_but_close(oracle):
    w = sxtest.rx_uniform(1 << 16)
    back = sxtest.oracle_tx(oracle, sxtest.oracle_rx(oracle, w), 3.0)
    assert (back == w).mean() < 0.1                           # never test loopback as identity (SURVEY.md A.4)
    assert np.abs(back.astype(np.int64) - w.astype(np.int64)).max() <= 132


def test_offsets_are_in_frames(oracle):
    w = sxtest.rx_uniform(64)
    out = np.zeros(128, np.float32)
    oracle.sxo_convert_rx_buffer(w.ctypes.data, 5, out.ctypes.data, 9, 20)
    assert np.array_equal(out[18:58], sxtest.oracle_rx(oracle, w[10:50]))
    assert (out[:18] == 0).all() and (out[58:] == 0).all()


# ---- timestamps (SoapySDR Time.hpp restatement; SURVEY.md Appendix C) ----------------------------
def test_time_kats(oracle):
    t2n, n2t = oracle.sxo_ticks_to_time_ns, oracle.sxo_time_ns_to_ticks
    assert t2n(256, 75000.0) == 3_413_333
    assert t2n(768, 75000.0) == 10_240_000
    assert t2n(75000, 75000.0) == 1_000_000_000
    assert n2t(10_240_000, 75000.0) == 768
    r = 32.0e6 / 1536
    assert t2n(256, r) == 12_288_000
    assert t2n(10**6, r) == 48_000_000_000


@pytest.mark.parametrize("rate", sxtest.RATES)
def test_time_round_trip_and_constant_latency(oracle, rate):
    t2n, n2t = oracle.sxo_ticks_to_time_ns, oracle.sxo_time_ns_to_ticks
    lat = int(round(768 * 1e9 / rate))
    for p in list(range(0, 256 * 4000, 256)) + [2**40 + 256 * k for k in range(100)] + [1, 7, 255, 75001]:
        assert n2t(t2n(p, rate), rate) == p
        assert n2t(t2n(p, rate) + lat, rate) == p + 768


@settings(max_examples=3000, deadline=None)
@given(st.floats(min_value=1.0e3, max_value=1.0e8, allow_nan=False, allow_infinity=False), st.integers(0, 2**45))
def test_time_round_trip_over_arbitrary_rates(oracle, rate, ticks):
    """What upstream SoapySDR documents for Time.hpp -- ticks -> ns -> ticks is the identity for any
    rate whose tick is longer than a nanosecond -- and agreement with exact rational arithmetic to
    within the one rounding each direction makes.  (A property of OUR restatement of TimeC.cpp:
    SoapySDR itself is not installed here, so parity with upstream stays unpinned; DESIGN.md.)"""
    from fractions import Fraction
    from hypothesis import assume
    assume((ticks + 1) * 1e9 / rate < 2**62)      # the timestamp itself must fit in int64
    t2n, n2t = oracle.sxo_ticks_to_time_ns, oracle.sxo_time_ns_to_ticks
    ns = t2n(ticks, rate)
    assert n2t(ns, rate) == ticks
    exact = Fraction(ticks) * 10**9 / Fraction(rate)
    assert abs(Fraction(ns) - exact) <= 1
    back = Fraction(ns) * Fraction(rate) / 10**9
    assert abs(back - ticks) <= Fraction(rate) / 10**9 + Fraction(1, 2)
    assert t2n(ticks + 1, rate) > ns              # strictly monotonic: distinct ticks, distinct stamps


def test_time_matches_shim_used_by_both_drivers(oracle):
    """csrc/host/harness_capi.cpp is compiled into the product module and into the reference
    build alike; the product's copy loads without a GPU."""
    import ctypes as C
    from sxxcvr_b200 import _build
    shim = C.CDLL(str(_build.build_soapy_module()))
    shim.sxh_ticks_to_time_ns.argtypes = [C.c_longlong, C.c_double]
    shim.sxh_ticks_to_time_ns.restype = C.c_longlong
    shim.sxh_time_ns_to_ticks.argtypes = [C.c_longlong, C.c_double]
    shim.sxh_time_ns_to_ticks.restype = C.c_longlong
    rng = np.random.default_rng(1)
    for rate in sxtest.RATES:
        for p in rng.integers(0, 2**45, size=200):
            p = int(p)
            assert shim.sxh_ticks_to_time_ns(p, rate) == oracle.sxo_ticks_to_time_ns(p, rate)
            assert shim.sxh_time_ns_to_ticks(p, rate) == oracle.sxo_time_ns_to_ticks(p, rate)


# ---- extensions, stats, synthetic source -------------------------------------------------------------
def test_cs16_extension_specification(oracle):
    w = np.array([0, 0x00010000, -0x00010000, 0x7FFFFFFF, -2**31, 0x0000FFFF, -1, 0x12345678], np.int64).astype(np.int32)
    assert sxtest.oracle_rx_cs16(oracle, w).tolist() == [0, 1, -1, 32767, -32768, 0, -1, 0x1234]
    s = np.array([0, 0, 1, -1, 32767, -32768, 33, 0], np.int16)
    out = bits(sxtest.oracle_tx_cs16(oracle, s, sxtest.THR2_DEFAULT))
    assert [int(x) for x in out] == [0, 0, 0x00010000, 0xFFFF0000, 0x7FFF0003, 0x80000000, 0x00210003, 0]


def test_s16_frame_extension_specification(oracle):
    s = np.array([0, 1, -1, 32767, -32768, 16384, -16384, 3], np.int16)
    f = sxtest.oracle_rx_s16(oracle, s)
    assert f.tolist() == [0.0, 2.0**-15, -(2.0**-15), 32767 / 32768, -1.0, 0.5, -0.5, 3 * 2.0**-15]
    x = np.array([1.0, -1.0, 0.5, -0.5, 2.0, np.nan, 1e-3, 0.0, 0.99997, -3e-5, np.inf, -np.inf], np.float32)
    out = sxtest.oracle_tx_s16(oracle, x, sxtest.THR2_DEFAULT).view(np.uint16)
    assert [int(v) for v in out] == [0x7FFF, 0x8000, 0x4003, 0xC000, 0x7FFC, 0x0000, 0x0023, 0x0000,
                                    0x7FFF, 0x0000, 0x7FFF, 0x8000]


def test_stats_definition(oracle):
    w = np.array([3, 0, 0x7FFFFFFC, 0x80000000, 2, 2, 0xFFFFFFFF, 1], dtype=np.uint32)
    s = sxtest.oracle_stats(oracle, w, 10)
    assert s[0] == int(w.astype(np.uint64).sum())
    assert s[1] == sum(int(x) * (2 * (10 + i) + 1) for i, x in enumerate(w)) % 2**64
    assert s[2] == int(np.bitwise_xor.reduce(w))
    assert s[3] == 8 and s[4] == 3 and s[5] == 2
    a, b = sxtest.oracle_stats(oracle, w[:3], 10), sxtest.oracle_stats(oracle, w[3:], 13)
    assert s == ((a[0] + b[0]) % 2**64, (a[1] + b[1]) % 2**64, a[2] ^ b[2], a[3] + b[3], a[4] + b[4], a[5] + b[5])


def test_synth_frames_are_a_pure_function_of_seed_and_index(oracle):
    a = sxtest.synth_frames(oracle, 0, 1000)
    b = sxtest.synth_frames(oracle, 500, 500)
    assert np.array_equal(a[1000:], b)
    assert not np.array_equal(a, sxtest.synth_frames(oracle, 0, 1000, seed=sxtest.SEED + 1))
    assert abs(float(a.astype(np.float64).mean())) < 2**31 * 0.05       # roughly uniform over the full range


# ---- bookkeeping arithmetic restated in the oracle ------------------------------------------------------
def test_ring_geometry(oracle):
    import ctypes as C
    for arg, want in [(0, (256, 65536)), (256, (256, 65536)), (1024, (1024, 65536)), (1000, (1000, 65000)),
                      (65536, (65536, 65536)), (100000, (65536, 65536)), (3, (3, 65535)), (40000, (40000, 40000))]:
        p, b = C.c_ulong(), C.c_ulong()
        oracle.sxo_alsa_sizes(arg, C.byref(p), C.byref(b))
        assert (p.value, b.value) == want


def test_overrun_and_underrun_arithmetic(oracle):
    assert oracle.sxo_rx_overrun_skip(65536, 65536, 256) == 0
    assert oracle.sxo_rx_overrun_skip(65537, 65536, 256) == 512
    assert oracle.sxo_rx_overrun_skip(65536 + 256, 65536, 256) == 768
    assert oracle.sxo_rx_overrun_skip(200000, 65536, 1024) == (134464 // 1024 + 2) * 1024
    assert oracle.sxo_tx_underrun_forward(100, 100, 256) == 0
    assert oracle.sxo_tx_underrun_forward(101, 100, 256) == 512
    assert oracle.sxo_tx_underrun_forward(100 + 256, 100, 256) == 768
