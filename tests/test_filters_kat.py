"""Known-answer tests of the filter building blocks, taken from the reference's own
test programs (radioDiags/Filters/test{Fir,Iir}Filter.cc, testDecimator.cc,
Int16/decimateAudio.cc), against the oracle and -- where built -- the compiled reference.
"""
import numpy as np
import pytest

import _oracle as O
import _pins

L = O.oracle()
have_ref = O.ref("radiodiags") is not None
f32 = np.float32

TAPS = np.array([1, 2, 3, 4, 1, 1, 1, 8], dtype=f32)        # testFirFilter.cc:25
IMPULSE = np.array([1] + [0] * 18, dtype=f32)               # testFirFilter.cc:26
STEP = np.ones(19, dtype=f32)                               # testFirFilter.cc:27


def fir_oracle(h, x):
    f = L.sdro_fir_new(len(h), O._ptr(np.ascontiguousarray(h, dtype=f32), O._pf))
    y = np.zeros(len(x), dtype=f32)
    L.sdro_fir_run(f, O._ptr(np.ascontiguousarray(x, dtype=f32), O._pf), len(x), O._ptr(y, O._pf))
    L.sdro_fir_free(f)
    return y


def iir_oracle(b, a, x):
    f = L.sdro_iir_new(len(b), O._ptr(np.ascontiguousarray(b, dtype=f32), O._pf), len(a),
                       O._ptr(np.ascontiguousarray(a, dtype=f32), O._pf))
    y = np.zeros(len(x), dtype=f32)
    L.sdro_iir_run(f, O._ptr(np.ascontiguousarray(x, dtype=f32), O._pf), len(x), O._ptr(y, O._pf))
    L.sdro_iir_free(f)
    return y


def dec16_oracle(h, M, x):
    d = L.sdro_dec16_new(len(h), O._ptr(np.ascontiguousarray(h, dtype=f32), O._pf), M)
    y = np.zeros(len(x) // M + 1, dtype=np.int16)
    n = L.sdro_dec16_run(d, O._ptr(np.ascontiguousarray(x, dtype=np.int16), O._pi16), len(x), O._ptr(y, O._pi16))
    L.sdro_dec16_free(d)
    return y[:n]


def test_fir_impulse_response_is_the_taps_newest_sample_meets_tap0():
    y = fir_oracle(TAPS, IMPULSE)
    assert np.array_equal(y[:8], TAPS) and not y[8:].any()


def test_fir_step_response_is_cumulative_sum():
    y = fir_oracle(TAPS, STEP)
    exp = np.concatenate([np.cumsum(TAPS), np.full(11, TAPS.sum())]).astype(f32)
    assert np.array_equal(y, exp)


def test_iir_one_pole_impulse_and_step():          # testIirFilter.cc:26-27: b={1}, a={0.5}
    y = iir_oracle([1], [0.5], IMPULSE)
    assert np.array_equal(y, np.array([(-0.5) ** n for n in range(19)], dtype=f32))
    y = iir_oracle([1], [0.5], STEP)
    e, acc = [], f32(0)
    for _ in range(19):
        acc = f32(f32(1) - f32(f32(0.5) * acc))
        e.append(acc)
    assert np.array_equal(y, np.array(e, dtype=f32))


def test_dc_block_impulse_and_step():              # testIirFilter.cc:28-29: b={1,-1}, a={-0.95}
    for x in (IMPULSE, STEP):
        y = iir_oracle([1, -1], [-0.95], x)
        e, x1, y1 = [], f32(0), f32(0)
        for v in x:
            yn = f32(f32(v + f32(f32(-1) * x1)) - f32(f32(-0.95) * y1))
            e.append(yn)
            x1, y1 = v, yn
        assert np.array_equal(y, np.array(e, dtype=f32))
    assert abs(float(iir_oracle([1, -1], [-0.95], STEP)[-1])) < 0.5  # DC decays


def q15(h):
    return np.array([np.int16(np.int32(np.round(f32(f32(v) * f32(32768)))) & 0xFFFF) for v in h]).astype(np.int16)


def q15_decimate_numpy(h, M, x):
    """y[m] = (16384 + sum_k q[k] x[M m + M-1-k]) >> 15, zero history, no clamp reached."""
    q = q15(h).astype(np.int64)
    xp = np.concatenate([np.zeros(len(h), dtype=np.int64), np.asarray(x, dtype=np.int64)])
    out = []
    for m in range(len(x) // M):
        n0 = len(h) + M * m + M - 1
        acc = 16384 + sum(int(q[k]) * int(xp[n0 - k]) for k in range(len(h)))
        out.append(np.int16(acc >> 15))
    return np.array(out, dtype=np.int16)


@pytest.mark.parametrize("M", [1, 2, 4])           # testDecimator.cc:43,72 use M=1 impulse, M=2 step
def test_q15_decimator_known_answers(M):
    h = TAPS / 16.0
    imp = np.zeros(24, dtype=np.int16)
    imp[0] = 1600
    step = np.full(24, 1600, dtype=np.int16)
    for x in (imp, step):
        assert np.array_equal(dec16_oracle(h, M, x), q15_decimate_numpy(h, M, x))
    if M == 1:
        assert np.array_equal(dec16_oracle(h, 1, imp)[:8], (TAPS * 100).astype(np.int16))


def test_tap_quantisation_quirks():
    # 1.0 -> 32768.0 -> (int16) -32768 (SsbDemodulator.cc:71, SURVEY A.5-5)
    assert q15([1.0])[0] == -32768
    y = dec16_oracle([0.0] * 15 + [1.0], 1, np.arange(1, 40, dtype=np.int16))
    assert np.array_equal(y[15:], -np.arange(1, 25, dtype=np.int16)) and not y[:15].any()


def test_q15_clamp_is_per_tap_and_order_dependent():
    # +max then -max: an unclamped sum would cancel; the per-tap clamp does not
    h = [0.9999, 0.9999, -0.9999, -0.9999]
    x = np.array([32767] * 8, dtype=np.int16)
    y = dec16_oracle(h, 1, x)
    q = q15(h).astype(np.int64)
    acc = 16384
    for k in range(4):
        acc += int(q[k]) * 32767
        acc = min(max(acc, -(1 << 30)), (1 << 30) - 1)
    assert y[-1] == np.int16(acc >> 15) and y[-1] != 0


def test_building_blocks_match_compiled_reference_on_random_input():
    R = O.ref("radiodiags")
    got, ref = [], []
    rng = np.random.default_rng(3)
    x = rng.integers(-32768, 32768, size=200000, dtype=np.int16)
    x[1000:1200] = 32767
    x[1200:1400] = -32768
    for fid, M in [(0, 4), (1, 4), (2, 2), (3, 4), (4, 4), (5, 2), (6, 1), (7, 4), (8, 1), (9, 1)]:
        # the float designs are not exported; compare through each library's own quantiser
        hq = O.q15_taps(fid).astype(f32) / f32(32768)
        hq = np.where(O.q15_taps(fid) == -32768, f32(1.0), hq).astype(f32)
        got.append(dec16_oracle(hq, M, x))
        if R:
            d = R.ref_dec16_new(len(hq), O._ptr(hq, O._pf), M)
            yr = np.zeros(len(x) // M + 1, dtype=np.int16)
            n = R.ref_dec16_run(d, O._ptr(x, O._pi16), len(x), O._ptr(yr, O._pi16))
            R.ref_dec16_free(d)
            ref.append(yr[:n])
    xf = rng.standard_normal(5000).astype(f32)
    got.append(fir_oracle(TAPS, xf))
    if R:
        f = R.ref_fir_new(8, O._ptr(TAPS, O._pf))
        yr = np.zeros(5000, dtype=f32)
        R.ref_fir_run(f, O._ptr(xf, O._pf), 5000, O._ptr(yr, O._pf))
        R.ref_fir_free(f)
        ref.append(yr)
    for b, a in [([1, -1], [-0.95]), ([0.0253863, 0.0253863], [-0.9492274]), ([1], [0.5])]:
        got.append(iir_oracle(b, a, xf))
        if R:
            bb, aa = np.array(b, dtype=f32), np.array(a, dtype=f32)
            f = R.ref_iir_new(len(bb), O._ptr(bb, O._pf), len(aa), O._ptr(aa, O._pf))
            yr = np.zeros(5000, dtype=f32)
            R.ref_iir_run(f, O._ptr(xf, O._pf), 5000, O._ptr(yr, O._pf))
            R.ref_iir_free(f)
            ref.append(yr)
    _pins.expect("building_blocks", got, ref if R else None)


def test_decimate_audio_program_shape():
    """Int16/decimateAudio.cc: 16-tap 4:1 Decimator_int16 over 10 s of 32 kS/s audio."""
    h32000 = np.array([-0.0084477, 0.0084043, 0.0075154, 0.0064417, 0.0039647, 0.0002320, -0.0034617,
                       -0.0054143, -0.0044711, -0.0008117, 0.0038463, 0.0071423, 0.0070406, 0.0031175,
                       -0.0030506, -0.0084477], dtype=f32)
    x = (12000 * np.sin(2 * np.pi * 440 * np.arange(320000) / 32000)).astype(np.int16)
    got = dec16_oracle(h32000, 4, x)
    assert got.size == 80000
    R, ref = O.ref("radiodiags"), None
    if R:
        d = R.ref_dec16_new(16, O._ptr(h32000, O._pf), 4)
        yr = np.zeros(80001, dtype=np.int16)
        n = R.ref_dec16_run(d, O._ptr(x, O._pi16), len(x), O._ptr(yr, O._pi16))
        R.ref_dec16_free(d)
        ref = [yr[:n]]
    _pins.expect("decimate_audio_program", [got], ref)
