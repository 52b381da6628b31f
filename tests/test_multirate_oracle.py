"""The generic multirate classes (SURVEY 8(f)-4: Filters/Decimator.cc, Interpolator.cc,
Int16/Decimator_int16.cc, Int16/Interpolator_int16.cc): the oracle's restatement against the
reference's own test programs (testDecimator.cc, testInterpolator.cc), the compiled reference
and the golden vectors it produced."""
import os
import re

import numpy as np
import pytest

import _oracle as O
import _pins

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = np.load(os.path.join(HERE, "golden", "golden_multirate_v1.npz"))
CASES = [m.split(",") for m in GOLD["meta"]]
have_ref = O.ref("radiodiags") is not None
f32 = np.float32


@pytest.mark.parametrize("name,kind,factor", CASES)
def test_oracle_reproduces_the_reference_golden_vectors(name, kind, factor):
    m = O.Multirate(int(kind), GOLD["taps_" + name], int(factor))
    assert np.array_equal(m.run(GOLD["x_" + name]), GOLD["y_" + name])


@pytest.mark.parametrize("name,kind,factor", CASES)
def test_result_does_not_depend_on_how_the_stream_is_cut(name, kind, factor):
    x, m = GOLD["x_" + name], O.Multirate(int(kind), GOLD["taps_" + name], int(factor))
    cuts = [0, 1, 2, 7, 8, 50, 51, 333, x.size]
    y = np.concatenate([m.run(x[a:b]) for a, b in zip(cuts[:-1], cuts[1:])])
    assert np.array_equal(y, GOLD["y_" + name])


def test_decimator_known_answers():
    # testDecimator.cc: M = 1 impulse gives the taps; M = 2 step gives every second partial sum
    h = np.array([1, 2, 3, 4, 1, 1, 1, 8], dtype=f32)
    imp = np.array([1] + [0] * 18, dtype=f32)
    y = O.Multirate(O.MR_DECIMATOR_F32, h, 1).run(imp)
    assert np.array_equal(y[:8], h) and not y[8:].any()
    y = O.Multirate(O.MR_DECIMATOR_F32, h, 2).run(np.ones(20, dtype=f32))
    full = np.concatenate([np.cumsum(h), np.full(12, h.sum())]).astype(f32)
    assert np.array_equal(y, full[1::2])


def test_interpolator_known_answers():
    # testInterpolator.cc: prototype {1..8}, L = 2: the impulse response is the prototype itself
    # (p0 = h0 h2 h4 h6, p1 = h1 h3 h5 h7), the step response the running sums of each phase
    h = np.arange(1, 9, dtype=f32)
    m = O.Multirate(O.MR_INTERPOLATOR_F32, h, 2)
    y = m.run(np.array([1] + [0] * 19, dtype=f32))
    assert np.array_equal(y[:8], h) and not y[8:].any()
    y = m.run(np.ones(20, dtype=f32))  # same object, as the reference's test does
    assert np.array_equal(y[:8], np.array([1, 2, 4, 6, 9, 12, 16, 20], dtype=f32))
    assert np.array_equal(y[8:10], np.array([16, 20], dtype=f32))


def test_int16_unity_tap_negates():
    # 1.0 * 32768 does not fit int16: the cast leaves -32768 (SURVEY A.5-5)
    x = np.array([100, -200, 32767, -32768, 5], dtype=np.int16)
    y = O.Multirate(O.MR_DECIMATOR_I16, np.array([1.0], dtype=f32), 1).run(x)
    # ... and -32768 * -32768 + 16384 runs into the clamp at 2^30 - 1
    exp = [min((1 << 14) - 32768 * int(v), 0x3fffffff) >> 15 for v in x]
    assert [int(v) for v in y] == exp == [-100, 200, -32767, 32767, -5]


@pytest.mark.parametrize("kind", [1, 2, 3, 4])
def test_oracle_matches_compiled_reference_on_random_filters(kind):
    got, ref = [], []
    rng = np.random.default_rng(100 + kind)
    for trial in range(12):
        factor = int(rng.integers(1, 7))
        q = int(rng.integers(1, 30))
        n_taps = q * factor if kind in (2, 4) else int(rng.integers(1, 100))
        taps = (rng.normal(0, 0.4, n_taps) * rng.choice([0.1, 1.0, 2.5])).astype(f32)
        n = int(rng.integers(1, 700))
        x = rng.integers(-32768, 32768, n).astype(np.int16 if kind >= 3 else f32)
        for out, impl in ((got, "oracle"), (ref, "ref")) if have_ref else ((got, "oracle"),):
            m = O.Multirate(kind, taps, factor, impl=impl)
            out.extend(m.run(piece) for piece in np.array_split(x, 3))
            m.reset()
            out.append(m.run(x))
    _pins.expect("multirate_random_filters/%d" % kind, got, ref if have_ref else None)


REF_FILTERS = "/root/reference/radioDiags/Filters"


def _taps_from_source(path, name):
    """The tap table of one of the reference's audio tools, parsed where the file lies."""
    src = open(path).read()
    body = re.search(name + r"\[\]\s*=\s*\{(.*?)\};", src, re.S).group(1)
    body = re.sub(r"//[^\n]*", "", body)
    return np.array([float(v) for v in body.replace("\n", " ").split(",") if v.strip()], dtype=f32)


@pytest.mark.skipif(not (have_ref and os.path.exists(REF_FILTERS + "/original32000.raw")),
                    reason="reference tree not mounted")
def test_the_references_audio_tools_inputs():
    # decimateAudio.cc:149 (Decimator, h32000, 4), Int16/decimateAudio.cc:149 (Decimator_int16),
    # interpolateAudio.cc:106 (Interpolator, h16000, 2), on the captures shipped next to them
    x32 = np.fromfile(REF_FILTERS + "/original32000.raw", dtype=np.int16)
    x8 = np.fromfile(REF_FILTERS + "/original8000.raw", dtype=np.int16)
    h32 = _taps_from_source(REF_FILTERS + "/decimateAudio.cc", "h32000")
    h16 = _taps_from_source(REF_FILTERS + "/interpolateAudio.cc", "h16000")
    assert h32.size == 80 and h16.size % 2 == 0
    for kind, taps, factor, x in ((1, h32, 4, x32.astype(f32)), (3, h32, 4, x32), (2, h16, 2, x8.astype(f32)),
                                  (4, h16, 2, x8)):
        ya = O.Multirate(kind, taps, factor).run(x)
        yb = O.Multirate(kind, taps, factor, impl="ref").run(x)
        assert ya.size == (x.size * factor if kind in (2, 4) else x.size // factor)
        assert ya.tobytes() == yb.tobytes()
