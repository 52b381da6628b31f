"""The IIR filter bank (SDR_FILTER_IIR_F32, sdr_filter_bank_create_iir): n_rows IirFilter objects
(Filters/IirFilter.cc) on the GPU, bit-identical to the oracle's IirFilter (and, where oracle/_ref is
built, to the compiled reference) however the stream is cut, whatever the segmentation does."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import _oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "rtlsdrdiags_b200", "host")
f32 = np.float32
gpu = pytest.mark.gpu

DEEMPH = ([0.0253863, 0.0253863], [-0.9492274])   # WbFmDemodulator's de-emphasis, 256 kS/s
DC_BLOCK = ([1, -1], [-0.95])                      # the AM / SSB DC block


class Iir:
    """One IirFilter object: the oracle's restatement, or with ref=True the compiled reference."""

    def __init__(self, b, a, ref=False):
        self.b, self.a = np.ascontiguousarray(b, dtype=f32), np.ascontiguousarray(a, dtype=f32)
        self.L, self.pre = (O.ref("radiodiags"), "ref_iir_") if ref else (O.oracle(), "sdro_iir_")
        if self.L is None:
            raise RuntimeError("oracle/_ref is not built")
        self.h = getattr(self.L, self.pre + "new")(self.b.size, O._ptr(self.b, O._pf), self.a.size, O._ptr(self.a, O._pf))
        assert self.h

    def __del__(self):
        if getattr(self, "h", None):
            getattr(self.L, self.pre + "free")(self.h)
            self.h = None

    def run(self, x):
        x = np.ascontiguousarray(x, dtype=f32)
        y = np.zeros(x.size, dtype=f32)
        getattr(self.L, self.pre + "run")(self.h, O._ptr(x, O._pf), x.size, O._ptr(y, O._pf))
        return y


def oracle_rows(b, a, x):
    return np.stack([Iir(b, a).run(r) for r in x])


def _bank(rows, b, a):
    import rtlsdrdiags_b200 as R
    return R.IirFilterBank(rows, b, a)


def stable_denominator(rng, na, radius=0.9):
    """Taps in IirFilter's order (a[0] meets y[n-na], a[k] meets y[n-k]) of a polynomial whose
    roots lie inside |z| < radius."""
    roots = []
    while len(roots) < na:
        r, th = radius * np.sqrt(rng.random()), np.pi * rng.random()
        if na - len(roots) >= 2 and rng.random() < 0.6:
            roots += [r * np.exp(1j * th), r * np.exp(-1j * th)]
        else:
            roots.append(r * np.sign(rng.random() - 0.5))
    c = np.real(np.poly(roots))          # 1, c1, .. c_na: y[n] = fir - sum c_k y[n-k]
    return np.concatenate([[c[na]], c[1:na]]).astype(f32)


# ---------------------------------------------------------------- CPU: argument checks, shapes
def test_argument_checks_without_a_device():
    import rtlsdrdiags_b200 as R
    L = R.load_library()
    h = C.c_void_p()
    t = (C.c_float * 80)(*([0.1] * 80))
    assert L.sdr_filter_bank_create_iir(0, 4, t, 0, t, 1, C.byref(h)) == -1    # nb = 0
    assert L.sdr_filter_bank_create_iir(0, 4, t, 2, t, 0, C.byref(h)) == -1    # na = 0
    assert L.sdr_filter_bank_create_iir(0, 4, t, 2, t, 9, C.byref(h)) == -1    # na = 9
    assert L.sdr_filter_bank_create_iir(0, 4, t, 65, t, 1, C.byref(h)) == -1   # nb = 65
    assert L.sdr_filter_bank_create_iir(0, 4, None, 2, t, 1, C.byref(h)) == -1
    assert L.sdr_filter_bank_create_iir(0, 4, t, 2, None, 1, C.byref(h)) == -1
    assert L.sdr_filter_bank_create_iir(0, 0, t, 2, t, 1, C.byref(h)) == -1    # no rows
    assert L.sdr_filter_bank_create_iir(0, 65536, t, 2, t, 1, C.byref(h)) == -1
    assert L.sdr_filter_bank_create_iir(0, 4, t, 2, t, 1, None) == -1
    assert L.sdr_filter_bank_create(0, R.FILTER_IIR_F32, 4, t, 2, 1, C.byref(h)) == -1  # only through _create_iir
    assert L.sdr_debug_filter_bank_set_iir_shape(None, 0, 0) == -1
    assert L.sdr_debug_filter_bank_redo_count(None, None) == -1


def _iir_exe(tmp_dir):
    from rtlsdrdiags_b200 import _build
    _build.build()
    exe = os.path.join(str(tmp_dir), "iir_main")
    pkg = os.path.join(ROOT, "rtlsdrdiags_b200")
    subprocess.run(["g++", "-O2", "-std=c++11", "-I", HOST, "-o", exe, os.path.join(ROOT, "tests", "host", "iir_main.cc"),
                    "-L", pkg, "-lsdr_b200", "-Wl,-rpath," + pkg, "-lm"], check=True)
    return exe


@pytest.fixture(scope="module")
def iir_exe(tmp_path_factory):
    return _iir_exe(tmp_path_factory.mktemp("iir_main"))


def test_drop_in_keeps_the_reference_surface(iir_exe, tmp_path):
    """IirFilter(int, float *, int, float *), filterData, resetFilterState (IirFilter.h); without a
    GPU the bank cannot be created and the driver says so."""
    h = open(os.path.join(HOST, "B200Filters.h")).read()
    assert "class IirFilter" in h
    assert ("IirFilter(int numberOfNumeratorTaps, float *numeratorTapsPtr, int numberOfDenominatorTaps, "
            "float *denominatorTapsPtr)") in h
    assert "float filterData(float x)" in h and "void resetFilterState(void)" in h
    import torch
    if not torch.cuda.is_available():
        taps = tmp_path / "taps.f32"
        np.array([0.5], dtype=f32).tofile(taps)
        assert subprocess.run([iir_exe, str(taps), str(taps), "block"], input=b"").returncode == 2


# ---------------------------------------------------------------- GPU
@gpu
@pytest.mark.parametrize("b,a", [([1], [0.5]), DC_BLOCK, DEEMPH])
def test_known_answers_on_several_rows(b, a):
    """testIirFilter.cc's filters (b={1}, a={0.5}; b={1,-1}, a={-0.95}) and the de-emphasis taps:
    impulse, step and noise rows at once."""
    rng = np.random.default_rng(1)
    n = 19 + 1000
    imp = np.zeros(n, dtype=f32)
    imp[0] = 1
    x = np.stack([imp, np.ones(n, dtype=f32), rng.standard_normal(n).astype(f32), -imp])
    bank = _bank(4, b, a)
    got = bank.run(x)
    assert got.dtype == f32 and got.shape == x.shape
    assert got.tobytes() == oracle_rows(b, a, x).tobytes()
    assert bank.launch_count == 1 and bank.out_count(77) == 77


@gpu
def test_random_filters_two_calls():
    """nb 1..64, na 1..8, poles inside the unit circle, 1..40 rows, up to ~9000 samples cut in two
    calls; plus marginal / unstable filters (|a0| >= 1) on short inputs whose outputs stay finite."""
    rng = np.random.default_rng(77)
    ref = O.ref("radiodiags")
    cases = []
    for trial in range(24):
        nb, na = int(rng.integers(1, 65)), int(rng.integers(1, 9))
        if trial < 8:
            nb = [1, 2, 3, 64, 5, 2, 1, 63][trial]
        b = (rng.standard_normal(nb) / np.sqrt(nb)).astype(f32)
        cases.append((b, stable_denominator(rng, na, rng.choice([0.5, 0.9, 0.99])), int(rng.integers(1, 9000)), 1000.0))
    cases += [(np.array([1], f32), np.array([-1], f32), 700, 1.0),                  # accumulator
              (np.array([0.5, 0.25], f32), np.array([-1.01], f32), 400, 1.0),       # slowly growing
              (np.array([1], f32), np.array([1.0, 0.0], f32), 600, 1.0),            # y[n] = x - y[n-2]
              (np.array([0.3, -0.2, 0.1], f32), np.array([1.5, -0.5, 0.2], f32), 120, 1.0)]
    for i, (b, a, n, amp) in enumerate(cases):
        rows = int(rng.integers(1, 41))
        x = (rng.standard_normal((rows, n)) * amp).astype(f32)
        bank = _bank(rows, b, a)
        if i % 3 == 1:
            bank.debug_set_iir_shape(8)        # segmented, the bank's own warm-up
        elif i % 3 == 2:
            bank.debug_set_iir_shape(4, 64)    # segmented, a warm-up too short to merge
        cut = int(rng.integers(0, n + 1))
        got = np.concatenate([bank.run(x[:, :cut]), bank.run(x[:, cut:])], axis=1)
        assert np.isfinite(got).all()
        exp = oracle_rows(b, a, x)
        assert got.tobytes() == exp.tobytes(), (i, b.size, a.size, n)
        if ref is not None and a.size >= 2:   # pins the oldest-slot order against the reference itself
            assert got.tobytes() == np.stack([Iir(b, a, ref=True).run(r) for r in x]).tobytes(), i


@gpu
@pytest.mark.parametrize("b,a", [DC_BLOCK, DEEMPH, ([0.1] * 9, [0.2, -0.1, 0.3])])
def test_stream_cut_into_ragged_calls(b, a):
    rng = np.random.default_rng(5)
    n = 5000
    x = rng.standard_normal((3, n)).astype(f32)
    exp = oracle_rows(b, a, x)
    bank = _bank(3, b, a)
    cuts = [0, 1, 2, 3, 10, 11, 77, 300, 301, n]
    got = np.concatenate([bank.run(x[:, c0:c1]) for c0, c1 in zip(cuts[:-1], cuts[1:])], axis=1)
    assert got.tobytes() == exp.tobytes()
    bank.reset()   # resetFilterState: the same input again gives the same output
    assert bank.run(x).tobytes() == exp.tobytes()


@gpu
@pytest.mark.parametrize("b,a", [DC_BLOCK, DEEMPH])
@pytest.mark.parametrize("signal", ["tone", "noise"])
def test_long_rows_at_the_automatic_shape_merge_without_redo(b, a, signal):
    rows, n = 6, 262144
    t = np.arange(n)
    rng = np.random.default_rng(11)
    if signal == "tone":
        x = np.stack([3000 * np.sin(2 * np.pi * (0.01 + 0.003 * r) * t + r) + 200 for r in range(rows)]).astype(f32)
    else:
        x = (rng.standard_normal((rows, n)) * 1000).astype(f32)
    bank = _bank(rows, b, a)
    got = np.concatenate([bank.run(x[:, :n // 2]), bank.run(x[:, n // 2:])], axis=1)
    assert got.tobytes() == oracle_rows(b, a, x).tobytes()
    assert bank.debug_redo_count() == 0


@gpu
@pytest.mark.parametrize("warm", [0, 5, 40])
def test_forced_redo_is_exact(warm):
    """Warm-ups far too short to merge: every segment but the first of every row is redone."""
    rows, n, S = 5, 8192, 8
    rng = np.random.default_rng(warm)
    x = (rng.standard_normal((rows, n)) * 100).astype(f32)
    bank = _bank(rows, *DEEMPH)
    bank.debug_set_iir_shape(S, warm)
    got = bank.run(x)
    assert got.tobytes() == oracle_rows(*DEEMPH, x).tobytes()
    assert bank.debug_redo_count() >= rows * (S - 1)
    # with a forced shape and the bank's own warm-up, the next call is exact too
    bank.debug_set_iir_shape(S)
    x2 = (rng.standard_normal((rows, n)) * 100).astype(f32)
    exp = np.stack([Iir(*DEEMPH).run(np.concatenate([x[r], x2[r]]))[n:] for r in range(rows)])
    assert bank.run(x2).tobytes() == exp.tobytes()


@gpu
def test_trajectories_that_never_merge():
    """The DC block on a burst followed by exact zeros: y settles on a denormal that 0.95 y rounds
    back to, which a segment started from 0 never reaches (tests/test_gpu_recurrence.py has the same
    case for the engine); and a filter with |a0| >= 1, which runs unsegmented."""
    rows, n = 4, 200000
    rng = np.random.default_rng(9)
    x = np.zeros((rows, n), dtype=f32)
    x[:, :1000] = rng.standard_normal((rows, 1000)) * 1000
    bank = _bank(rows, *DC_BLOCK)
    got = bank.run(x)
    exp = oracle_rows(*DC_BLOCK, x)
    assert exp[:, -1].any() and np.abs(exp[:, -1]).max() < 1e-38   # stuck on a denormal
    assert got.tobytes() == exp.tobytes()
    assert bank.debug_redo_count() > 0
    b, a = [0.5], [-1.0]            # y[n] = 0.5 x + y[n-1]: never decays
    x = np.sign(rng.standard_normal((rows, n))).astype(f32)
    bank = _bank(rows, b, a)
    assert bank.run(x).tobytes() == oracle_rows(b, a, x).tobytes()
    assert bank.debug_redo_count() == 0


@gpu
def test_signed_zeros_and_subnormals():
    """Products that are -0 (b x and a y) and subnormal inputs and states: a kernel that loses the
    numerator's leading `0 +` or flushes denormals to zero differs here."""
    z = np.zeros(64, dtype=f32)
    nz = -z
    tiny = np.array([1e-45, -1e-45, 3e-39, -2e-40, 1e-38, 0, -0.0] * 9, dtype=f32)
    cases = [([-1], [0.5], z), ([1], [-0.5], nz), ([-1, 1], [0.25, -0.5], np.concatenate([z, nz])),
             ([-0.0], [0.5], np.ones(64, f32)), ([1], [-0.0], nz), ([0.5, 0.5], [-0.75], tiny),
             ([1e-3], [-0.99, 0.5], tiny), ([1, -1], [-0.95], tiny)]
    for b, a, x in cases:
        xs = np.stack([x, -x, x[::-1]])
        got = _bank(3, b, a).run(xs)
        assert got.tobytes() == oracle_rows(b, a, xs).tobytes(), (b, a)


@gpu
def test_device_resident_large_bank_is_cut_invariant():
    """4096 rows x 64 Ki samples through the de-emphasis in one call and in three calls at unaligned
    offsets give the same bytes; every 512th row equals the oracle."""
    import torch
    import rtlsdrdiags_b200 as R
    rows, n = 4096, 65536
    g = torch.Generator(device="cuda").manual_seed(3)
    x = (torch.rand((rows, n), device="cuda", generator=g) * 20000 - 10000).contiguous()
    b1 = R.IirFilterBank(rows, *DEEMPH)
    y = torch.zeros((rows, n), device="cuda")
    assert b1.run_device(x.data_ptr(), n, n, y.data_ptr(), n) == n
    b1.sync()
    b2 = R.IirFilterBank(rows, *DEEMPH)
    y2 = torch.zeros((rows, n + 8), device="cuda")
    for c0, c1 in ((0, 1001), (1001, 30002), (30002, n)):
        assert b2.run_device(x.data_ptr() + 4 * c0, n, c1 - c0, y2.data_ptr() + 4 * (c0 + 3), n + 8) == c1 - c0
    b2.sync()
    assert torch.equal(y, y2[:, 3:n + 3])
    xs, ys = x[::512].cpu().numpy(), y[::512].cpu().numpy()
    assert ys.tobytes() == oracle_rows(*DEEMPH, xs).tobytes()


@gpu
def test_iir_bank_refuses_q15_taps():
    import rtlsdrdiags_b200 as R
    bank = _bank(2, *DC_BLOCK)
    q = np.zeros(2, dtype=np.int16)
    assert bank.L.sdr_filter_bank_taps_q15(bank.b, q.ctypes.data_as(C.c_void_p)) == -1
    with pytest.raises(R.SdrError):
        bank.taps_q15()
    with pytest.raises(R.SdrError):
        bank.debug_set_iir_shape(3)   # not a power of two


@gpu
@pytest.mark.parametrize("how", ["block", "sample"])
@pytest.mark.parametrize("b,a", [DC_BLOCK, DEEMPH, ([0.2, -0.1, 0.05, 0.3], [0.1, -0.3, 0.2])])
def test_iir_filter_drop_in(iir_exe, tmp_path, how, b, a):
    """IirFilter (Filters/IirFilter.h) over a one-row bank: three uneven block calls, then
    resetFilterState() and the whole input again; or one filterData(x) per sample."""
    rng = np.random.default_rng(len(b) + len(a))
    bf, af = tmp_path / "b.f32", tmp_path / "a.f32"
    np.asarray(b, dtype=f32).tofile(bf)
    np.asarray(a, dtype=f32).tofile(af)
    n = 3000 if how == "block" else 200
    x = rng.standard_normal(n).astype(f32)
    r = subprocess.run([iir_exe, str(bf), str(af), how], input=x.tobytes(), capture_output=True, timeout=600)
    assert r.returncode == 0, r.stderr.decode()
    got = np.frombuffer(r.stdout, dtype=f32)
    exp = Iir(b, a).run(x)
    assert got.tobytes() == (np.concatenate([exp, exp]) if how == "block" else exp).tobytes()
