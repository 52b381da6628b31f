"""The engine against the UNMODIFIED reference itself: where oracle/_ref holds the reference's own
sources compiled in place (oracle/Makefile), the CUDA output is compared with IqDataProcessor ->
{Am,Fm,WbFm,Ssb}Demodulator directly; elsewhere with the restatement in oracle/sdr_oracle.c and
with the digests of the reference's output in tests/golden/reference_pins_v1.json. All five modes,
noise and modulated carriers, state carried over several blocks, gains, a mode switch and a reset."""
import numpy as np
import pytest

import _oracle as O
import _pins
import _signals as S

pytestmark = pytest.mark.gpu
Chain = O.RefChain if O.ref("radiodiags") is not None else O.OracleChain


def _ref_rows(modes, iq, gains=None):
    rows = []
    for ch, m in enumerate(modes):
        r = Chain()
        r.set_mode(int(m))
        if gains is not None and int(m):
            r.set_gain(O.MODE_TO_KIND[int(m)], float(gains[ch]))
        rows.append(r.accept_u8(iq[ch]))
    return rows


@pytest.mark.parametrize("mode", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("signal", ["noise", "tone"])
def test_modes_match_the_compiled_reference(mode, signal):
    import rtlsdrdiags_b200 as R
    n, nbytes = 16, 4 * 32768
    e = R.Engine(n, 0, 32768)
    e.set_modes(np.full(n, mode, dtype=np.uint8))
    iq = S.noise(n, nbytes, seed=100 + mode) if signal == "noise" else S.tone_bank([mode] * n, nbytes, seed=mode)
    pcm, counts = e.demodulate(iq)
    assert (counts == 512).all()
    _pins.expect("gpu_modes/%d/%s" % (mode, signal), list(pcm), _ref_rows([mode] * n, iq))
    e.close()


def test_long_calls_mixed_bank_gains_switch_and_reset():
    """Sixteen reference blocks per call (the bench's call shape: segmented recurrence, TMA tiles,
    tensor-core stages) against the reference fed the same bytes in 32768-byte blocks."""
    import rtlsdrdiags_b200 as R
    n, blocks = 10, 16
    modes = np.array([1 + ch % 5 for ch in range(n)], dtype=np.uint8)
    gains = [300.0, 20000.0, 30000.0, 150.0, 700.0, 30.0, 5000.0, 90000.0, 300.0, 1.0]
    e = R.Engine(n, 0, blocks * 32768)
    e.set_modes(modes)
    refs = []
    for ch in range(n):
        r = Chain()
        r.set_mode(int(modes[ch]))
        r.set_gain(O.MODE_TO_KIND[int(modes[ch])], gains[ch])
        e.set_gain(ch, R.MODE_TO_KIND[int(modes[ch])], gains[ch])
        refs.append(r)
    iq = S.tone_bank(modes, 3 * blocks * 32768, seed=31)
    iq[5:] = S.noise(n - 5, iq.shape[1], seed=32)
    got, exp = [], []
    for k in range(3):
        piece = np.ascontiguousarray(iq[:, k * blocks * 32768:(k + 1) * blocks * 32768])
        if k == 1:   # switch two channels and reset one demodulator between calls
            e.set_mode(0, 5)
            refs[0].set_mode(5)
            e.set_mode(7, 1)
            refs[7].set_mode(1)
            e.reset(3, R.MODE_TO_KIND[int(modes[3])])
            refs[3].reset(O.MODE_TO_KIND[int(modes[3])])
        e.accept_iq_host(piece)
        pcm, _ = e.get_pcm()
        got.extend(pcm.copy())
        exp.extend(refs[ch].accept_u8(piece[ch]) for ch in range(n))
    _pins.expect("gpu_long_calls", got, exp)
    e.close()
