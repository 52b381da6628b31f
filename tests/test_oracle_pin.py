"""Pins the oracle (oracle/sdr_oracle.c) to the reference.

1. against tests/golden/golden_v1.npz -- outputs the UNMODIFIED reference produced
   when compiled in place (tests/golden/make_golden.py); always runs;
2. against the compiled reference itself (oracle/_ref) on seeded random inputs,
   quirk vectors, gains and ragged blocks -- live where oracle/_ref was built, and
   everywhere against the digests of its output in tests/golden/reference_pins_v1.json;
3. against the md5s of the only IQ capture the reference ships
   (demodulatorResearch/yoyo.iq) -- runs where /root/reference is mounted.
"""
import hashlib
import os

import numpy as np
import pytest

import _oracle as O
import _pins

GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_v1.npz"))
NAMES = {1: "am", 2: "fm", 3: "wbfm", 4: "lsb", 5: "usb"}
have_ref = O.ref("radiodiags") is not None and O.ref("research") is not None
YOYO = "/root/reference/demodulatorResearch/yoyo.iq"


@pytest.mark.parametrize("mode", [1, 2, 3, 4, 5])
def test_oracle_matches_golden_product_path(mode):
    iq = GOLD["iq_u8"]
    exp = GOLD["pcm_" + NAMES[mode]]
    for ch in range(iq.shape[0]):
        c = O.OracleChain()
        c.set_mode(mode)
        assert np.array_equal(c.accept_u8(iq[ch]), exp[ch]), "channel %d" % ch


@pytest.mark.parametrize("mode", [1, 2, 3, 4, 5])
def test_oracle_matches_golden_research_tree(mode):
    iq = GOLD["iq_s8"]
    exp = GOLD["research_" + NAMES[mode]]
    for ch in range(iq.shape[0]):
        c = O.OracleChain(O.VARIANT_RESEARCH)
        assert np.array_equal(c.accept_s8(mode, iq[ch]), exp[ch])


@pytest.mark.parametrize("mode", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("gmul", [1.0, 4.0, 1e6, 0.0])
def test_oracle_matches_compiled_reference_noise_and_quirks(mode, gmul):
    rng = np.random.default_rng(1000 * mode + int(gmul))
    u8 = rng.integers(0, 256, size=32768 * 4, dtype=np.uint8)
    u8[:4096] = 0
    u8[4096:8192] = 255
    u8[8192:12288:2] = 0
    u8[8193:12288:2] = 255
    kind = O.MODE_TO_KIND[mode]
    base = {1: 300.0, 2: 10185.916, 3: 40743.664, 4: 300.0}[kind]
    chains = [O.OracleChain()] + ([O.RefChain()] if have_ref else [])
    for x in chains:
        x.set_mode(mode)
        x.set_gain(kind, base * gmul)
    out = [[x.accept_u8(u8)] for x in chains]
    _pins.expect("noise_and_quirks/%d/%g" % (mode, gmul), out[0], out[1] if have_ref else None)


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_oracle_matches_compiled_reference_ragged_blocks_and_resets(mode):
    rng = np.random.default_rng(mode)
    chains = [O.OracleChain()] + ([O.RefChain()] if have_ref else [])
    out = [[] for _ in chains]
    for x in chains:
        x.set_mode(mode)
    kind = O.MODE_TO_KIND[mode]
    for i, n in enumerate([8, 24, 32768, 1000, 4096 + 8, 16, 2, 32768, 6]):
        u8 = rng.integers(0, 256, size=n, dtype=np.uint8)
        for x, o in zip(chains, out):
            o.append(x.accept_u8(u8))
            if i == 4:
                x.reset(kind)
    _pins.expect("ragged_blocks_and_resets/%d" % mode, out[0], out[1] if have_ref else None)


def test_oracle_mode_switch_keeps_idle_state_like_reference():
    rng = np.random.default_rng(5)
    chains = [O.OracleChain()] + ([O.RefChain()] if have_ref else [])
    out = [[] for _ in chains]
    for mode in [3, 2, 3, 4, 1, 5, 0, 4, 2]:
        u8 = rng.integers(0, 256, size=32768, dtype=np.uint8)
        for x, o in zip(chains, out):
            x.set_mode(mode)
            o.append(x.accept_u8(u8))
    _pins.expect("mode_switch", out[0], out[1] if have_ref else None)


@pytest.mark.parametrize("mode", [1, 2, 3, 4, 5])
def test_oracle_matches_research_tree_direct_entry(mode):
    s8 = np.random.default_rng(70 + mode).integers(-128, 128, size=32768 * 3, dtype=np.int8)
    exp = None
    if have_ref:
        d = O.RefDemod(O.MODE_TO_KIND[mode], "research")
        if mode in (4, 5):
            d.set_lsb(mode == 4)
        exp = [d.accept(s8, block=16384)]
    c = O.OracleChain(O.VARIANT_RESEARCH)
    _pins.expect("research_direct_entry/%d" % mode, [c.accept_s8(mode, s8)], exp)


@pytest.mark.skipif(not os.path.exists(YOYO), reason="reference tree not mounted")
@pytest.mark.parametrize("mode", [1, 2, 3, 4, 5])
def test_oracle_reproduces_yoyo_md5s(mode):
    yoyo = np.fromfile(YOYO, dtype=np.int8)
    assert hashlib.md5(yoyo.tobytes()).hexdigest() == str(GOLD["yoyo_md5_input"])
    c = O.OracleChain(O.VARIANT_RESEARCH)
    got = hashlib.md5(c.accept_s8(mode, yoyo).tobytes()).hexdigest()
    assert got == str(GOLD["yoyo_md5_research_" + NAMES[mode]])
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        "make_golden", os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    c = O.OracleChain()
    c.set_mode(mode)
    got = hashlib.md5(c.accept_u8(mg.unrotate_to_u8(yoyo)).tobytes()).hexdigest()
    assert got == str(GOLD["yoyo_md5_radiodiags_" + NAMES[mode]])


def _amp_block(rng, amp, nbytes):
    return np.clip(np.round(128 + amp * rng.standard_normal(nbytes)), 0, 255).astype(np.uint8)


@pytest.mark.parametrize("threshold,gain", [(-200, 0), (-30, 0), (-20, 0), (-12, 3), (-6, 0), (-25, 10), (0, 0)])
def test_squelch_oracle_matches_compiled_reference(threshold, gain):
    """Squelch::run (Squelch.cc:227-273) through IqDataProcessor: gate, one-block tail,
    tuner gain, the values handed to both signal callbacks, and the PCM that does or does
    not come out -- restatement against the reference compiled in place."""
    rng = np.random.default_rng(abs(threshold) * 7 + gain)
    chains = [O.OracleChain()] + ([O.RefChain()] if have_ref else [])
    out = [[] for _ in chains]
    try:
        for c in chains:
            c.set_mode(2)
            c.set_threshold(threshold)
            c.set_rx_gain(gain)
        seen = set()
        for step, amp in enumerate([0.5, 70.0, 1.0, 0.5, 10.0, 33.0, 0.6, 0.6, 100.0, 3.0, 127.0, 0.0]):
            nbytes = 32768 if step % 3 else 4096
            blk = _amp_block(rng, amp, nbytes)
            for c, o in zip(chains, out):
                o.append(c.accept_u8(blk, block=nbytes) if isinstance(c, O.RefChain) else c.accept_u8(blk))
                o.append(np.array(c.signal(), dtype=np.int64))
            seen.add(bool(out[0][-2].size))
        if threshold in (-30, -20, -12, -25):
            assert seen == {True, False}
        _pins.expect("squelch/%d/%d" % (threshold, gain), out[0], out[1] if have_ref else None)
    finally:
        if have_ref:
            chains[1].set_rx_gain(0)


def test_squelch_db_table_matches_compiled_reference_over_all_magnitudes():
    """Constant-amplitude blocks sweep the detector's magnitude over its whole range, so every
    entry of DbfsCalculator's table (DbfsCalculator.cc:30-50) is exercised."""
    chains = [O.OracleChain()] + ([O.RefChain()] if have_ref else [])
    out = [[] for _ in chains]
    for c in chains:
        c.set_mode(1)
        c.set_threshold(-18)
    for i in range(0, 128, 3):
        for q in (0, i // 2, i):
            blk = np.empty(1024, dtype=np.uint8)
            blk[0::2] = 128 + i
            blk[1::2] = 128 - q
            for c, o in zip(chains, out):
                o.append(c.accept_u8(blk, block=1024) if isinstance(c, O.RefChain) else c.accept_u8(blk))
                o.append(np.array(c.signal(), dtype=np.int64))
    _pins.expect("squelch_db_table", out[0], out[1] if have_ref else None)


SQ = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_squelch_v1.npz"))


@pytest.mark.parametrize("i", range(7))
def test_squelch_oracle_matches_golden(i):
    """tests/golden/golden_squelch_v1.npz: what the compiled reference's squelch decided,
    reported and let through (always runs, also where oracle/_ref is absent)."""
    thr, gain = (int(v) for v in SQ["cfg"][i])
    c = O.OracleChain()
    c.set_mode(2)
    c.set_threshold(thr)
    c.set_rx_gain(gain)
    pcm = []
    for b, blk in enumerate(SQ["blocks"]):
        pcm.append(c.accept_u8(blk))
        assert c.signal() == (bool(SQ["allowed"][i, b]), int(SQ["magnitude"][i, b])), b
        assert pcm[-1].size == SQ["counts"][i, b]
    assert np.array_equal(np.concatenate(pcm), SQ["pcm_%d" % i])
