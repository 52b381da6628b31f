"""Squelch per reference block (sdr_set_squelch_block_bytes): a multi-block call, ring tick or bank
tick is gated, demodulated and reported block by block, as the reference's acceptIqData judges every
block it is handed (IqDataProcessor.cc:722-840, Squelch.cc:227-273). Checked against the same engine
fed one block per call, against the oracle fed block by block, and against the golden vectors."""
import ctypes as C
import os

import numpy as np
import pytest

import _oracle as O

pytestmark = pytest.mark.gpu

SDR_E_ARG, SDR_E_EMPTY = -1, -6
THRESHOLDS = [-200, -30, -20, -15, -12, -9, -6, -3]
GAINS = [0, 0, 5, 0, 3, 0, 0, 10]
# per-block amplitudes: loud blocks between quiet ones, so gates open, hold for the one-block tail
# and close again inside a call
SCHEDULE = [1.0, 60.0, 2.0, 1.0, 12.0, 30.0, 0.5, 0.5, 90.0, 4.0, 1.0, 40.0, 2.0, 1.0, 70.0, 1.0, 0.5, 25.0, 3.0,
            1.0, 50.0, 1.0, 8.0]


def _stream(rng, n, n_blocks, block, fmt, last=None):
    """n channels of n_blocks blocks following SCHEDULE, the channels' amplitudes spread 0.5x..1.5x;
    `last` bytes for the final block. u8 offset-binary or s8 rotated bytes, as uint8."""
    blocks = []
    for k in range(n_blocks):
        amps = SCHEDULE[k % len(SCHEDULE)] * (0.5 + np.arange(n) / n)
        nb = block if (last is None or k + 1 < n_blocks) else last
        x = np.asarray(amps)[:, None] * rng.standard_normal((n, nb))
        if fmt == 0:
            blocks.append(np.clip(np.round(128 + x), 0, 255).astype(np.uint8))
        else:
            blocks.append(np.clip(np.round(x), -128, 127).astype(np.int8).view(np.uint8))
    return np.ascontiguousarray(np.concatenate(blocks, axis=1))


def _configure(e, chains, n, gains=True):
    for ch in range(n):
        thr, g = THRESHOLDS[ch % 8], (GAINS[ch % 8] if gains else 0)
        e.set_squelch_threshold(ch, thr)
        e.set_receive_gain_db(ch, g)
        for c in chains:
            c[ch].set_threshold(thr)
            c[ch].set_rx_gain(g)


def _oracle_call(chains, iq, block):
    """Feed each channel's chain the call block by block (block 0: as one): (pcm per channel, gates
    [B][n], magnitudes [B][n])."""
    n, nbytes = iq.shape
    block = block or nbytes
    pcm, allowed, mag = [[] for _ in range(n)], [], []
    for off in range(0, nbytes, block):
        a_row, m_row = [], []
        for ch in range(n):
            pcm[ch].append(chains[ch].accept_u8(iq[ch, off:off + block]))
            a, m = chains[ch].signal()
            a_row.append(a)
            m_row.append(m)
        allowed.append(a_row)
        mag.append(m_row)
    return [np.concatenate(p) for p in pcm], np.array(allowed), np.array(mag, dtype=np.uint32)


def _check(what, pcm, counts, want):
    for ch, w in enumerate(want):
        assert counts[ch] == w.size, "%s channel %d: count %d vs %d" % (what, ch, counts[ch], w.size)
        if w.size:
            assert np.array_equal(pcm[ch][:counts[ch]], w), "%s channel %d" % (what, ch)


def _chains(modes):
    out = []
    for m in modes:
        c = O.OracleChain()
        c.set_mode(int(m))
        out.append(c)
    return out


@pytest.mark.parametrize("fmt", [0, 2], ids=["u8_offset", "s8_rotated"])
def test_same_stream_two_ways(fmt):
    """Per-block mode fed calls of 1, 3 and 16 blocks and one with a trailing 4096-byte block equals
    today's mode fed the same stream one block per call: compacted PCM, counts, every block's gate and
    magnitude, and get_signal of the last block."""
    import rtlsdrdiags_b200 as R
    n, block = 30, 32768
    rng = np.random.default_rng(21 + fmt)
    modes = np.array([ch % 6 for ch in range(n)], dtype=np.uint8)
    a = R.Engine(n, 0, 16 * block)
    b = R.Engine(n, 0, block)
    for e in (a, b):
        e.set_modes(modes)
        for ch in range(n):
            e.set_squelch_threshold(ch, THRESHOLDS[ch % 8] if ch % 5 else -11)
            e.set_receive_gain_db(ch, GAINS[(ch + 3) % 8])
    a.set_squelch_block_bytes(block)
    calls = [(1, None), (3, None), (16, None), (3, 4096)]
    flips = 0
    for i, (nb, last) in enumerate(calls):
        iq = _stream(rng, n, nb, block, fmt, last)
        a.accept_iq_host(iq, fmt)
        pcm, counts = a.get_pcm()
        allowed, mag = a.get_signal_blocks()
        assert allowed.shape == (nb, n)
        want_pcm = [[] for _ in range(n)]
        for k, off in enumerate(range(0, iq.shape[1], block)):
            b.accept_iq_host(np.ascontiguousarray(iq[:, off:off + block]), fmt)
            bp, bc = b.get_pcm()
            ba, bm = b.get_signal()
            assert np.array_equal(allowed[k], ba), "call %d block %d gates" % (i, k)
            assert np.array_equal(mag[k], bm), "call %d block %d magnitudes" % (i, k)
            for ch in range(n):
                want_pcm[ch].append(bp[ch, :bc[ch]])
        flips += int((allowed[1:] != allowed[:-1]).sum())
        _check("call %d" % i, pcm, counts, [np.concatenate(w) for w in want_pcm])
        la, lm = a.get_signal()
        assert np.array_equal(la, ba) and np.array_equal(lm, bm)
    assert flips > 20  # gates did change inside calls


def test_against_oracle_block_by_block():
    """Multi-block calls against OracleChain fed block by block, and against the compiled reference
    fed its 32768-byte reads where oracle/_ref is built."""
    import rtlsdrdiags_b200 as R
    n, block = 24, 32768
    rng = np.random.default_rng(7)
    modes = np.array([ch % 6 for ch in range(n)], dtype=np.uint8)
    e = R.Engine(n, 0, 6 * block)
    e.set_modes(modes)
    e.set_squelch_block_bytes(block)
    chains = _chains(modes)
    try:
        refs = []
        for m in modes:
            r = O.RefChain()
            r.set_mode(int(m))
            refs.append(r)
    except Exception:
        refs = None
    # the reference's receive gain is process-wide: keep it at 0 here
    _configure(e, [chains] + ([refs] if refs else []), n, gains=False)
    stream, got = [], [[] for _ in range(n)]
    for i, (nb, last) in enumerate([(4, None), (6, None), (2, 6336)]):
        iq = _stream(rng, n, nb, block, 0, last)
        stream.append(iq)
        e.accept_iq_host(iq)
        pcm, counts = e.get_pcm()
        allowed, mag = e.get_signal_blocks()
        want, wa, wm = _oracle_call(chains, iq, block)
        _check("call %d" % i, pcm, counts, want)
        assert np.array_equal(allowed, wa) and np.array_equal(mag, wm), "call %d reports" % i
        for ch in range(n):
            got[ch].append(pcm[ch, :counts[ch]])
    if refs:
        full = np.concatenate(stream, axis=1)
        for ch in range(n):
            assert np.array_equal(np.concatenate(got[ch]), refs[ch].accept_u8(full[ch], block=block)), ch


def test_golden_vectors_in_blocks():
    """The golden squelch vectors (12 blocks of 4096 bytes, 7 configurations) as one 49152-byte call
    with the squelch block at 4096, and as calls of 5 + 7 blocks."""
    import rtlsdrdiags_b200 as R
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_squelch_v1.npz"))
    n = len(g["cfg"])
    stream = np.ascontiguousarray(np.broadcast_to(np.concatenate(list(g["blocks"])), (n, 12 * 4096)))
    for cuts in ([12], [5, 7]):
        e = R.Engine(n, 0, 12 * 4096)
        e.set_modes(np.full(n, 2, dtype=np.uint8))
        e.set_squelch_block_bytes(4096)
        for i, (thr, gain) in enumerate(g["cfg"]):
            e.set_squelch_threshold(i, int(thr))
            e.set_receive_gain_db(i, int(gain))
        out, allowed, mag, counts = [[] for _ in range(n)], [], [], []
        first = 0
        for nb in cuts:
            e.accept_iq_host(np.ascontiguousarray(stream[:, first * 4096:(first + nb) * 4096]))
            pcm, c = e.get_pcm()
            a, m = e.get_signal_blocks()
            allowed.append(a)
            mag.append(m)
            for i in range(n):
                out[i].append(pcm[i, :c[i]])
            counts.append(c)
            first += nb
        allowed, mag = np.concatenate(allowed).T, np.concatenate(mag).T
        assert np.array_equal(allowed.astype(np.uint8), g["allowed"]), cuts
        assert np.array_equal(mag, g["magnitude"]), cuts
        # per call: the sum of the golden per-block counts of its blocks
        first = 0
        for c, nb in zip(counts, cuts):
            assert np.array_equal(c, g["counts"][:, first:first + nb].sum(axis=1)), cuts
            first += nb
        for i in range(n):
            assert np.array_equal(np.concatenate(out[i]), g["pcm_%d" % i]), (cuts, i)


def test_setting_and_arming_change_between_calls():
    """The setting switched 0 -> 32768 -> 8192 -> 0 between calls, the squelch armed and disarmed
    mid-run, and reports-only mode: per-block magnitudes, nothing gated, one demodulation pass."""
    import rtlsdrdiags_b200 as R
    n, call = 12, 4 * 32768
    rng = np.random.default_rng(33)
    modes = np.array([1 + ch % 5 for ch in range(n)], dtype=np.uint8)
    e = R.Engine(n, 0, call)
    e.set_modes(modes)
    chains = _chains(modes)
    armed = False

    def arm(on):
        for ch in range(n):
            thr = THRESHOLDS[ch % 8] if on else -200
            e.set_squelch_threshold(ch, thr)
            chains[ch].set_threshold(thr)

    steps = [(0, True), (32768, True), (32768, False), (8192, True), (8192, True), (32768, "reports"),
             (0, "reports"), (0, True), (8192, False), (32768, True)]
    for i, (setting, mode) in enumerate(steps):
        e.set_squelch_block_bytes(setting)
        if mode == "reports":
            arm(False)
            e.enable_signal_reports(True)
        elif mode != armed:
            e.enable_signal_reports(False)
            arm(mode)
        armed = mode if mode != "reports" else False
        iq = _stream(rng, n, 4, 32768, 0)
        before = e.launch_count
        e.accept_iq_host(iq)
        launches = e.launch_count - before
        pcm, counts = e.get_pcm()
        want, wa, wm = _oracle_call(chains, iq, setting)
        _check("step %d" % i, pcm, counts, want)
        if mode is False:
            with pytest.raises(R.SdrError):
                e.get_signal_blocks()
            assert launches == 6  # one pass: AM and SSB FIR + recurrence, NBFM, WBFM
            continue
        allowed, mag = e.get_signal_blocks()
        assert np.array_equal(allowed, wa) and np.array_equal(mag, wm), "step %d reports" % i
        blocks = call // setting if setting else 1
        assert allowed.shape[0] == blocks
        if mode == "reports":
            assert allowed.all()
        if mode == "reports" or blocks == 1:
            assert launches == 7  # squelch + one pass
        else:
            assert launches == 1 + 6 * blocks + 1  # squelch + a pass per block + compaction


@pytest.mark.parametrize("n_slots", [2, 3, 8])
def test_ingest_ring_blocks(n_slots):
    """4-block ticks through rings of depth 2, 3 and 8: every retired tick's per-block reports, PCM and
    counts against the oracle, with the setting changed between commits while ticks are in flight."""
    import rtlsdrdiags_b200 as R
    n, sq, tick, T = 24, 4096, 4 * 4096, 12
    rng = np.random.default_rng(40 + n_slots)
    modes = np.array([ch % 6 for ch in range(n)], dtype=np.uint8)
    e = R.Engine(n, 0, tick)
    e.set_modes(modes)
    q = R.Ingest(e, n_slots, tick)
    chains = _chains(modes)
    _configure(e, [chains], n)
    settings = {0: sq, 4: 8192, 6: 0, 8: sq, 10: 16384}
    expected, retired = [], 0

    def retire():
        nonlocal retired
        ts, pcm, counts = q.retire()
        assert ts == retired
        want, wa, wm = expected[retired]
        _check("tick %d" % retired, pcm, counts, want)
        a, m = q.retired_signal_blocks()
        assert np.array_equal(a, wa) and np.array_equal(m, wm), "tick %d reports" % retired
        la, lm = q.retired_signal()
        assert np.array_equal(la, wa[-1]) and np.array_equal(lm, wm[-1])
        retired += 1

    setting = 0
    for t in range(T):
        setting = settings.get(t, setting)
        e.set_squelch_block_bytes(setting)
        iq = _stream(rng, n, 4, sq, 0)
        expected.append(_oracle_call(chains, iq, setting))
        if t >= n_slots - 1:
            retire()
        q.accept(t, iq)
    while retired < T:
        retire()


def test_bank_blocks_over_all_devices():
    """Per-block reports gathered in global channel order and compacted PCM, with the channels whose
    gates flip straddling the shard boundaries."""
    import torch
    import rtlsdrdiags_b200 as R
    devs = list(range(torch.cuda.device_count()))
    n, sq, tick = 8 * len(devs) + 3, 8192, 4 * 8192
    rng = np.random.default_rng(55)
    modes = np.array([1 + ch % 5 for ch in range(n)], dtype=np.uint8)
    b = R.Bank(n, devs, tick, n_slots=3)
    b.set_modes(modes)
    b.set_squelch_block_bytes(sq)
    chains = _chains(modes)
    for ch in range(n):
        thr = THRESHOLDS[ch % 8]
        b.set_squelch_threshold(ch, thr)
        chains[ch].set_threshold(thr)
    expected = []
    for t in range(6):
        iq = _stream(rng, n, 4, sq, 0)
        expected.append(_oracle_call(chains, iq, sq))
        b.acquire()[:] = iq
        b.commit(t)
        if t >= 1:
            ts, pcm, counts = b.retire()
            want, wa, wm = expected[ts]
            _check("tick %d" % ts, pcm, counts, want)
            a, m = b.retired_signal_blocks()
            assert np.array_equal(a, wa) and np.array_equal(m, wm), "tick %d reports" % ts
            la, lm = b.retired_signal()
            assert np.array_equal(la, wa[-1]) and np.array_equal(lm, wm[-1])
    ts, pcm, counts = b.retire()
    _check("tick %d" % ts, pcm, counts, expected[ts][0])


def test_error_codes():
    import rtlsdrdiags_b200 as R
    L = R.load_library()
    e = R.Engine(4, 0, 16384)
    for bad in (1024, 3000, 2048 * 3 + 64, 32768):
        assert L.sdr_set_squelch_block_bytes(e.h, bad) == SDR_E_ARG, bad
    assert L.sdr_set_squelch_block_bytes(None, 2048) == SDR_E_ARG
    assert L.sdr_set_squelch_block_bytes(e.h, 16384) == 0
    nb = C.c_uint32()
    assert L.sdr_get_signal_blocks(e.h, None, None, C.byref(nb)) == SDR_E_ARG  # before any call
    e.set_modes(np.full(4, 1, dtype=np.uint8))
    e.accept_iq_host(np.full((4, 16384), 128, dtype=np.uint8))
    assert L.sdr_get_signal_blocks(e.h, None, None, C.byref(nb)) == SDR_E_ARG  # the call ran no squelch
    q = R.Ingest(e, 2, 16384)
    a, m = C.c_void_p(), C.c_void_p()
    assert L.sdr_ingest_retired_signal_blocks(q.q, C.byref(a), C.byref(m), C.byref(nb)) == SDR_E_EMPTY
    q.accept(0, np.full((4, 16384), 128, dtype=np.uint8))
    q.retire()
    assert L.sdr_ingest_retired_signal_blocks(q.q, C.byref(a), C.byref(m), C.byref(nb)) == SDR_E_ARG
    e.set_squelch_block_bytes(2048)
    e.enable_signal_reports(True)
    q.accept(1, np.full((4, 16384), 128, dtype=np.uint8))
    q.retire()
    assert L.sdr_ingest_retired_signal_blocks(q.q, C.byref(a), C.byref(m), C.byref(nb)) == 0 and nb.value == 8
    q.close()
    b = R.Bank(6, [0], 8192, n_slots=2)
    assert L.sdr_bank_retired_signal_blocks(b.b, C.byref(a), C.byref(m), C.byref(nb)) == SDR_E_EMPTY
    assert L.sdr_bank_set_squelch_block_bytes(b.b, 4096 + 64) == SDR_E_ARG
    assert L.sdr_bank_set_squelch_block_bytes(b.b, 16384) == SDR_E_ARG
    b.acquire()[:] = 128
    b.commit(0)
    b.retire()
    assert L.sdr_bank_retired_signal_blocks(b.b, C.byref(a), C.byref(m), C.byref(nb)) == SDR_E_ARG  # no squelch
