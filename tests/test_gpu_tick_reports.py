"""Per-tick signal reports and IQ dump through the ingest ring and the multi-device bank: every
retired tick hands back its own gate, mean magnitude (IqDataProcessor.cc:771-790) and dumped
blocks (IqDataProcessor.cc:756-760), however many newer ticks are in flight, checked against the
oracle tick by tick."""
import ctypes as C
import os

import numpy as np
import pytest

import _oracle as O

pytestmark = pytest.mark.gpu

SDR_E_ARG, SDR_E_EMPTY = -1, -6
THRESHOLDS = [-200, -30, -20, -15, -12, -9, -6, -3]
GAINS = [0, 0, 5, 0, 3, 0, 0, 10]


def _block(rng, n, amps, nbytes):
    """One block per channel: gaussian noise of the given per-channel amplitude around 128."""
    x = 128 + np.asarray(amps, dtype=np.float64)[:, None] * rng.standard_normal((n, nbytes))
    return np.clip(np.round(x), 0, 255).astype(np.uint8)


def _devices():
    import torch
    return list(range(torch.cuda.device_count()))


class _Radios:
    """The oracle's chains for a bank of radios, plus the per-tick expectations computed at commit."""

    def __init__(self, modes):
        self.chains = []
        for m in modes:
            c = O.OracleChain()
            c.set_mode(int(m))
            self.chains.append(c)

    def tick(self, iq, nbytes):
        pcm, allowed, mag = [], [], []
        for ch, c in enumerate(self.chains):
            pcm.append(c.accept_u8(iq[ch, :nbytes]))
            a, m = c.signal()
            allowed.append(a)
            mag.append(m)
        return pcm, np.array(allowed), np.array(mag, dtype=np.uint32)


def _check_pcm(what, pcm, counts, want):
    for ch, w in enumerate(want):
        assert counts[ch] == w.size, "%s channel %d: count %d vs %d" % (what, ch, counts[ch], w.size)
        if w.size:
            assert np.array_equal(pcm[ch][:counts[ch]], w), "%s channel %d" % (what, ch)


@pytest.mark.parametrize("n_slots,lag", [(2, 0), (2, 1), (3, 0), (3, 1), (3, 2), (8, 0), (8, 1), (8, 7)])
def test_ring_reports_every_tick(n_slots, lag):
    """Retiring lag ticks behind the newest commit (the ring full at lag = n_slots - 1), each tick's
    gate, magnitudes, counts and PCM are its own, through short ticks and setters that change
    between commits while ticks are in flight."""
    import rtlsdrdiags_b200 as R
    n, block, T = 24, 8192, 14
    rng = np.random.default_rng(100 + 10 * n_slots + lag)
    modes = np.array([ch % 6 for ch in range(n)], dtype=np.uint8)
    e = R.Engine(n, 0, block)
    e.set_modes(modes)
    q = R.Ingest(e, n_slots, block)
    radios = _Radios(modes)
    schedule = [1.0, 60.0, 2.0, 1.0, 12.0, 30.0, 0.5, 0.5, 90.0, 4.0, 1.0, 40.0, 2.0, 1.0]
    sizes = [block] * T
    sizes[3], sizes[8], sizes[10] = 4096, block - 64, 4096
    expected, ran = [], []
    retired = 0

    def retire():
        nonlocal retired
        ts, pcm, counts = q.retire()
        assert ts == 500 + retired
        want_pcm, want_allowed, want_mag = expected[retired]
        _check_pcm("tick %d" % retired, pcm, counts, want_pcm)
        if ran[retired]:
            allowed, mag = q.retired_signal()
            assert np.array_equal(allowed, want_allowed), "tick %d gate" % retired
            assert np.array_equal(mag, want_mag), "tick %d magnitude" % retired
        else:
            with pytest.raises(R.SdrError):
                q.retired_signal()
        retired += 1

    squelch_runs = False
    for t in range(T):
        if t == 2:                      # reports on: the squelch runs from this tick on
            e.enable_signal_reports(True)
            squelch_runs = True
        if t == 4:                      # per-channel thresholds and tuner gains
            for ch in range(n):
                thr, g = THRESHOLDS[ch % 8], GAINS[ch % 8]
                e.set_squelch_threshold(ch, thr)
                e.set_receive_gain_db(ch, g)
                radios.chains[ch].set_threshold(thr)
                radios.chains[ch].set_rx_gain(g)
        if t == 7:                      # one threshold change with ticks in flight
            for ch in (2, 9, 17):
                e.set_squelch_threshold(ch, -25)
                radios.chains[ch].set_threshold(-25)
        if t == 9:                      # one gain change with ticks in flight
            for ch in (4, 13):
                e.set_receive_gain_db(ch, 20)
                radios.chains[ch].set_rx_gain(20)
        if t == 12:                     # disarmed, reports off: no squelch for the last ticks
            e.enable_signal_reports(False)
            for ch in range(n):
                e.set_squelch_threshold(ch, -200)
                radios.chains[ch].set_threshold(-200)
            squelch_runs = False
        amps = schedule[t] * (0.5 + np.arange(n) / n)
        iq = _block(rng, n, amps, block)
        expected.append(radios.tick(iq, sizes[t]))
        ran.append(squelch_runs)
        if t % 2:
            q.accept(500 + t, iq[:, :sizes[t]])
        else:
            q.acquire()[:, :sizes[t]] = iq[:, :sizes[t]]
            q.commit(500 + t, sizes[t])
        if t >= lag:
            retire()
    while retired < T:
        retire()
    # the schedule really moves the gate: some ticks open, some closed
    assert any(not a.all() for (_, a, _), r in zip(expected, ran) if r)


def test_ring_golden_vectors_depth_3():
    """golden_squelch_v1.npz's seven configurations as seven channels fed through a 3-slot ring,
    retired two ticks behind: decisions, magnitudes, counts and PCM as the compiled reference gave."""
    import rtlsdrdiags_b200 as R
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_squelch_v1.npz"))
    n = len(g["cfg"])
    blocks = g["blocks"]
    e = R.Engine(n, 0, blocks.shape[1])
    e.set_modes(np.full(n, 2, dtype=np.uint8))
    for i, (thr, gain) in enumerate(g["cfg"]):
        e.set_squelch_threshold(i, int(thr))
        e.set_receive_gain_db(i, int(gain))
    q = R.Ingest(e, 3, blocks.shape[1])
    out = [[] for _ in range(n)]
    retired = 0

    def retire():
        nonlocal retired
        ts, pcm, counts = q.retire()
        assert ts == retired
        allowed, mag = q.retired_signal()
        assert np.array_equal(allowed.astype(np.uint8), g["allowed"][:, retired]), retired
        assert np.array_equal(mag, g["magnitude"][:, retired]), retired
        assert np.array_equal(counts, g["counts"][:, retired]), retired
        for i in range(n):
            out[i].append(pcm[i][:counts[i]])
        retired += 1

    for b, blk in enumerate(blocks):
        q.accept(b, np.ascontiguousarray(np.broadcast_to(blk, (n, blk.size))))
        if b >= 2:
            retire()
    while retired < len(blocks):
        retire()
    for i in range(n):
        assert np.array_equal(np.concatenate(out[i]), g["pcm_%d" % i])


@pytest.mark.parametrize("fmt", ["u8", "s8"])
def test_ring_iq_dump_every_tick(fmt):
    """A dumped subset toggled between commits while ticks are in flight, a squelched channel
    among them: each retired tick's rows, channels and byte count are that tick's."""
    import rtlsdrdiags_b200 as R
    n, block, T = 10, 8192, 8
    rng = np.random.default_rng(31 if fmt == "u8" else 32)
    modes = np.array([ch % 6 for ch in range(n)], dtype=np.uint8)
    e = R.Engine(n, 0, block)
    e.set_modes(modes)
    e.set_squelch_threshold(2, 0)       # never opens on this noise: squelched, yet dumped
    q = R.Ingest(e, 3, block)
    sizes = [block, 4096, block, block - 64, block, 4096, block, block]
    plan = {0: {1, 2, 5}, 2: {2, 5, 9}, 4: set(), 5: {0, 2}, 7: set(range(n))}
    on = set()
    expected = []
    retired = 0

    def retire():
        nonlocal retired
        _, _, counts = q.retire()
        assert counts[2] == 0
        want_rows, want_bytes = expected[retired]
        got = q.retired_iq_dump()
        assert sorted(got) == sorted(want_rows), "tick %d channels" % retired
        for ch, row in got.items():
            assert row.size == want_bytes, "tick %d channel %d" % (retired, ch)
            assert np.array_equal(row, want_rows[ch]), "tick %d channel %d" % (retired, ch)
        retired += 1

    for t in range(T):
        if t in plan:
            for ch in range(n):
                e.set_iq_dump(ch, ch in plan[t])
            on = plan[t]
        u8 = _block(rng, n, [30.0] * n, block)
        nb = sizes[t]
        if fmt == "u8":
            rows = {ch: O.front_end(u8[ch, :nb]) for ch in sorted(on)}
            q.accept(t, u8[:, :nb])
        else:
            s8 = np.stack([O.front_end(u8[ch, :nb]) for ch in range(n)])
            rows = {ch: s8[ch].copy() for ch in sorted(on)}
            q.accept(t, s8, R.IQ_S8_ROTATED)
        expected.append((rows, nb))
        if t >= 2:
            retire()
    while retired < T:
        retire()
    # the raw ABI: channels ascending, rows block_bytes apart, n_bytes of the retired tick
    rows, stride, nb, chans, nr = C.c_void_p(), C.c_uint64(), C.c_uint64(), C.c_void_p(), C.c_uint32()
    assert e.L.sdr_ingest_retired_iq_dump(q.q, C.byref(rows), C.byref(stride), C.byref(nb), C.byref(chans),
                                          C.byref(nr)) == 0
    assert (nr.value, stride.value, nb.value) == (n, block, sizes[-1])
    assert list(np.frombuffer((C.c_uint32 * n).from_address(chans.value), dtype=np.uint32)) == list(range(n))


@pytest.mark.parametrize("n", [7, 203])
def test_bank_reports_and_dump_over_all_devices(n):
    """The bank gathers every shard's gate and magnitudes into one [n_channels] array per tick and
    its dump rows in global channel order; dumped channels straddle shard boundaries, and some ticks
    leave a shard without any."""
    import rtlsdrdiags_b200 as R
    devs = _devices()[: max(1, min(len(_devices()), n))]
    block, T = 8192, 9
    b = R.Bank(n, devs, block, n_slots=3)
    first = [s[1] for s in b.shards()]
    modes = np.array([ch % 6 for ch in range(n)], dtype=np.uint8)
    b.set_modes(modes)
    radios = _Radios(modes)
    rng = np.random.default_rng(n)
    sizes = [block] * T
    sizes[4], sizes[7] = 4096, block - 64
    if len(first) > 1:                  # around the first boundary, then only shard 1's rows
        straddle = {0, first[1] - 1, first[1]} | ({first[2] - 1, first[2]} if len(first) > 2 else set())
        later = {first[1], first[1] + 1 if first[1] + 1 < n else first[1]}
    else:
        straddle, later = {0, n // 2, n - 1}, {n - 1}
    plan = {0: straddle, 3: set(), 5: later}
    schedule = [20.0, 1.0, 60.0, 2.0, 1.0, 30.0, 0.5, 90.0, 1.0]
    expected, ran = [], []
    retired = 0
    on, squelch_runs = set(), False

    def retire():
        nonlocal retired
        ts, pcm, counts = b.retire()
        assert ts == retired
        want_pcm, want_allowed, want_mag, want_rows, nb = expected[retired]
        _check_pcm("tick %d" % retired, pcm, counts, want_pcm)
        if ran[retired]:
            allowed, mag = b.retired_signal()
            assert np.array_equal(allowed, want_allowed), "tick %d gate" % retired
            assert np.array_equal(mag, want_mag), "tick %d magnitude" % retired
        else:
            with pytest.raises(R.SdrError):
                b.retired_signal()
        got = b.retired_iq_dump()
        assert list(got) == sorted(want_rows), "tick %d channels" % retired
        for ch, row in got.items():
            assert row.size == nb and np.array_equal(row, want_rows[ch]), "tick %d channel %d" % (retired, ch)
        retired += 1

    for t in range(T):
        if t == 1:
            b.enable_signal_reports(True)
            squelch_runs = True
        if t == 2:
            for ch in range(n):
                thr, g = THRESHOLDS[ch % 8], GAINS[ch % 8]
                b.set_squelch_threshold(ch, thr)
                b.set_receive_gain_db(ch, g)
                radios.chains[ch].set_threshold(thr)
                radios.chains[ch].set_rx_gain(g)
        if t == 5:                      # changes while ticks are in flight
            b.set_squelch_threshold(n - 1, -25)
            radios.chains[n - 1].set_threshold(-25)
            b.set_receive_gain_db(1, 20)
            radios.chains[1].set_rx_gain(20)
        if t in plan:
            for ch in on - plan[t]:
                b.set_iq_dump(ch, False)
            for ch in plan[t] - on:
                b.set_iq_dump(ch, True)
            on = plan[t]
        amps = schedule[t] * (0.5 + np.arange(n) / n)
        iq = _block(rng, n, amps, block)
        nb = sizes[t]
        pcm, allowed, mag = radios.tick(iq, nb)
        expected.append((pcm, allowed, mag, {ch: O.front_end(iq[ch, :nb]) for ch in on}, nb))
        ran.append(squelch_runs)
        b.acquire()[:, :nb] = iq[:, :nb]
        b.commit(t, nb)
        if t >= 2:
            retire()
    while retired < T:
        retire()
    b.close()


def test_retired_error_codes():
    """SDR_E_EMPTY before any retire and once the retired tick's slot is committed again; SDR_E_ARG
    for a tick without a squelch; a tick without a dump has zero rows."""
    import rtlsdrdiags_b200 as R
    n, block = 4, 4096
    e = R.Engine(n, 0, block)
    e.set_modes(np.full(n, 2, dtype=np.uint8))
    q = R.Ingest(e, 2, block)
    L = e.L
    a, m = C.c_void_p(), C.c_void_p()
    rows, stride, nb, chans, nr = C.c_void_p(), C.c_uint64(), C.c_uint64(), C.c_void_p(), C.c_uint32()

    def dump_rc(handle, fn):
        return fn(handle, C.byref(rows), C.byref(stride), C.byref(nb), C.byref(chans), C.byref(nr))

    assert L.sdr_ingest_retired_signal(q.q, C.byref(a), C.byref(m)) == SDR_E_EMPTY
    assert dump_rc(q.q, L.sdr_ingest_retired_iq_dump) == SDR_E_EMPTY
    assert L.sdr_ingest_retired_signal(None, None, None) == SDR_E_ARG
    iq = np.random.default_rng(3).integers(0, 256, size=(n, block), dtype=np.uint8)
    q.accept(1, iq)
    q.retire()
    assert L.sdr_ingest_retired_signal(q.q, C.byref(a), C.byref(m)) == SDR_E_ARG   # no squelch ran
    assert dump_rc(q.q, L.sdr_ingest_retired_iq_dump) == 0
    assert (nr.value, nb.value, rows.value) == (0, block, None)
    assert q.retired_iq_dump() == {}
    e.enable_signal_reports(True)
    q.accept(2, iq)
    q.retire()
    assert L.sdr_ingest_retired_signal(q.q, None, None) == 0
    allowed, mag = q.retired_signal()
    assert allowed.all() and (mag > 0).all()
    q.accept(3, iq)                     # the other slot
    q.accept(4, iq)                     # the retired tick's slot, committed again
    assert L.sdr_ingest_retired_signal(q.q, C.byref(a), C.byref(m)) == SDR_E_EMPTY
    q.retire()
    q.retire()

    b = R.Bank(6, _devices()[:1], block, n_slots=2)
    assert L.sdr_bank_retired_signal(b.b, C.byref(a), C.byref(m)) == SDR_E_EMPTY
    assert dump_rc(b.b, L.sdr_bank_retired_iq_dump) == SDR_E_EMPTY
    b.acquire()[:] = np.random.default_rng(4).integers(0, 256, size=(6, block), dtype=np.uint8)
    b.commit(0)
    b.retire()
    assert L.sdr_bank_retired_signal(b.b, C.byref(a), C.byref(m)) == SDR_E_ARG
    with pytest.raises(R.SdrError):
        b.retired_signal()
    assert b.retired_iq_dump() == {}
    assert L.sdr_bank_set_iq_dump(b.b, 6, 1) == SDR_E_ARG
    assert L.sdr_bank_set_receive_gain_db(b.b, 6, 0) == SDR_E_ARG
    b.close()
