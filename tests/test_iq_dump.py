"""IQ dump / .iq wire format (SURVEY 8f-2): IqDataProcessor.cc:756-760 hands the converted,
Fs/4-rotated block to UdpClient::sendData, which cuts it into datagrams of at most 2048 bytes
(UdpClient.cc:77, 199-231). The compiled reference really sends them here, to a socket on
127.0.0.1; the oracle restates bytes and datagram sizes; the engine emits the same bytes."""
import socket

import numpy as np
import pytest

import _oracle as O
import _pins
import _signals as S

have_ref = O.ref("radiodiags") is not None


def _listener():
    s = socket.socket(socket.AF_INET, socket.SOCK_DGRAM)
    s.setsockopt(socket.SOL_SOCKET, socket.SO_RCVBUF, 1 << 22)
    s.bind(("127.0.0.1", 0))
    s.settimeout(2.0)
    return s, s.getsockname()[1]


def _drain(sock, n):
    return [sock.recv(4096) for _ in range(n)]


@pytest.mark.parametrize("nbytes", [32768, 4096, 5000, 2048, 1000, 8])
def test_oracle_dump_matches_datagrams_the_reference_sends(nbytes):
    u8 = S.noise(1, nbytes, seed=nbytes)[0]
    u8[:16] = [0, 0, 0, 0, 0, 0, 0, 0, 255, 255, 255, 255, 255, 255, 255, 255][:min(16, nbytes)]
    sizes = O.dump_datagrams(nbytes)
    got = [np.array(sizes, dtype=np.int64), O.front_end(u8)]
    if not have_ref:
        _pins.expect("iq_dump_datagrams/%d" % nbytes, got)
        return
    sock, port = _listener()
    try:
        r = O.RefChain(dump_port=port)
        r.set_mode(3)          # WBFM rewrites the buffer after the dump: must not show
        r.set_threshold(0)     # squelched: the dump is sent all the same
        r.set_dump(True)
        r.accept_u8(u8, block=nbytes)
        sent = _drain(sock, len(sizes))
        _pins.expect("iq_dump_datagrams/%d" % nbytes, got,
                     [np.array([len(g) for g in sent], dtype=np.int64), np.frombuffer(b"".join(sent), dtype=np.int8)])
        r.set_dump(False)
        r.accept_u8(u8, block=nbytes)
        sock.settimeout(0.2)
        with pytest.raises(socket.timeout):
            sock.recv(4096)
    finally:
        sock.close()


def test_front_end_is_what_the_signed_entry_consumes():
    """The dump is the .iq format: feeding it to the demodulator entry (accept_s8) gives the
    PCM the u8 entry gives."""
    u8 = S.noise(1, 32768 * 2, seed=5)[0]
    s8 = O.front_end(u8[:32768]), O.front_end(u8[32768:])
    for mode in (1, 2, 3, 4, 5):
        a, b = O.OracleChain(), O.OracleChain()
        a.set_mode(mode)
        exp = np.concatenate([a.accept_u8(u8[:32768]), a.accept_u8(u8[32768:])])
        got = np.concatenate([b.accept_s8(mode, s8[0]), b.accept_s8(mode, s8[1])])
        assert np.array_equal(exp, got)


@pytest.mark.gpu
@pytest.mark.parametrize("nbytes", [32768, 64, 4096 + 64])
def test_engine_dump_matches_oracle(nbytes):
    import rtlsdrdiags_b200 as R
    n = 9
    iq = S.noise(n, nbytes, seed=77)
    iq[0, :16] = 0
    iq[2, :16] = 255
    e = R.Engine(n, 0, 32768)
    e.set_modes(np.array([ch % 6 for ch in range(n)], dtype=np.uint8))
    for ch in (0, 2, 3, 8):
        e.set_iq_dump(ch, True)
    e.set_squelch_threshold(3, 0)   # closed: dumped all the same
    e.accept_iq_host(iq)
    pcm, counts = e.get_pcm()
    assert counts[3] == 0
    for ch in (0, 2, 3, 8):
        assert np.array_equal(e.get_iq_dump(ch), O.front_end(iq[ch])), ch
    with pytest.raises(R.SdrError):
        e.get_iq_dump(1)
    # signed input is passed through unchanged; disabling takes effect at the next call
    e.set_iq_dump(2, False)
    s8 = np.stack([O.front_end(iq[ch]) for ch in range(n)])
    e.accept_iq_host(s8, R.IQ_S8_ROTATED)
    assert np.array_equal(e.get_iq_dump(8), s8[8])
    with pytest.raises(R.SdrError):
        e.get_iq_dump(2)
    # the PCM of the demodulated channels is unaffected by dumping
    for ch in (1, 2, 4, 8):
        c = O.OracleChain()
        c.set_mode(ch % 6)
        assert np.array_equal(pcm[ch][:counts[ch]], c.accept_u8(iq[ch]))
