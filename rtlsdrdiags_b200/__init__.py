"""B200-native IQ->PCM demodulation engine: Python binding of the C ABI in
include/sdr_b200.h (ctypes over rtlsdrdiags_b200/libsdr_b200.so).

The binding is thin on purpose: the product is the CUDA library. There is no
CPU fallback -- importing works anywhere, but creating an Engine without the
compiled library or without a CUDA device raises.
"""
import ctypes as C
import os

import numpy as np

from . import _build

MODE_NONE, MODE_AM, MODE_FM, MODE_WBFM, MODE_LSB, MODE_USB = range(6)
KIND_AM, KIND_FM, KIND_WBFM, KIND_SSB = 1, 2, 3, 4
SCALING_RADIODIAGS, SCALING_RESEARCH = 0, 1
IQ_HOST, IQ_DEVICE, IQ_U8_OFFSET, IQ_S8_ROTATED = 0, 1, 0, 2
MODE_TO_KIND = {MODE_AM: KIND_AM, MODE_FM: KIND_FM, MODE_WBFM: KIND_WBFM,
                MODE_LSB: KIND_SSB, MODE_USB: KIND_SSB}
BLOCK_BYTES = 32768  # the reference's IQ block: 16384 complex samples = 64 ms -> 512 PCM samples

# every symbol include/sdr_b200.h declares
ABI_SYMBOLS = ["sdr_engine_create", "sdr_engine_destroy", "sdr_set_stream", "sdr_set_scaling",
               "sdr_set_mode", "sdr_set_modes", "sdr_set_gain", "sdr_set_gain_all", "sdr_reset",
               "sdr_accept_iq", "sdr_get_pcm", "sdr_pcm_device", "sdr_sync", "sdr_join", "sdr_set_launch_shape",
               "sdr_launch_count", "sdr_state_bytes", "sdr_last_error", "sdr_version", "sdr_set_squelch_threshold",
               "sdr_set_receive_gain_db", "sdr_enable_signal_reports", "sdr_get_signal", "sdr_set_iq_dump",
               "sdr_get_iq_dump", "sdr_iq_dump_device", "sdr_ingest_create", "sdr_ingest_destroy",
               "sdr_ingest_accept", "sdr_ingest_acquire", "sdr_ingest_commit", "sdr_ingest_retire", "sdr_ingest_stats",
               "sdr_bank_create", "sdr_bank_destroy", "sdr_bank_device_count", "sdr_bank_shard", "sdr_bank_set_mode",
               "sdr_bank_set_modes", "sdr_bank_set_gain", "sdr_bank_reset", "sdr_bank_set_squelch_threshold",
               "sdr_bank_acquire", "sdr_bank_commit", "sdr_bank_retire", "sdr_bank_last_error",
               "sdr_filter_bank_create", "sdr_filter_bank_destroy", "sdr_filter_bank_set_stream",
               "sdr_filter_bank_reset", "sdr_filter_bank_out_count", "sdr_filter_bank_run", "sdr_filter_bank_sync",
               "sdr_filter_bank_taps_q15", "sdr_filter_bank_launch_count", "sdr_filter_bank_last_error",
               "sdr_filter_bank_create_iir", "sdr_ingest_retired_signal", "sdr_ingest_retired_iq_dump",
               "sdr_bank_set_receive_gain_db", "sdr_bank_set_iq_dump", "sdr_bank_enable_signal_reports",
               "sdr_bank_retired_signal", "sdr_bank_retired_iq_dump", "sdr_set_squelch_block_bytes",
               "sdr_get_signal_blocks", "sdr_ingest_retired_signal_blocks", "sdr_bank_set_squelch_block_bytes",
               "sdr_bank_retired_signal_blocks"]


class SdrError(RuntimeError):
    pass


_lib = None


def load_library(build_if_missing=True):
    """dlopen libsdr_b200.so (building it in-tree first if it is absent or stale)."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing and _build.is_stale():
        _build.build()
    if not os.path.exists(_build.LIB):
        raise SdrError("libsdr_b200.so is not built (run `python -m rtlsdrdiags_b200._build`); "
                       "there is no CPU fallback")
    L = C.CDLL(os.environ.get("SDR_B200_LIB") or _build.LIB)  # SDR_B200_LIB: an A/B build of the same library
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
    L.sdr_engine_create.argtypes = [u32, i32, u64, C.POINTER(vp)]
    L.sdr_engine_destroy.argtypes = [vp]
    L.sdr_set_stream.argtypes = [vp, vp]
    L.sdr_set_scaling.argtypes = [vp, i32]
    L.sdr_set_mode.argtypes = [vp, u32, i32]
    L.sdr_set_modes.argtypes = [vp, vp]
    L.sdr_set_gain.argtypes = [vp, u32, i32, C.c_float]
    L.sdr_set_gain_all.argtypes = [vp, i32, C.c_float]
    L.sdr_reset.argtypes = [vp, u32, i32]
    L.sdr_accept_iq.argtypes = [vp, vp, u64, u64, u32]
    L.sdr_get_pcm.argtypes = [vp, vp, vp]
    L.sdr_pcm_device.argtypes = [vp, C.POINTER(vp), C.POINTER(u64)]
    L.sdr_sync.argtypes = [vp]
    L.sdr_join.argtypes = [vp]
    L.sdr_set_squelch_threshold.argtypes = [vp, u32, C.c_int32]
    L.sdr_set_receive_gain_db.argtypes = [vp, u32, u32]
    L.sdr_enable_signal_reports.argtypes = [vp, i32]
    L.sdr_get_signal.argtypes = [vp, vp, vp]
    L.sdr_set_squelch_block_bytes.argtypes = [vp, u64]
    L.sdr_get_signal_blocks.argtypes = [vp, vp, vp, C.POINTER(u32)]
    L.sdr_set_iq_dump.argtypes = [vp, u32, i32]
    L.sdr_get_iq_dump.argtypes = [vp, u32, vp, u64, C.POINTER(u64)]
    L.sdr_iq_dump_device.argtypes = [vp, C.POINTER(vp), C.POINTER(u64), C.POINTER(u32)]
    L.sdr_ingest_create.argtypes = [vp, u32, u64, C.POINTER(vp)]
    L.sdr_ingest_destroy.argtypes = [vp]
    L.sdr_ingest_accept.argtypes = [vp, u32, vp, u64, u64, u32]
    L.sdr_ingest_acquire.argtypes = [vp, C.POINTER(vp), C.POINTER(u64)]
    L.sdr_ingest_commit.argtypes = [vp, u32, u64, u32]
    L.sdr_ingest_retire.argtypes = [vp, C.POINTER(u32), C.POINTER(vp), C.POINTER(u32), C.POINTER(vp)]
    L.sdr_ingest_stats.argtypes = [vp, C.POINTER(u32), C.POINTER(u32), C.POINTER(u64), C.POINTER(u32)]
    L.sdr_ingest_retired_signal.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
    L.sdr_ingest_retired_signal_blocks.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(u32)]
    L.sdr_ingest_retired_iq_dump.argtypes = [vp, C.POINTER(vp), C.POINTER(u64), C.POINTER(u64), C.POINTER(vp),
                                             C.POINTER(u32)]
    L.sdr_set_launch_shape.argtypes = [vp, i32, u32, u32]
    L.sdr_launch_count.argtypes = [vp]
    L.sdr_launch_count.restype = u64
    L.sdr_state_bytes.argtypes = [i32]
    L.sdr_last_error.argtypes = [vp]
    L.sdr_last_error.restype = C.c_char_p
    L.sdr_version.restype = C.c_char_p
    # diagnostics, not part of include/sdr_b200.h
    L.sdr_debug_set_dc_shape.argtypes = [vp, u32, u32]
    L.sdr_debug_dc_redo_count.argtypes = [vp, C.POINTER(u32)]
    L.sdr_debug_set_tile_loader.argtypes = [vp, i32]
    L.sdr_debug_set_wbfm_kernel.argtypes = [vp, i32]
    L.sdr_debug_wb_prefilter_counts.argtypes = [vp, C.POINTER(u32), C.POINTER(u32)]
    L.sdr_bank_create.argtypes = [u32, C.POINTER(i32), u32, u64, u32, C.POINTER(vp)]
    L.sdr_bank_destroy.argtypes = [vp]
    L.sdr_bank_device_count.argtypes = [vp]
    L.sdr_bank_device_count.restype = u32
    L.sdr_bank_shard.argtypes = [vp, u32, C.POINTER(i32), C.POINTER(u32), C.POINTER(u32), C.POINTER(vp)]
    L.sdr_bank_set_mode.argtypes = [vp, u32, i32]
    L.sdr_bank_set_modes.argtypes = [vp, vp]
    L.sdr_bank_set_gain.argtypes = [vp, u32, i32, C.c_float]
    L.sdr_bank_reset.argtypes = [vp, u32, i32]
    L.sdr_bank_set_squelch_threshold.argtypes = [vp, u32, C.c_int32]
    L.sdr_bank_set_receive_gain_db.argtypes = [vp, u32, u32]
    L.sdr_bank_set_iq_dump.argtypes = [vp, u32, i32]
    L.sdr_bank_enable_signal_reports.argtypes = [vp, i32]
    L.sdr_bank_retired_signal.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
    L.sdr_bank_set_squelch_block_bytes.argtypes = [vp, u64]
    L.sdr_bank_retired_signal_blocks.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(u32)]
    L.sdr_bank_retired_iq_dump.argtypes = [vp, C.POINTER(vp), C.POINTER(u64), C.POINTER(u64), C.POINTER(vp),
                                           C.POINTER(u32)]
    L.sdr_bank_acquire.argtypes = [vp, C.POINTER(vp), C.POINTER(u64)]
    L.sdr_bank_commit.argtypes = [vp, u32, u64, u32]
    L.sdr_bank_retire.argtypes = [vp, C.POINTER(u32), C.POINTER(vp), C.POINTER(u32), C.POINTER(vp)]
    L.sdr_bank_last_error.argtypes = [vp]
    L.sdr_bank_last_error.restype = C.c_char_p
    L.sdr_filter_bank_create.argtypes = [i32, i32, u32, vp, u32, u32, C.POINTER(vp)]
    L.sdr_filter_bank_destroy.argtypes = [vp]
    L.sdr_filter_bank_set_stream.argtypes = [vp, vp]
    L.sdr_filter_bank_reset.argtypes = [vp]
    L.sdr_filter_bank_out_count.argtypes = [vp, u64]
    L.sdr_filter_bank_out_count.restype = u64
    L.sdr_filter_bank_run.argtypes = [vp, vp, u64, u64, vp, u64, C.POINTER(u64), u32]
    L.sdr_filter_bank_sync.argtypes = [vp]
    L.sdr_filter_bank_taps_q15.argtypes = [vp, vp]
    L.sdr_filter_bank_launch_count.argtypes = [vp]
    L.sdr_filter_bank_launch_count.restype = u64
    L.sdr_filter_bank_last_error.argtypes = [vp]
    L.sdr_filter_bank_last_error.restype = C.c_char_p
    L.sdr_filter_bank_create_iir.argtypes = [i32, u32, vp, u32, vp, u32, C.POINTER(vp)]
    L.sdr_debug_filter_bank_set_iir_shape.argtypes = [vp, u32, u32]
    L.sdr_debug_filter_bank_redo_count.argtypes = [vp, C.POINTER(u32)]
    _lib = L
    return L


def _retired_signal(fn, handle, n, ck):
    """(allowed [n] bool, magnitude [n] uint32) through sdr_ingest_retired_signal / sdr_bank_retired_signal."""
    a, m = C.c_void_p(), C.c_void_p()
    ck(fn(handle, C.byref(a), C.byref(m)))
    allowed = np.frombuffer((C.c_uint8 * n).from_address(a.value), dtype=np.uint8).astype(bool)
    mag = np.frombuffer((C.c_uint32 * n).from_address(m.value), dtype=np.uint32).copy()
    return allowed, mag


def _retired_signal_blocks(fn, handle, n, ck):
    """(allowed [n_blocks][n] bool, magnitude [n_blocks][n] uint32) through sdr_ingest_retired_signal_blocks /
    sdr_bank_retired_signal_blocks."""
    a, m, nb = C.c_void_p(), C.c_void_p(), C.c_uint32()
    ck(fn(handle, C.byref(a), C.byref(m), C.byref(nb)))
    cells = nb.value * n
    allowed = np.frombuffer((C.c_uint8 * cells).from_address(a.value), dtype=np.uint8).astype(bool)
    mag = np.frombuffer((C.c_uint32 * cells).from_address(m.value), dtype=np.uint32).copy()
    return allowed.reshape(nb.value, n), mag.reshape(nb.value, n)


def _retired_iq_dump(fn, handle, ck):
    """{channel: int8 row} through sdr_ingest_retired_iq_dump / sdr_bank_retired_iq_dump (copies)."""
    rows, stride, nb, chans, nr = C.c_void_p(), C.c_uint64(), C.c_uint64(), C.c_void_p(), C.c_uint32()
    ck(fn(handle, C.byref(rows), C.byref(stride), C.byref(nb), C.byref(chans), C.byref(nr)))
    if nr.value == 0:
        return {}
    ch = np.frombuffer((C.c_uint32 * nr.value).from_address(chans.value), dtype=np.uint32)
    buf = np.frombuffer((C.c_int8 * (nr.value * stride.value)).from_address(rows.value), dtype=np.int8)
    buf = buf.reshape(nr.value, stride.value)
    return {int(c): buf[i, :nb.value].copy() for i, c in enumerate(ch)}


class Engine:
    """A bank of `n_channels` radios on one GPU (one IqDataProcessor plus the four
    demodulators per channel in the reference's terms)."""

    def __init__(self, n_channels, device=0, max_bytes_per_channel=BLOCK_BYTES):
        self.L = load_library()
        self.n = int(n_channels)
        self.max_bytes = int(max_bytes_per_channel)
        h = C.c_void_p()
        rc = self.L.sdr_engine_create(self.n, int(device), self.max_bytes, C.byref(h))
        if rc != 0:
            raise SdrError("sdr_engine_create failed (%d): %s" % (rc, self.L.sdr_last_error(None).decode()))
        self.h = h
        self._keep = None
        self.last_samples = 0  # PCM samples per channel produced by the last accept

    def close(self):
        if getattr(self, "h", None):
            self.L.sdr_engine_destroy(self.h)
            self.h = None

    __del__ = close

    def _ck(self, rc):
        if rc != 0:
            raise SdrError("sdr error %d: %s" % (rc, self.L.sdr_last_error(self.h).decode()))

    # ---- control surface (the reference's setters) ----
    def set_stream(self, cuda_stream_handle):
        self._ck(self.L.sdr_set_stream(self.h, C.c_void_p(cuda_stream_handle or 0)))

    def set_scaling(self, scaling):
        self._ck(self.L.sdr_set_scaling(self.h, scaling))

    def set_mode(self, channel, mode):
        self._ck(self.L.sdr_set_mode(self.h, channel, mode))

    def set_modes(self, modes):
        m = np.ascontiguousarray(modes, dtype=np.uint8)
        if m.size != self.n:
            raise SdrError("modes must have one entry per channel")
        self._ck(self.L.sdr_set_modes(self.h, m.ctypes.data_as(C.c_void_p)))

    def set_gain(self, channel, kind, gain):
        self._ck(self.L.sdr_set_gain(self.h, channel, kind, float(gain)))

    def set_gain_all(self, kind, gain):
        self._ck(self.L.sdr_set_gain_all(self.h, kind, float(gain)))

    def reset(self, channel, kind):
        self._ck(self.L.sdr_reset(self.h, channel, kind))

    def set_squelch_threshold(self, channel, dbfs):
        self._ck(self.L.sdr_set_squelch_threshold(self.h, channel, int(dbfs)))

    def set_receive_gain_db(self, channel, gain_db):
        self._ck(self.L.sdr_set_receive_gain_db(self.h, channel, int(gain_db)))

    def enable_signal_reports(self, on=True):
        self._ck(self.L.sdr_enable_signal_reports(self.h, int(bool(on))))

    def get_signal(self):
        """(allowed [n] bool, magnitude [n] uint32) of the last accept. Synchronises."""
        a = np.empty(self.n, dtype=np.uint8)
        m = np.empty(self.n, dtype=np.uint32)
        self._ck(self.L.sdr_get_signal(self.h, a.ctypes.data_as(C.c_void_p), m.ctypes.data_as(C.c_void_p)))
        return a.astype(bool), m

    def set_squelch_block_bytes(self, block_bytes):
        """Length in bytes of the block the squelch judges (the reference's acceptIqData length, 32768);
        0 = one decision per call. From the next call on."""
        self._ck(self.L.sdr_set_squelch_block_bytes(self.h, int(block_bytes)))

    def get_signal_blocks(self):
        """(allowed [n_blocks][n] bool, magnitude [n_blocks][n] uint32) of every squelch block of the last
        accept. Synchronises."""
        nb = C.c_uint32()
        self._ck(self.L.sdr_get_signal_blocks(self.h, None, None, C.byref(nb)))
        a = np.empty((nb.value, self.n), dtype=np.uint8)
        m = np.empty((nb.value, self.n), dtype=np.uint32)
        self._ck(self.L.sdr_get_signal_blocks(self.h, a.ctypes.data_as(C.c_void_p), m.ctypes.data_as(C.c_void_p),
                                              C.byref(nb)))
        return a.astype(bool), m

    def set_iq_dump(self, channel, on=True):
        """IqDataProcessor::enableIqDump / disableIqDump for one channel of the bank."""
        self._ck(self.L.sdr_set_iq_dump(self.h, channel, int(bool(on))))

    def get_iq_dump(self, channel):
        """The last accept's block of `channel` as the reference hands it to UdpClient::sendData
        (signed, Fs/4-rotated int8). Synchronises."""
        n = C.c_uint64()
        self._ck(self.L.sdr_get_iq_dump(self.h, channel, None, C.c_uint64(0), C.byref(n)))
        out = np.empty(n.value, dtype=np.int8)
        self._ck(self.L.sdr_get_iq_dump(self.h, channel, out.ctypes.data_as(C.c_void_p), C.c_uint64(out.size),
                                        C.byref(n)))
        return out

    def set_launch_shape(self, kind, channels_per_cta=0, threads=0):
        self._ck(self.L.sdr_set_launch_shape(self.h, kind, channels_per_cta, threads))

    # ---- data path ----
    def accept_iq_host(self, iq, fmt=IQ_U8_OFFSET):
        """iq: numpy [n_channels][bytes] uint8 or int8 in host memory (pinned or not)."""
        a = np.ascontiguousarray(iq)
        if a.ndim != 2 or a.shape[0] != self.n or a.itemsize != 1:
            raise SdrError("iq must be [n_channels][bytes] of 1-byte samples")
        self._keep = a  # the copy is asynchronous
        self._ck(self.L.sdr_accept_iq(self.h, a.ctypes.data_as(C.c_void_p), a.shape[1], a.strides[0],
                                      IQ_HOST | fmt))
        self.last_samples = a.shape[1] // 64

    def accept_iq_ptr(self, ptr, bytes_per_channel, channel_stride, flags):
        self._ck(self.L.sdr_accept_iq(self.h, C.c_void_p(ptr), bytes_per_channel, channel_stride, flags))
        self.last_samples = bytes_per_channel // 64

    def accept_iq_device(self, iq_tensor, fmt=IQ_U8_OFFSET):
        """iq_tensor: torch uint8/int8 CUDA tensor [n_channels][bytes], row-contiguous."""
        if iq_tensor.dim() != 2 or iq_tensor.shape[0] != self.n or iq_tensor.stride(1) != 1:
            raise SdrError("iq tensor must be [n_channels][bytes] with unit inner stride")
        self.accept_iq_ptr(iq_tensor.data_ptr(), iq_tensor.shape[1], iq_tensor.stride(0), IQ_DEVICE | fmt)

    def get_pcm(self, out=None):
        """Returns (pcm [n_channels][samples] int16, counts [n_channels] uint32). Synchronises."""
        samples = self.last_samples
        if out is None:
            out = np.empty((self.n, samples), dtype=np.int16)
        counts = np.empty(self.n, dtype=np.uint32)
        self._ck(self.L.sdr_get_pcm(self.h, out.ctypes.data_as(C.c_void_p), counts.ctypes.data_as(C.c_void_p)))
        return out, counts

    def get_pcm_ptr(self, host_ptr):
        self._ck(self.L.sdr_get_pcm(self.h, C.c_void_p(host_ptr), None))

    def pcm_device(self):
        p, s = C.c_void_p(), C.c_uint64()
        self._ck(self.L.sdr_pcm_device(self.h, C.byref(p), C.byref(s)))
        return p.value, s.value

    def sync(self):
        self._ck(self.L.sdr_sync(self.h))

    def join(self):
        """Make the engine's stream wait for its internal second stream (no host blocking)."""
        self._ck(self.L.sdr_join(self.h))

    @property
    def launch_count(self):
        return int(self.L.sdr_launch_count(self.h))

    # ---- diagnostics (tests, tuning) ----
    def debug_set_dc_shape(self, seg_count=0, warm_rows=32):
        """Segmentation of the AM/SSB recurrence kernel: seg_count 0 = per call; warm_rows = rows of
        32 PCM samples a segment warms up on."""
        self._ck(self.L.sdr_debug_set_dc_shape(self.h, int(seg_count), int(warm_rows)))

    def debug_set_tile_loader(self, loader=True):
        """AM/SSB FIR kernel: full tiles by TMA (cp.async.bulk.tensor; True / 1 = default depth, 2..4 =
        that many slot buffers per warp) or by cp.async (False / 0)."""
        self._ck(self.L.sdr_debug_set_tile_loader(self.h, int(loader)))

    def debug_set_wbfm_kernel(self, generation=0):
        """WBFM kernel generation: 0 = default, 1 = table in global memory, 2 = table in shared memory with
        one channel per worker warp, 3 = two channels per worker warp, 4 = the pre-filter on the tcgen05
        tensor cores (geometry of 2 or 3 by bank size; 5 / 6 force two / one channel(s) per warp); + 16 = 2 or 3
        with the pre-filter on the legacy mma.sync path."""
        self._ck(self.L.sdr_debug_set_wbfm_kernel(self.h, int(generation)))

    def debug_wb_prefilter_counts(self):
        """(tensor-core, CUDA-core) counts of WBFM (half-)tiles by where their pre-filter ran, since the
        first call of this method (which switches the counting on)."""
        a, b = C.c_uint32(), C.c_uint32()
        self._ck(self.L.sdr_debug_wb_prefilter_counts(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def debug_dc_redo_count(self):
        """Segments the recurrence kernel had to redo serially since the engine was created."""
        n = C.c_uint32()
        self._ck(self.L.sdr_debug_dc_redo_count(self.h, C.byref(n)))
        return n.value

    def demodulate(self, iq, fmt=IQ_U8_OFFSET):
        """Convenience: one accept + get_pcm on host arrays. Long streams are cut into
        max_bytes_per_channel pieces; state carries across pieces and calls."""
        a = np.ascontiguousarray(iq)
        total = a.shape[1]
        outs = []
        for off in range(0, total, self.max_bytes):
            piece = np.ascontiguousarray(a[:, off:off + self.max_bytes])
            self.accept_iq_host(piece, fmt)
            pcm, counts = self.get_pcm()
            outs.append(pcm)
        return np.concatenate(outs, axis=1), counts


class Ingest:
    """The bank's DataConsumer (DataConsumer.cc:220-352): a ring of pinned ticks whose
    host->device copy, demodulation and PCM read-back overlap. Ticks retire in order."""

    def __init__(self, engine, n_slots=3, block_bytes=BLOCK_BYTES):
        self.e = engine
        self.L = engine.L
        self.block_bytes = int(block_bytes)
        q = C.c_void_p()
        engine._ck(self.L.sdr_ingest_create(engine.h, int(n_slots), self.block_bytes, C.byref(q)))
        self.q = q

    def close(self):
        if getattr(self, "q", None) and getattr(self.e, "h", None):
            self.L.sdr_ingest_destroy(self.q)
        self.q = None

    __del__ = close

    def accept(self, timestamp, iq, fmt=IQ_U8_OFFSET):
        """DataConsumer::acceptData for the whole bank: iq is [n_channels][bytes]."""
        a = np.ascontiguousarray(iq)
        if a.ndim != 2 or a.shape[0] != self.e.n or a.itemsize != 1:
            raise SdrError("iq must be [n_channels][bytes] of 1-byte items")
        self.e._ck(self.L.sdr_ingest_accept(self.q, int(timestamp) & 0xFFFFFFFF, a.ctypes.data_as(C.c_void_p),
                                            a.shape[1], a.strides[0], fmt))

    def acquire(self):
        """The next free slot as a writable [n_channels][block_bytes] uint8 view of pinned memory."""
        p, stride = C.c_void_p(), C.c_uint64()
        self.e._ck(self.L.sdr_ingest_acquire(self.q, C.byref(p), C.byref(stride)))
        buf = (C.c_uint8 * (self.e.n * stride.value)).from_address(p.value)
        return np.frombuffer(buf, dtype=np.uint8).reshape(self.e.n, stride.value)

    def commit(self, timestamp, bytes_per_channel=None, fmt=IQ_U8_OFFSET):
        self.e._ck(self.L.sdr_ingest_commit(self.q, int(timestamp) & 0xFFFFFFFF,
                                            self.block_bytes if bytes_per_channel is None else int(bytes_per_channel),
                                            fmt))

    def retire(self, copy=True):
        """(timestamp, pcm [n_channels][samples], counts [n_channels]) of the oldest tick in flight."""
        ts, samples, p, c = C.c_uint32(), C.c_uint32(), C.c_void_p(), C.c_void_p()
        self.e._ck(self.L.sdr_ingest_retire(self.q, C.byref(ts), C.byref(p), C.byref(samples), C.byref(c)))
        n = self.e.n
        pcm = np.frombuffer((C.c_int16 * (n * samples.value)).from_address(p.value), dtype=np.int16)
        counts = np.frombuffer((C.c_uint32 * n).from_address(c.value), dtype=np.uint32)
        pcm = pcm.reshape(n, samples.value)
        return ts.value, (pcm.copy() if copy else pcm), (counts.copy() if copy else counts)

    def retired_signal(self):
        """(allowed [n] bool, magnitude [n] uint32) of the last retired tick: the signal-state and
        signal-magnitude reports (IqDataProcessor.cc:771-790). Raises if that tick ran no squelch."""
        return _retired_signal(self.L.sdr_ingest_retired_signal, self.q, self.e.n, self.e._ck)

    def retired_signal_blocks(self):
        """(allowed [n_blocks][n] bool, magnitude [n_blocks][n] uint32) of every squelch block of the last
        retired tick. Raises if that tick ran no squelch."""
        return _retired_signal_blocks(self.L.sdr_ingest_retired_signal_blocks, self.q, self.e.n, self.e._ck)

    def retired_iq_dump(self):
        """{channel: int8 array} of the last retired tick's IQ dump (IqDataProcessor.cc:756-760)."""
        return _retired_iq_dump(self.L.sdr_ingest_retired_iq_dump, self.q, self.e._ck)

    def stats(self):
        ts, short, ticks, fl = C.c_uint32(), C.c_uint32(), C.c_uint64(), C.c_uint32()
        self.e._ck(self.L.sdr_ingest_stats(self.q, C.byref(ts), C.byref(short), C.byref(ticks), C.byref(fl)))
        return {"last_timestamp": ts.value, "short_blocks": short.value, "ticks": ticks.value,
                "in_flight": fl.value}


class Bank:
    """n_channels radios over several GPUs of one box (sdr_bank_*): contiguous channel shards, one
    pinned tick array and one pinned PCM array per slot shared by all devices."""

    def __init__(self, n_channels, devices, block_bytes=BLOCK_BYTES, n_slots=3):
        self.L = load_library()
        self.n, self.block_bytes = int(n_channels), int(block_bytes)
        devs = (C.c_int * len(devices))(*[int(d) for d in devices])
        b = C.c_void_p()
        rc = self.L.sdr_bank_create(self.n, devs, len(devices), self.block_bytes, int(n_slots), C.byref(b))
        if rc != 0:
            raise SdrError("sdr_bank_create failed (%d): %s" % (rc, self.L.sdr_bank_last_error(None).decode()))
        self.b = b

    def close(self):
        if getattr(self, "b", None):
            self.L.sdr_bank_destroy(self.b)
            self.b = None

    __del__ = close

    def _ck(self, rc):
        if rc != 0:
            raise SdrError("sdr error %d: %s" % (rc, self.L.sdr_bank_last_error(self.b).decode()))

    def shards(self):
        """[(device, first_channel, n_channels)] per shard."""
        out = []
        for i in range(self.L.sdr_bank_device_count(self.b)):
            d, f, n = C.c_int(), C.c_uint32(), C.c_uint32()
            self._ck(self.L.sdr_bank_shard(self.b, i, C.byref(d), C.byref(f), C.byref(n), None))
            out.append((d.value, f.value, n.value))
        return out

    def set_mode(self, channel, mode):
        self._ck(self.L.sdr_bank_set_mode(self.b, channel, mode))

    def set_modes(self, modes):
        m = np.ascontiguousarray(modes, dtype=np.uint8)
        if m.size != self.n:
            raise SdrError("modes must have one entry per channel")
        self._ck(self.L.sdr_bank_set_modes(self.b, m.ctypes.data_as(C.c_void_p)))

    def set_gain(self, channel, kind, gain):
        self._ck(self.L.sdr_bank_set_gain(self.b, channel, kind, float(gain)))

    def reset(self, channel, kind):
        self._ck(self.L.sdr_bank_reset(self.b, channel, kind))

    def set_squelch_threshold(self, channel, dbfs):
        self._ck(self.L.sdr_bank_set_squelch_threshold(self.b, channel, int(dbfs)))

    def set_receive_gain_db(self, channel, gain_db):
        self._ck(self.L.sdr_bank_set_receive_gain_db(self.b, channel, int(gain_db)))

    def enable_signal_reports(self, on=True):
        self._ck(self.L.sdr_bank_enable_signal_reports(self.b, int(bool(on))))

    def set_iq_dump(self, channel, on=True):
        self._ck(self.L.sdr_bank_set_iq_dump(self.b, channel, int(bool(on))))

    def retired_signal(self):
        """(allowed [n] bool, magnitude [n] uint32) of the last retired tick, gathered over all shards.
        Raises unless every shard ran the squelch for that tick."""
        return _retired_signal(self.L.sdr_bank_retired_signal, self.b, self.n, self._ck)

    def set_squelch_block_bytes(self, block_bytes):
        """Engine.set_squelch_block_bytes on every shard."""
        self._ck(self.L.sdr_bank_set_squelch_block_bytes(self.b, int(block_bytes)))

    def retired_signal_blocks(self):
        """(allowed [n_blocks][n] bool, magnitude [n_blocks][n] uint32) of every squelch block of the last
        retired tick, gathered over all shards."""
        return _retired_signal_blocks(self.L.sdr_bank_retired_signal_blocks, self.b, self.n, self._ck)

    def retired_iq_dump(self):
        """{global channel: int8 array} of the last retired tick's IQ dump."""
        return _retired_iq_dump(self.L.sdr_bank_retired_iq_dump, self.b, self._ck)

    def acquire(self):
        """The next free tick as a writable [n_channels][block_bytes] uint8 view of pinned memory."""
        p, stride = C.c_void_p(), C.c_uint64()
        self._ck(self.L.sdr_bank_acquire(self.b, C.byref(p), C.byref(stride)))
        buf = (C.c_uint8 * (self.n * stride.value)).from_address(p.value)
        return np.frombuffer(buf, dtype=np.uint8).reshape(self.n, stride.value)

    def commit(self, timestamp, bytes_per_channel=None, fmt=IQ_U8_OFFSET):
        self._ck(self.L.sdr_bank_commit(self.b, int(timestamp) & 0xFFFFFFFF,
                                        self.block_bytes if bytes_per_channel is None else int(bytes_per_channel), fmt))

    def retire(self, copy=True):
        """(timestamp, pcm [n_channels][samples], counts [n_channels]) of the oldest tick in flight."""
        ts, samples, p, c = C.c_uint32(), C.c_uint32(), C.c_void_p(), C.c_void_p()
        self._ck(self.L.sdr_bank_retire(self.b, C.byref(ts), C.byref(p), C.byref(samples), C.byref(c)))
        pcm = np.frombuffer((C.c_int16 * (self.n * samples.value)).from_address(p.value), dtype=np.int16)
        counts = np.frombuffer((C.c_uint32 * self.n).from_address(c.value), dtype=np.uint32)
        pcm = pcm.reshape(self.n, samples.value)
        return ts.value, (pcm.copy() if copy else pcm), (counts.copy() if copy else counts)


FILTER_DECIMATOR_F32, FILTER_INTERPOLATOR_F32, FILTER_DECIMATOR_I16, FILTER_INTERPOLATOR_I16 = 1, 2, 3, 4
FILTER_IIR_F32 = 5


class FilterBank:
    """`n_rows` independent Decimator / Interpolator / Decimator_int16 / Interpolator_int16
    objects with the same taps on one GPU (Filters/Decimator.cc, Filters/Interpolator.cc,
    Filters/Int16/*.cc); factor 1 makes a decimator the plain FirFilter / FirFilter_int16."""

    def __init__(self, kind, n_rows, taps, factor, device=0):
        self.L = load_library()
        self.kind, self.rows, self.factor = int(kind), int(n_rows), int(factor)
        self.dtype = np.float32 if kind in (FILTER_DECIMATOR_F32, FILTER_INTERPOLATOR_F32) else np.int16
        h = np.ascontiguousarray(taps, dtype=np.float32)
        self.n_taps = h.size
        b = C.c_void_p()
        rc = self.L.sdr_filter_bank_create(int(device), self.kind, self.rows, h.ctypes.data_as(C.c_void_p), h.size,
                                           self.factor, C.byref(b))
        if rc != 0:
            raise SdrError("sdr_filter_bank_create failed (%d): %s" % (rc, self.L.sdr_filter_bank_last_error(None).decode()))
        self.b = b

    def close(self):
        if getattr(self, "b", None):
            self.L.sdr_filter_bank_destroy(self.b)
            self.b = None

    __del__ = close

    def _ck(self, rc):
        if rc != 0:
            raise SdrError("sdr error %d: %s" % (rc, self.L.sdr_filter_bank_last_error(self.b).decode()))

    def reset(self):
        self._ck(self.L.sdr_filter_bank_reset(self.b))

    def set_stream(self, cuda_stream_handle):
        self._ck(self.L.sdr_filter_bank_set_stream(self.b, C.c_void_p(cuda_stream_handle or 0)))

    def out_count(self, n_in):
        return int(self.L.sdr_filter_bank_out_count(self.b, int(n_in)))

    def taps_q15(self):
        q = np.zeros(self.n_taps, dtype=np.int16)
        self.L.sdr_filter_bank_taps_q15(self.b, q.ctypes.data_as(C.c_void_p))
        return q

    @property
    def launch_count(self):
        return int(self.L.sdr_filter_bank_launch_count(self.b))

    def run(self, x):
        """x: [n_rows][n] host samples; returns [n_rows][n_out]."""
        x = np.ascontiguousarray(x, dtype=self.dtype)
        if x.ndim != 2 or x.shape[0] != self.rows:
            raise SdrError("x must be [n_rows][n]")
        n_out = self.out_count(x.shape[1])
        out = np.zeros((self.rows, max(n_out, 1)), dtype=self.dtype)
        got = C.c_uint64()
        self._ck(self.L.sdr_filter_bank_run(self.b, x.ctypes.data_as(C.c_void_p), x.shape[1], x.shape[1],
                                            out.ctypes.data_as(C.c_void_p), out.shape[1], C.byref(got), IQ_HOST))
        return out[:, :got.value]

    def run_device(self, in_ptr, in_stride, n_in, out_ptr, out_stride):
        """Device pointers (e.g. torch tensors' data_ptr()); queued on the bank's stream."""
        got = C.c_uint64()
        self._ck(self.L.sdr_filter_bank_run(self.b, C.c_void_p(in_ptr), int(in_stride), int(n_in), C.c_void_p(out_ptr),
                                            int(out_stride), C.byref(got), IQ_DEVICE))
        return got.value

    def sync(self):
        self._ck(self.L.sdr_filter_bank_sync(self.b))


class IirFilterBank(FilterBank):
    """`n_rows` independent IirFilter(len(b), b, len(a), a) objects (Filters/IirFilter.cc) on one GPU:
    float in, float out, one output per input; 1 <= len(b) <= 64, 1 <= len(a) <= 8."""

    def __init__(self, n_rows, b, a, device=0):
        self.L = load_library()
        self.kind, self.rows, self.factor = FILTER_IIR_F32, int(n_rows), 1
        self.dtype = np.float32
        hb = np.ascontiguousarray(b, dtype=np.float32)
        ha = np.ascontiguousarray(a, dtype=np.float32)
        self.n_taps = hb.size
        h = C.c_void_p()
        rc = self.L.sdr_filter_bank_create_iir(int(device), self.rows, hb.ctypes.data_as(C.c_void_p), hb.size,
                                               ha.ctypes.data_as(C.c_void_p), ha.size, C.byref(h))
        if rc != 0:
            raise SdrError("sdr_filter_bank_create_iir failed (%d): %s" % (rc, self.L.sdr_filter_bank_last_error(None).decode()))
        self.b = h

    def taps_q15(self):
        raise SdrError("there is no Q15 IirFilter")

    # ---- diagnostics (tests, tuning) ----
    def debug_set_iir_shape(self, seg_count=0, warm=None):
        """Segmentation: seg_count 0 = chosen per call, else a power of two <= 32 segments per row;
        warm = samples a segment warms up on (rounded up to blocks of 32), None = the bank's own."""
        self._ck(self.L.sdr_debug_filter_bank_set_iir_shape(self.b, int(seg_count),
                                                            0xFFFFFFFF if warm is None else int(warm)))

    def debug_redo_count(self):
        """Segments redone serially since the bank was created. Synchronises."""
        n = C.c_uint32()
        self._ck(self.L.sdr_debug_filter_bank_redo_count(self.b, C.byref(n)))
        return n.value
