// Host side of the demodulation engine and its C ABI (include/sdr_b200.h).
//
// One engine owns, for a bank of n_channels radios on one GPU:
//   * per-kind continuation state blobs in HBM ([n_channels][STATE_BYTES] each;
//     the reference keeps four demodulator objects per radio and a mode switch
//     leaves the idle ones untouched, IqDataProcessor.cc:793-835),
//   * per-channel mode / gain / sideband tables, mirrored on the host,
//   * per-kind channel lists (channels bucketed by mode so every CTA is
//     mode-uniform), the two atan2 tables, an IQ staging buffer and the PCM buffer.
// sdr_accept_iq queues one launch per demodulator kind that has channels (AM and SSB: a FIR
// kernel plus a recurrence kernel on a second stream). No CPU path exists.
#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/sdr_b200.h"
#include "sdr_config.h"

namespace {

using namespace sdr;

thread_local std::string g_create_error;

struct Shape { uint32_t G = 0, NT = 0; };  // 0 = choose

}  // namespace

struct sdr_engine {
  int device = 0;
  uint32_t n = 0;
  uint64_t max_bytes = 0;
  int n_sm = 148;
  int smem_optin = 227 * 1024;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  // AM/SSB: the recurrence kernels run on rec_stream, one call behind the FIR kernels on
  // `stream`; the numerators travel through scratch[kind][call index % RING]
  cudaStream_t rec_stream = nullptr;
  // RING: how many calls' numerators / gates exist at once. Call k's recurrence kernel runs beside
  // call k+1's FIR kernel and is a small fraction of its length (segment-parallel, see
  // dc_block_kernel), so call k+2 never waits for it; the third buffer is slack.
  static constexpr int RING_MAX = 3;
  static constexpr int ring = RING_MAX;
  cudaEvent_t ev_fir[RING_MAX] = {}, ev_rec[RING_MAX] = {};
  // bounded run-ahead: a caller that queues calls faster than the GPU retires them is held once
  // RUN_AHEAD calls are in flight (see sdr_accept_iq)
  static constexpr int RUN_AHEAD = 32, PACE = 2 * RUN_AHEAD;
  cudaEvent_t ev_pace[PACE] = {};
  int16_t *d_scratch[5][RING_MAX] = {};
  // AM/SSB FIR kernel: full tiles by TMA (cp.async.bulk.tensor through a tensor map of the caller's
  // IQ array, rebuilt when pointer, stride or length change) or by cp.async
  int tile_loader = 2;  // 0 = cp.async (two slot buffers), 2 / 3 / 4 = TMA with that many slot buffers
  bool stage1_mma = false;  // with TMA: stage 1 of the AM / SSB cascade on the tensor cores (measured slower, see DESIGN.md)
  int wb_kernel = 0;  // 0 = default (SDR_WB_KERNEL, or 4 / 2 by bank size), 1..4 = that generation of the WBFM kernel
  volatile uint32_t *h_wb_clip = nullptr;  // pinned: counters[3] after the last generation-4 launch that has finished
  uint32_t wb_clip_seen = 0;               // its value when last looked at
  uint64_t wb4_units = 0;                  // (half-)tiles per worker warp in the last generation-4 launch
  int wb_clip_hold = 0;                    // calls left on generation 3 because the input clips
  int wb4_geometry = 0;  // generation 4: 0 = by bank size, 1 = two channels per worker warp, 2 = one
  bool wb_count = false;  // sdr_debug_wb_prefilter_counts was called: the kernels count their tiles
  bool wb_prefilter_mma = false;  // generations 2, 3: the pre-filter on the tensor cores (WbMma; measured: no faster)
  int fir_ctas_per_sm = 5;  // __launch_bounds__ of the FIR kernel: 5 or 6 CTAs per SM (it needs 80 registers either way now)
  uint32_t *d_am_tab = nullptr;  // am_mma_table()
  CUtensorMap tmap;
  const void *tmap_iq = nullptr;
  uint64_t tmap_stride = 0, tmap_rows = 0;
  // dc_block_kernel's segmentation (0 = chosen per call) and its redo counter
  uint32_t dc_seg_count = 0, dc_warm_rows = 28;  // 896 steps: beyond the latest merge seen (807)
  uint32_t *d_counters = nullptr;
  // Two counters. seq numbers the public calls: it picks the PCM buffer, the dump / gate /
  // magnitude ring entries and the pace events. pass numbers the demodulation passes: it picks
  // the scratch buffer and the ev_fir / ev_rec entry (par = pass % RING) and gives each pass its
  // call_id. A call is one pass, or one pass per block while the squelch gates block by block
  // (see accept_iq); with the squelch block at 0 the two counters are equal.
  uint64_t seq = 0;        // sdr_accept_iq calls so far
  uint64_t pass = 0;       // demodulation passes so far
  const uint8_t *pass_allowed = nullptr;  // gate row of the pass being queued, or null = all open
  int16_t *pass_pcm = nullptr;            // where the pass being queued writes its PCM columns
  bool rec_pending = false;  // work on rec_stream that `stream` has not waited for yet
  // Mixed banks: the WBFM kernel (one long-lived CTA per SM that leaves issue slots, registers
  // and shared memory unused) runs on its own stream next to the other kinds' kernels
  cudaStream_t wb_stream = nullptr;
  cudaEvent_t ev_in = nullptr, ev_wb = nullptr;
  bool wb_pending = false;   // work on wb_stream that `stream` has not waited for yet
  int scaling = SDR_SCALING_RADIODIAGS;

  // host mirrors (index 1..4 = kind)
  std::vector<uint8_t> mode, lsb;
  std::vector<float> gain[5], scale[5];
  std::vector<uint32_t> list[5];
  bool lists_dirty = true, lsb_dirty = true, scale_dirty[5] = {true, true, true, true, true};

  // device
  uint8_t *d_state[5] = {};
  float *d_scale[5] = {};
  uint32_t *d_list[5] = {};
  uint8_t *d_lsb = nullptr;
  float *d_lut_fm = nullptr, *d_lut_wbfm = nullptr;
  float *d_lut_wbfm_half = nullptr;  // q >= 0 half plane for wbfm_tile2_kernel, [129][256]
  uint32_t *d_fm_tab = nullptr;  // tensor-core tuner tables, fm_mma_table()
  uint32_t *d_wb_tab = nullptr;  // tensor-core WBFM pre-filter table, wb_mma_table()
  uint8_t *d_wb4_tab = nullptr;  // tap matrices of the tcgen05 WBFM pre-filter, wb_umma_table()
  uint8_t *d_iq = nullptr;
  // two PCM buffers, used by alternate calls: the read-back of call k (sdr_get_pcm, the ingest
  // ring's device->host copy) does not hold up the kernels of call k+1
  int16_t *d_pcm2[2] = {nullptr, nullptr};
  uint64_t pcm_stride = 0;
  int16_t *pcm_of(uint64_t call) const { return d_pcm2[call & 1]; }

  // squelch (IqDataProcessor's Squelch object, one per channel)
  std::vector<int32_t> threshold;   // dBFS, -200 = the reference's always-open default
  std::vector<uint32_t> rx_gain_db; // radio_adjustableReceiveGainInDb per radio
  bool squelch_dirty = false, squelch_armed = false, signal_reports = false;
  int32_t *d_threshold = nullptr;
  uint32_t *d_rx_gain = nullptr;
  // squelch block: bytes of the block the squelch judges (the reference's acceptIqData length),
  // 0 = one decision per call
  uint64_t squelch_block = 0;
  uint32_t sig_rows = 1;  // block rows in each entry of d_allowed and d_magnitude
  // gates and mean magnitudes, [RING_MAX][sig_rows][n]: entry call % RING_MAX, row = block
  uint8_t *d_allowed = nullptr;
  uint32_t *d_magnitude = nullptr;
  uint8_t *allowed_of(uint64_t call) const { return d_allowed + (size_t)(call % RING_MAX) * sig_rows * n; }
  uint32_t *magnitude_of(uint64_t call) const { return d_magnitude + (size_t)(call % RING_MAX) * sig_rows * n; }
  uint32_t last_blocks = 1;       // blocks the last call's squelch judged (rows of its entry)
  uint64_t last_block_bytes = 0;  // their length, the last one's excepted
  uint8_t *d_tracking = nullptr;
  int32_t *d_db_table = nullptr;
  bool last_gated = false;  // the last accept ran the squelch kernel with the gate in force
  // blocks were accepted without the squelch kernel after d_tracking came to exist: every one of
  // them passed, so the reference's trackers all stand in `Tracking` (SignalTracker.cc:104-145)
  bool tracking_stale = false;

  // IQ dump (IqDataProcessor::enableIqDump): channels whose converted block is kept
  std::vector<uint8_t> dump_on;
  std::vector<uint32_t> dump_list;
  bool dump_dirty = false;
  uint32_t dump_count = 0;    // channels with dump_on set: the rows the next call dumps
  uint32_t *d_dump_list = nullptr;
  int8_t *d_dump = nullptr;   // [RING_MAX][dump_rows][max_bytes], entry call % RING_MAX
  size_t dump_rows = 0;       // rows each entry of d_dump holds
  uint64_t dump_bytes = 0;    // bytes per channel of the last dump (0 = none)
  int8_t *dump_of(uint64_t call) const { return d_dump + (size_t)(call % RING_MAX) * dump_rows * max_bytes; }
  // the ingest ring's device->host stream, which copies out of d_dump: drained before d_dump is freed
  cudaStream_t dump_reader = nullptr;

  // SDR_TRACE=1: per call [FIR start, FIR end, dc_block start, dc_block end] in globaltimer ns (tools/probe_timeline.py)
  unsigned long long *d_trace = nullptr;
  static constexpr uint64_t TRACE_CALLS = 4096;
  Shape shape[5];
  uint32_t last_samples = 0;  // PCM samples per channel of the last accept
  uint64_t launches = 0;
  std::string err;
  // a call failed after part of its work was queued: events, ring slots and carried state are no
  // longer in step, so every later data-path call returns this error again
  bool poisoned = false;
  std::string poison_text;
};

namespace {

int fail(sdr_engine *e, int code, const char *what, cudaError_t ce = cudaSuccess) {
  char buf[512];
  if (ce != cudaSuccess) snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(ce));
  else snprintf(buf, sizeof buf, "%s", what);
  if (e) e->err = buf;
  else g_create_error = buf;
  return code;
}

#define SDR_CK(e, call)                                                 \
  do {                                                                  \
    cudaError_t _ce = (call);                                           \
    if (_ce != cudaSuccess) return fail((e), SDR_E_CUDA, #call, _ce);   \
  } while (0)

int state_bytes(int kind) {
  switch (kind) {
    case SDR_KIND_AM: return AmSsbTile<false>::STATE_BYTES;
    case SDR_KIND_FM: return FmTile::STATE_BYTES;
    case SDR_KIND_WBFM: return WbTile::STATE_BYTES;
    case SDR_KIND_SSB: return AmSsbTile<true>::STATE_BYTES;
  }
  return -1;
}
int kind_of_mode(int mode) {
  switch (mode) {
    case SDR_MODE_AM: return SDR_KIND_AM;
    case SDR_MODE_FM: return SDR_KIND_FM;
    case SDR_MODE_WBFM: return SDR_KIND_WBFM;
    case SDR_MODE_LSB:
    case SDR_MODE_USB: return SDR_KIND_SSB;
  }
  return 0;
}

// reference constructor defaults: AmDemodulator.cc:102, FmDemodulator.cc:154,
// WbFmDemodulator.cc:173 (research tree: 64000), SsbDemodulator.cc:146
float default_gain(int kind, int scaling) {
  switch (kind) {
    case SDR_KIND_AM: return 300;
    case SDR_KIND_FM: return (float)(64000 / (2 * M_PI));
    case SDR_KIND_WBFM:
      return scaling == SDR_SCALING_RESEARCH ? (float)(64000 / (2 * M_PI)) : (float)(256000 / (2 * M_PI));
    case SDR_KIND_SSB: return 300;
  }
  return 0;
}

// what the kernels multiply by. FM/WBFM: frequencyDeviationToPcm, two float ops
// (FmDemodulator.cc:465-471, WbFmDemodulator.cc:444-450).
float scale_of(int kind, float gain, int scaling) {
  if (kind == SDR_KIND_AM || kind == SDR_KIND_SSB || scaling == SDR_SCALING_RESEARCH) return gain;
  volatile float k = gain / (kind == SDR_KIND_FM ? 15000.0f : 75000.0f);
  k = k * 32767.0f;
  return k;
}

// main stream waits for everything queued on rec_stream
int join_streams(sdr_engine *e) {
  if (e->rec_pending) {
    SDR_CK(e, cudaStreamWaitEvent(e->stream, e->ev_rec[(e->pass + (uint64_t)e->ring - 1) % (uint64_t)e->ring], 0));
    e->rec_pending = false;
  }
  if (e->wb_pending) {
    SDR_CK(e, cudaStreamWaitEvent(e->stream, e->ev_wb, 0));
    e->wb_pending = false;
  }
  return SDR_OK;
}

// The IQ array as the TMA sees it: uint8 [n_channels][rows of 128 bytes][128], of which only the
// rows of FULL tiles (16 rows = 2048 bytes) are ever asked for, so the map never reaches past
// a channel's valid bytes. The boxes are {128, 16, 1} with the hardware's 128-byte swizzle.
typedef CUresult (*TensorMapEncodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                         const cuuint64_t *, const cuuint32_t *, const cuuint32_t *,
                                         CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                         CUtensorMapFloatOOBfill);
int iq_tensor_map(sdr_engine *e, const uint8_t *iq, uint64_t ch_stride, uint32_t n_samples) {
  const uint64_t rows = (uint64_t)(n_samples / TILE) * (TILE_BYTES / 128);
  if (e->tmap_iq == iq && e->tmap_stride == ch_stride && e->tmap_rows == rows) return SDR_OK;
  static TensorMapEncodeTiled encode = nullptr;
  if (!encode) {
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    SDR_CK(e, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr));
    if (!fn || qr != cudaDriverEntryPointSuccess) return fail(e, SDR_E_CUDA, "the driver has no cuTensorMapEncodeTiled");
    encode = (TensorMapEncodeTiled)fn;
  }
  if (rows == 0) {  // no full tile in this call: the kernel issues no TMA; keep any valid map
    memset(&e->tmap, 0, sizeof e->tmap);
  } else {
    const cuuint64_t dims[3] = {128, rows, e->n};
    const cuuint64_t strides[2] = {128, ch_stride};
    const cuuint32_t box[3] = {128, TILE_BYTES / 128, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = encode(&e->tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t *>(iq), dims, strides, box,
                              estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      char msg[96];
      snprintf(msg, sizeof msg, "cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
      return fail(e, SDR_E_CUDA, msg);
    }
  }
  e->tmap_iq = iq;
  e->tmap_stride = ch_stride;
  e->tmap_rows = rows;
  return SDR_OK;
}

// Taps of the tensor-core stage 1 of the AM / SSB kernel (AmSsbTile::stage1_mma): D = A * B with A =
// raw input bytes. A row h, K index kb = 0..63: the raw byte 32 h - 32 + kb of the tile, i.e. sample
// js = floor((kb - 32) / 2) relative to the half-window's first sample, I at even bytes. B[kb][n]:
// column n < 4 gives I' output n of the half-window, n >= 4 gives Q' output n - 4. Output p is
// sum_k q[k] x'[4 p + 3 - k] (Decimator_int16.cc:310-351; AmDemodulator.cc:349-374) where x' is the
// rotated sample (IqDataProcessor.cc:567-611): I' = I0, -Q1, -I2, Q3; Q' = Q0, I1, -Q2, -I3 by
// js mod 4 -- or plain I, Q for input that is already rotated. The taps are doubled (the int8 result
// is then byte 2 of the accumulator, see Doubled in sdr_tile.cuh) and split as 256 * hi + lo with both
// parts int8. The accumulators start at the doubled rounding constant 1 << 15 (lo) and, for u8 input
// (u = s + 128), at -128 * the column sum.
// Layout per format: [lane][12]: words 0-7 the B fragments [hi / lo][k-step][b0, b1] (mma.m16n8k32 B
// fragment: b0 = (k 4tq..4tq+3, column g), b1 = (k 16+4tq.., column g)), words 8-11 the starts of the
// lane's accumulator columns [hi 2tq, hi 2tq+1, lo 2tq, lo 2tq+1].
std::vector<uint32_t> am_mma_table() {
  std::vector<uint32_t> tab(2 * 32 * 12, 0);
  for (int f = 0; f < 2; ++f) {
    int B[64][8] = {};
    for (int kb = 0; kb < 64; ++kb) {
      const int js = (kb - 32) >> 1, c = kb & 1, jm = ((js % 4) + 4) % 4;
      int arm, sign;
      if (f == 0) {
        static const int arm_of[4][2] = {{0, 1}, {1, 0}, {0, 1}, {1, 0}};     // [jm][c]: 0 = I', 1 = Q'
        static const int sign_of[4][2] = {{1, 1}, {1, -1}, {-1, -1}, {-1, 1}};
        arm = arm_of[jm][c];
        sign = sign_of[jm][c];
      } else {
        arm = c;
        sign = 1;
      }
      for (int pp = 0; pp < 4; ++pp) {
        const int k = 4 * pp + 3 - js;
        if (k >= 0 && k < taps::AM1::N) B[kb][4 * arm + pp] = sign * 2 * taps::AM1::tap(k);
      }
    }
    auto part = [](int v, int h) {
      const int lo = ((v + 128) & 255) - 128;
      return h == 0 ? (v - lo) / 256 : lo;
    };
    for (int lane = 0; lane < 32; ++lane) {
      const int g = lane >> 2, tq = lane & 3;
      uint32_t *t = tab.data() + ((size_t)f * 32 + lane) * 12;
      for (int h = 0; h < 2; ++h)
        for (int s2 = 0; s2 < 2; ++s2)
          for (int r = 0; r < 2; ++r) {
            const int k0 = 32 * s2 + 16 * r + 4 * tq;
            uint32_t w = 0;
            for (int b = 0; b < 4; ++b) w |= (uint32_t)(uint8_t)(int8_t)part(B[k0 + b][g], h) << (8 * b);
            t[(h * 2 + s2) * 2 + r] = w;
          }
      for (int i = 0; i < 4; ++i) {
        const int h = i >> 1, col = 2 * tq + (i & 1);
        int sum = 0;
        for (int kb = 0; kb < 64; ++kb) sum += part(B[kb][col], h);
        t[8 + i] = (uint32_t)((h == 1 ? 1 << 15 : 0) - (f == 0 ? 128 * sum : 0));
      }
    }
  }
  return tab;
}

// AM / SSB: FIR kernel on the engine's stream, recurrence kernel on rec_stream.
template <bool SSB>
int launch_amssb(sdr_engine *e, int kind, const uint8_t *iq, uint64_t ch_stride, uint32_t n_samples, int fmt) {
  using T = AmSsbTile<SSB>;
  const uint32_t n_list = (uint32_t)e->list[kind].size();
  if (n_list == 0) return SDR_OK;
  const int par = (int)(e->pass % (uint64_t)e->ring);
  const uint32_t n_tiles = (n_samples + TILE - 1) / TILE;
  if (!e->d_scratch[kind][par]) {
    // every buffer of the ring at the kind's first call: no allocation may fall into a later call
    const size_t max_tiles = (size_t)((e->max_bytes / 2 + TILE - 1) / TILE);
    for (int i = 0; i < e->ring; ++i)
      if (!e->d_scratch[kind][i])
        SDR_CK(e, cudaMalloc(&e->d_scratch[kind][i], (size_t)e->n * max_tiles * 32 * sizeof(int16_t)));
  }
  // The launch's tiles are dealt out in equal shares to 72 (AM) or 48 (SSB) worker warps per SM: 18 or 12 CTAs of 4
  // warps, of which six are resident at a time (80 registers since the window rings) -- three or two full waves.
  // Shares small enough that SMs which also host the previous call's recurrence CTAs simply take fewer of them,
  // large enough (>= 8 tiles) that the warm-up tiles (AM one, SSB two per share) stay small: AM x1024 x 16 blocks
  // 0.1148 ms with 48, 0.1124 with 72, 0.1131 with 96; SSB x8192 0.1251 with 48, 0.1270 with 72
  // (profiles/r02_window_rings.txt; round 1's sweep at 96 registers: profiles/r01v5_am_sweep.txt).
  static const int wps_env = getenv("SDR_AM_WARPS_PER_SM") ? atoi(getenv("SDR_AM_WARPS_PER_SM")) : 0;
  const uint64_t total_tiles = (uint64_t)n_list * n_tiles;
  uint64_t n_warps = (uint64_t)e->n_sm * (wps_env > 0 ? wps_env : (SSB ? 48 : 72));
  // ... and no shorter than 16 tiles: in a small bank (the AM / SSB shares of a mixed bank: 32 tiles per channel and call) a
  // share of 8 spends 1/9 (AM) or 2/10 (SSB) of its work on warm-up tiles. mixed x8192: 0.3388 ms with 8, 0.3175-0.3188
  // with 16, 0.3262 with 24, 0.3190-0.3201 with 32 (profiles/r02_window_rings.txt). NBFM keeps 8: it wants the warps more.
  static const int min_share_env = getenv("SDR_AM_MIN_SHARE") ? atoi(getenv("SDR_AM_MIN_SHARE")) : 0;  // tuning override
  const uint64_t min_share = min_share_env > 0 ? (uint64_t)min_share_env : 16;
  n_warps = std::min<uint64_t>(n_warps, (total_tiles + min_share - 1) / min_share);
  n_warps = std::max<uint64_t>(n_warps, 1);
  LaunchParams p = {};
  p.iq = iq;
  p.ch_stride = ch_stride;
  p.n_samples = n_samples;
  p.fmt = fmt;
  p.chan_ids = e->d_list[kind];
  p.n_list = n_list;
  p.G = 4;
  p.state = e->d_state[kind];
  p.state_stride = (uint32_t)T::STATE_BYTES;
  p.scale = e->d_scale[kind];
  p.lsb = e->d_lsb;
  p.pcm = e->pass_pcm;
  p.pcm_stride = e->pcm_stride;
  p.lut = nullptr;
  p.aux = (uint32_t)n_warps;
  p.call_id = (uint32_t)(e->pass % 0x7fffffffull) + 1;
  p.scratch = e->d_scratch[kind][par];
  p.allowed = e->pass_allowed;
  p.trace = e->d_trace ? e->d_trace + 4 * (e->pass % sdr_engine::TRACE_CALLS) : nullptr;
  const uint32_t grid = (uint32_t)((n_warps + 3) / 4);
  if (e->tile_loader == 0) {
    if (e->fir_ctas_per_sm == 6) amssb_fir_kernel<SSB, false, 2, false, 6><<<grid, 128, 4 * 2 * TILE_BYTES, e->stream>>>(p, e->tmap);
    else amssb_fir_kernel<SSB, false, 2, false><<<grid, 128, 4 * 2 * TILE_BYTES, e->stream>>>(p, e->tmap);
  } else if (e->fir_ctas_per_sm == 6 && !e->stage1_mma) {
    const int rc = iq_tensor_map(e, iq, ch_stride, n_samples);
    if (rc) return rc;
    if (e->tile_loader == 2) amssb_fir_kernel<SSB, true, 2, false, 6><<<grid, 128, 4 * 2 * TILE_BYTES, e->stream>>>(p, e->tmap);
    else amssb_fir_kernel<SSB, true, 4, false, 6><<<grid, 128, 4 * 4 * TILE_BYTES, e->stream>>>(p, e->tmap);
  } else {
    int rc = iq_tensor_map(e, iq, ch_stride, n_samples);
    if (rc) return rc;
    if (e->stage1_mma && !e->d_am_tab) {
      const std::vector<uint32_t> tab = am_mma_table();
      SDR_CK(e, cudaMalloc(&e->d_am_tab, tab.size() * 4));
      SDR_CK(e, cudaMemcpy(e->d_am_tab, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice));
    }
    p.tab = e->d_am_tab;
    const int nst = e->tile_loader;
    const size_t smem = (size_t)4 * nst * TILE_BYTES;
    if (e->stage1_mma) {
      if (nst == 2) amssb_fir_kernel<SSB, true, 2, true><<<grid, 128, smem, e->stream>>>(p, e->tmap);
      else if (nst == 3) amssb_fir_kernel<SSB, true, 3, true><<<grid, 128, smem, e->stream>>>(p, e->tmap);
      else amssb_fir_kernel<SSB, true, 4, true><<<grid, 128, smem, e->stream>>>(p, e->tmap);
    } else {
      if (nst == 2) amssb_fir_kernel<SSB, true, 2, false><<<grid, 128, smem, e->stream>>>(p, e->tmap);
      else if (nst == 3) amssb_fir_kernel<SSB, true, 3, false><<<grid, 128, smem, e->stream>>>(p, e->tmap);
      else amssb_fir_kernel<SSB, true, 4, false><<<grid, 128, smem, e->stream>>>(p, e->tmap);
    }
  }
  SDR_CK(e, cudaGetLastError());
  e->launches++;
  return SDR_OK;
}

// Segmentation of one call's recurrence (dc_block_kernel): rows of 32 PCM samples, segments of
// at least 32 rows (so the warm-up rows, which are read a second time, stay below the segment's
// own), at most 32 segments per channel (the lanes of one warp), none for short calls.
void dc_segments(const sdr_engine *e, uint32_t n_rows, uint32_t *seg_count, uint32_t *seg_rows) {
  uint32_t S = 1;
  if (e->dc_seg_count) {
    S = e->dc_seg_count;
  } else if (n_rows >= 64) {
    while (S < 32 && n_rows / (2 * S) >= 32) S *= 2;
  }
  while (S > 1 && (n_rows + S - 1) / S * (S - 1) >= n_rows) S /= 2;  // no empty segments in the middle
  *seg_count = S;
  *seg_rows = (n_rows + S - 1) / S;
}

int launch_dc_block(sdr_engine *e, int kind, uint32_t n_samples) {
  const uint32_t n_list = (uint32_t)e->list[kind].size();
  if (n_list == 0) return SDR_OK;
  const int par = (int)(e->pass % (uint64_t)e->ring);
  const int nreg = kind == SDR_KIND_SSB ? AmSsbTile<true>::NREG : AmSsbTile<false>::NREG;
  LaunchParams p = {};
  p.n_samples = n_samples;
  p.chan_ids = e->d_list[kind];
  p.n_list = n_list;
  p.state = e->d_state[kind];
  p.state_stride = (uint32_t)state_bytes(kind);
  p.scale = e->d_scale[kind];
  p.pcm = e->pass_pcm;
  p.pcm_stride = e->pcm_stride;
  p.aux = (uint32_t)nreg * 256;  // byte offset of the IIR tail in the state blob (after both carry buffers)
  p.scratch = e->d_scratch[kind][par];
  p.allowed = e->pass_allowed;
  p.trace = e->d_trace ? e->d_trace + 4 * (e->pass % sdr_engine::TRACE_CALLS) + 2 : nullptr;
  dc_segments(e, (n_samples + TILE - 1) / TILE, &p.seg_count, &p.seg_rows);
  p.warm_rows = e->dc_warm_rows;
  p.counters = e->d_counters;
  const uint64_t lanes = (uint64_t)n_list * p.seg_count;
  dc_block_kernel<<<(uint32_t)((lanes + 31) / 32), 64, 0, e->rec_stream>>>(p);
  SDR_CK(e, cudaGetLastError());
  e->launches++;
  return SDR_OK;
}

// Tables of the tensor-core tuner (FmTile::theta_mma): D = A * B with B = raw input bytes.
// A[row][kk]: row p < 8 gives I' output p of a window, row 8 + p gives Q'; kk = 0..127 indexes
// the raw bytes from 64 before the window's first byte to its last (sample j = floor((kk-64)/2),
// I at even bytes). Output p is sum_k q[k] x'[4p + 3 - k] (Decimator_int16.cc:310-351) where x' is
// the rotated sample (IqDataProcessor.cc:567-611): I' = I0, -Q1, -I2, Q3; Q' = Q0, I1, -Q2, -I3
// by j mod 4 -- or plain I, Q for input that is already rotated. Each int16 tap is split as
// 256 * hi + lo with both parts int8. The accumulators start at the rounding constant 1 << 14
// (lo) and, for u8 input (u = s + 128), at -128 * sum of the row.
// Layout per format: nine entries of [lane][4 words]: entries 0-7 the A fragments [hi/lo][k-step],
// entry 8 the starts [hi row g, hi row g+8, lo row g, lo row g+8]; mma.m16n8k32 A fragment: word 0 =
// (row g, k 4tq..4tq+3), 1 = (row g+8, same k), 2 = (row g, k+16), 3 = (row g+8, k+16).
std::vector<uint32_t> fm_mma_table() {
  std::vector<uint32_t> tab(2 * FM_TAB_WORDS_PER_FMT, 0);
  for (int f = 0; f < 2; ++f) {
    int A[16][128] = {};
    for (int kk = 0; kk < 128; ++kk) {
      const int j = (kk - 64) >> 1, c = kk & 1, jm = ((j % 4) + 4) % 4;
      int arm, sign;  // which output arm this byte feeds and with what sign
      if (f == 0) {
        static const int arm_of[4][2] = {{0, 1}, {1, 0}, {0, 1}, {1, 0}};     // [jm][c]: 0 = I', 1 = Q'
        static const int sign_of[4][2] = {{1, 1}, {1, -1}, {-1, -1}, {-1, 1}};
        arm = arm_of[jm][c];
        sign = sign_of[jm][c];
      } else {
        arm = c;
        sign = 1;
      }
      for (int pp = 0; pp < 8; ++pp) {
        const int k = 4 * pp + 3 - j;
        if (k >= 0 && k < taps::FM_TUNER::N) A[8 * arm + pp][kk] = sign * taps::FM_TUNER::tap(k);
      }
    }
    uint32_t *t = tab.data() + (size_t)f * FM_TAB_WORDS_PER_FMT;
    auto part = [](int v, int h) {
      const int lo = ((v + 128) & 255) - 128;
      return h == 0 ? (v - lo) / 256 : lo;
    };
    for (int lane = 0; lane < 32; ++lane) {
      const int g = lane >> 2, tq = lane & 3;
      for (int h = 0; h < 2; ++h)
        for (int s4 = 0; s4 < 4; ++s4)
          for (int r = 0; r < 4; ++r) {
            const int row = g + 8 * (r & 1), k0 = 32 * s4 + 16 * (r >> 1) + 4 * tq;
            uint32_t w = 0;
            for (int b = 0; b < 4; ++b) w |= (uint32_t)(uint8_t)(int8_t)part(A[row][k0 + b], h) << (8 * b);
            t[((h * 4 + s4) * 32 + lane) * 4 + r] = w;
          }
      for (int i = 0; i < 4; ++i) {
        const int h = i >> 1, row = g + 8 * (i & 1);
        int sum = 0;
        for (int kk = 0; kk < 128; ++kk) sum += part(A[row][kk], h);
        int start = (h == 1 ? 1 << 14 : 0) - (f == 0 ? 128 * sum : 0);
        t[(8 * 32 + lane) * 4 + i] = (uint32_t)start;
      }
    }
  }
  return tab;
}

// Table of the tensor-core WBFM pre-filter (WbMma::prefilter): D = A * B with B = raw u8 input bytes.
// A[row][kb]: row o < 8 gives I' output o of an M-tile (eight consecutive samples = one 16-byte granule),
// row 8 + o gives Q'; kb = 0..47 indexes the raw bytes from 32 before the granule's first to its last
// (complex sample c = kb >> 1 counted from 16 before the granule, I at even bytes). Output o is
// sum_k 2 h[k] x'[16 + o - k] (FirFilter_int16.cc:151-213 with the taps doubled, WbTile::Pre2) where x' is the
// rotated sample (IqDataProcessor.cc:567-611): I' = I0, -Q1, -I2, Q3; Q' = Q0, I1, -Q2, -I3 by c mod 4 (a
// granule starts a rotation period). Each tap is split as 256 * hi + lo with both parts int8.
// The accumulators' starts -- the doubled rounding constant 1 << 15 (lo) and, for u = s + 128, -128 * the row
// sum -- ride in the K dimension: the first MMA of an accumulator is an m16n8k32 whose K 0..15 is the granule
// kb 0..15 and whose K 16..31 meets the constant granule C (twelve bytes 255, four bytes 1): start = 255 * (sum
// of the twelve A entries there) + (sum of the last four), every entry an int8.
// Layout: four A fragments of [lane][4 words] (mma.m16n8k32: row g, row g+8, row g k+16, row g+8 k+16; k 4tq..4tq+3):
//   0, 1: hi and lo of [kb 0..15 | start]      2, 3: hi and lo of kb 16..47
// then the four words of C.
std::vector<uint32_t> wb_mma_table() {
  std::vector<uint32_t> tab(WB_TAB_WORDS, 0);
  int A[16][48] = {};
  for (int kb = 0; kb < 48; ++kb) {
    const int c = kb >> 1, comp = kb & 1, cm = c & 3;
    static const int arm_of[4][2] = {{0, 1}, {1, 0}, {0, 1}, {1, 0}};     // [c mod 4][comp]: 0 = I', 1 = Q'
    static const int sign_of[4][2] = {{1, 1}, {1, -1}, {-1, -1}, {-1, 1}};
    for (int o = 0; o < 8; ++o) {
      const int k = 16 + o - c;
      if (k >= 0 && k < taps::WB_PRE::N) A[8 * arm_of[cm][comp] + o][kb] = sign_of[cm][comp] * 2 * taps::WB_PRE::tap(k);
    }
  }
  auto part = [](int v, int h) {
    const int lo = ((v + 128) & 255) - 128;
    return h == 0 ? (v - lo) / 256 : lo;
  };
  // E[h][row][0..63]: K 0..15 = kb 0..15, K 16..31 = the start spread over C's weights, K 32..63 = kb 16..47
  static int E[2][16][64];
  for (int h = 0; h < 2; ++h)
    for (int row = 0; row < 16; ++row) {
      int sum = 0;
      for (int kb = 0; kb < 48; ++kb) {
        const int v = part(A[row][kb], h);
        sum += v;
        E[h][row][kb < 16 ? kb : 16 + kb] = v;
      }
      const int start = (h == 1 ? 1 << 15 : 0) - 128 * sum;
      int big = (start >= 0 ? start + 127 : start - 127) / 255;  // start = 255 * big + small, |small| <= 127
      int small = start - 255 * big;
      for (int i = 0; i < 12; ++i) {  // big over twelve int8 entries, small over four
        const int left = 12 - i, v = big >= 0 ? (big + left - 1) / left : -((-big + left - 1) / left);
        E[h][row][16 + i] = v;
        big -= v;
      }
      for (int i = 0; i < 4; ++i) {
        const int left = 4 - i, v = small >= 0 ? (small + left - 1) / left : -((-small + left - 1) / left);
        E[h][row][28 + i] = v;
        small -= v;
      }
    }
  auto word = [&](int h, int row, int k0) {
    uint32_t w = 0;
    for (int b = 0; b < 4; ++b) {
      const int v = E[h][row][k0 + b];
      if (v < -128 || v > 127) abort();  // cannot happen: |start| < 255 * 12 * 127
      w |= (uint32_t)(uint8_t)(int8_t)v << (8 * b);
    }
    return w;
  };
  for (int lane = 0; lane < 32; ++lane) {
    const int g = lane >> 2, tq = lane & 3;
    for (int h = 0; h < 2; ++h)
      for (int s2 = 0; s2 < 2; ++s2)
        for (int r = 0; r < 4; ++r)
          tab[((2 * s2 + h) * 32 + lane) * 4 + r] = word(h, g + 8 * (r & 1), 32 * s2 + 16 * (r >> 1) + 4 * tq);
  }
  tab[WB_TAB_A_WORDS + 0] = tab[WB_TAB_A_WORDS + 1] = tab[WB_TAB_A_WORDS + 2] = 0xffffffffu;
  tab[WB_TAB_A_WORDS + 3] = 0x01010101u;
  return tab;
}

int launch_fm_tile(sdr_engine *e, const uint8_t *iq, uint64_t ch_stride, uint32_t n_samples, int fmt) {
  const int kind = SDR_KIND_FM;
  const uint32_t n_list = (uint32_t)e->list[kind].size();
  if (n_list == 0) return SDR_OK;
  const uint32_t G = 4;  // worker warps per CTA; they never synchronise
  const int smem = (int)G * FM_WARP_SMEM;
  if (!e->d_fm_tab) {
    const std::vector<uint32_t> tab = fm_mma_table();
    SDR_CK(e, cudaMalloc(&e->d_fm_tab, tab.size() * 4));
    SDR_CK(e, cudaMemcpy(e->d_fm_tab, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice));
  }
  // equal shares of the launch's tiles, as for AM/SSB (launch_amssb)
  static const int wps_env = getenv("SDR_FM_WARPS_PER_SM") ? atoi(getenv("SDR_FM_WARPS_PER_SM")) : 0;
  const uint32_t n_tiles = (n_samples + TILE - 1) / TILE;
  const uint64_t total_tiles = (uint64_t)n_list * n_tiles;
  uint64_t n_warps = (uint64_t)e->n_sm * (wps_env > 0 ? wps_env : 48);
  static const int min_share_env = getenv("SDR_FM_MIN_SHARE") ? atoi(getenv("SDR_FM_MIN_SHARE")) : 0;  // tuning override
  const uint64_t min_share = min_share_env > 0 ? (uint64_t)min_share_env : 8;
  n_warps = std::min<uint64_t>(n_warps, (total_tiles + min_share - 1) / min_share);
  n_warps = std::max<uint64_t>(n_warps, 1);
  LaunchParams p = {};
  p.iq = iq;
  p.ch_stride = ch_stride;
  p.n_samples = n_samples;
  p.fmt = fmt;
  p.chan_ids = e->d_list[kind];
  p.n_list = n_list;
  p.G = G;
  p.state = e->d_state[kind];
  p.state_stride = (uint32_t)FmTile::STATE_BYTES;
  p.scale = e->d_scale[kind];
  p.lsb = e->d_lsb;
  p.pcm = e->pass_pcm;
  p.pcm_stride = e->pcm_stride;
  p.lut = e->d_lut_fm;
  p.aux = (uint32_t)n_warps;
  p.call_id = (uint32_t)(e->pass % 0x7fffffffull) + 1;
  p.tab = e->d_fm_tab;
  p.scratch = nullptr;
  p.allowed = e->pass_allowed;
  const uint32_t grid = (uint32_t)((n_warps + G - 1) / G);
  static const int minb_env = getenv("SDR_FM_MIN_CTAS") ? atoi(getenv("SDR_FM_MIN_CTAS")) : 0;
  switch (minb_env) {
    case 5: fm_tile_kernel<5><<<grid, 32 * G, smem, e->stream>>>(p); break;
    case 6: fm_tile_kernel<6><<<grid, 32 * G, smem, e->stream>>>(p); break;
    default: fm_tile_kernel<4><<<grid, 32 * G, smem, e->stream>>>(p); break;
  }
  SDR_CK(e, cudaGetLastError());
  e->launches++;
  return SDR_OK;
}

// Tap matrices of the tcgen05 WBFM pre-filter (wbfm_tile4_kernel, WbUmma): D = A * B with A = raw u8 input bytes,
// 64 per row. B[ks][part] is 32 columns x K = 32: column n = 2 p + arm gives I' (arm 0) or Q' (arm 1) of sample p
// (0..15) of a group of 16; K step ks covers the raw bytes 32 ks - 32 .. 32 ks - 1 counted from the group's first
// (complex sample c = kb >> 1 counted from 16 before the group, I at even bytes). Output p is
// sum_k 2 h[k] x'[16 + p - k] (FirFilter_int16.cc:151-213 with the taps doubled, WbTile::Pre2), x' the rotated sample
// (IqDataProcessor.cc:567-611; a group starts a rotation period). part 0 / 1: the tap's high / low byte, 256 * hi + lo
// with both int8. The accumulator starts are not here: WbUmma::start_of, stored into tensor memory by the kernel.
// Element (n, k) of a matrix sits at WbUmma::b_offset(n, k).
std::vector<uint8_t> wb_umma_table() {
  std::vector<uint8_t> tab(WB4_TAB_BYTES, 0);
  auto part = [](int v, int h) {
    const int lo = ((v + 128) & 255) - 128;
    return h == 0 ? (v - lo) / 256 : lo;
  };
  for (int kb = 0; kb < 64; ++kb) {
    const int c = kb >> 1, comp = kb & 1, cm = c & 3;
    // which arm this raw component feeds at phase cm: I' = I0, -Q1, -I2, Q3; Q' = Q0, I1, -Q2, -I3
    const int arm = (cm & 1) ? 1 - comp : comp;
    for (int pp = 0; pp < 16; ++pp) {
      const int k = 16 + pp - c;
      if (k < 0 || k >= taps::WB_PRE::N) continue;
      const int v = WbUmma::sign_of(cm, arm) * 2 * taps::WB_PRE::tap(k);
      for (int h = 0; h < 2; ++h)
        tab[((kb >> 5) * 2 + h) * WB4_B_TILE + WbUmma::b_offset(2 * pp + arm, kb & 31)] = (uint8_t)(int8_t)part(v, h);
    }
  }
  return tab;
}

int wb_tab_ready(sdr_engine *e) {
  if (!e->d_wb_tab) {
    const std::vector<uint32_t> tab = wb_mma_table();
    SDR_CK(e, cudaMalloc(&e->d_wb_tab, tab.size() * 4));
    SDR_CK(e, cudaMemcpy(e->d_wb_tab, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice));
  }
  return SDR_OK;
}

// wbfm_tile3_kernel: two channels per worker warp, up to 28 channels per CTA behind one recurrence warp
int launch_wbfm_tile3(sdr_engine *e, const uint8_t *iq, uint64_t ch_stride, uint32_t n_samples, int fmt,
                      cudaStream_t stream) {
  using T = WbTile3;
  int rc_tab = SDR_OK;
  const int kind = SDR_KIND_WBFM;
  const uint32_t n_list = (uint32_t)e->list[kind].size();
  // one CTA per SM (table and rings fill shared memory): spread the channels evenly over the waves,
  // an even number of channels per CTA
  // (24 or 26 channels per CTA -- three workers on every scheduler -- were measured and lost:
  // 0.909 ms against 0.783 for WBFM x8192, profiles/r02_wbfm_generations.txt)
  static const int g_env = getenv("SDR_WB_G") ? atoi(getenv("SDR_WB_G")) : 0;  // tuning override
  const long max_g = g_env ? g_env : 2 * T::MAX_WORKERS;
  const long slots = e->n_sm;
  const long W = ((long)n_list + slots * max_g - 1) / (slots * max_g);
  uint32_t G = (uint32_t)(((long)n_list + slots * W - 1) / (slots * W));
  if (e->shape[kind].G) G = e->shape[kind].G;
  G = (G + 1) & ~1u;
  if (G > 2u * (uint32_t)T::MAX_WORKERS) G = 2u * (uint32_t)T::MAX_WORKERS;
  if (G < 2) G = 2;
  const int workers = (int)G / 2;
  static const bool mma_env = getenv("SDR_WB_MMA") && atoi(getenv("SDR_WB_MMA")) != 0;  // A/B switch
  const bool mma = e->wb_prefilter_mma || mma_env;
  const int smem = T::smem_bytes(workers, mma);
  if (mma && (rc_tab = wb_tab_ready(e))) return rc_tab;
  LaunchParams p = {};
  p.iq = iq;
  p.ch_stride = ch_stride;
  p.n_samples = n_samples;
  p.fmt = fmt;
  p.chan_ids = e->d_list[kind];
  p.n_list = n_list;
  p.G = G;
  p.state = e->d_state[kind];
  p.state_stride = (uint32_t)WbTile::STATE_BYTES;
  p.scale = e->d_scale[kind];
  p.lsb = e->d_lsb;
  p.pcm = e->pass_pcm;
  p.pcm_stride = e->pcm_stride;
  p.lut = e->d_lut_wbfm_half;
  p.aux = (uint32_t)std::min(workers, (int)T::REC_WARP);
  p.scratch = nullptr;
  p.allowed = e->pass_allowed;
  p.tab = e->d_wb_tab;
  p.counters = e->wb_count ? e->d_counters : nullptr;  // one atomic per tile: only when somebody asked
  const uint32_t grid = (n_list + G - 1) / G;
  if (mma) {
    SDR_CK(e, cudaFuncSetAttribute(wbfm_tile3_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    wbfm_tile3_kernel<true><<<grid, 32 * (workers + 1), smem, stream>>>(p);
  } else {
    SDR_CK(e, cudaFuncSetAttribute(wbfm_tile3_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    wbfm_tile3_kernel<false><<<grid, 32 * (workers + 1), smem, stream>>>(p);
  }
  SDR_CK(e, cudaGetLastError());
  e->launches++;
  return SDR_OK;
}

// wbfm_tile2_kernel: the atan2 half-plane table in shared memory, 15 channels per CTA
int launch_wbfm_tile2(sdr_engine *e, const uint8_t *iq, uint64_t ch_stride, uint32_t n_samples, int fmt,
                      cudaStream_t stream) {
  using T = WbTile2;
  const int kind = SDR_KIND_WBFM;
  const uint32_t n_list = (uint32_t)e->list[kind].size();
  // one CTA per SM (table and rings fill shared memory): spread the channels evenly over the
  // waves. 14 workers leave the recurrence warp's scheduler two warps lighter than the others.
  static const int g_env = getenv("SDR_WB_G") ? atoi(getenv("SDR_WB_G")) : 0;  // tuning override
  const long max_g = g_env ? g_env : 14;
  const long slots = e->n_sm;
  const long W = ((long)n_list + slots * max_g - 1) / (slots * max_g);
  uint32_t G = (uint32_t)(((long)n_list + slots * W - 1) / (slots * W));
  // A round is as long as the recurrence warp's 1024 dependent steps whatever the number of workers up to 14, and
  // a CTA keeps its SM to itself: when other modes share the GPU, 14 channels per CTA cost this kernel nothing and
  // leave them the SMs it does not need (mixed x8192: 0.373 -> 0.348 ms, profiles/r02_wbfm4.txt)
  bool others = false;
  for (int k2 = SDR_KIND_AM; k2 <= SDR_KIND_SSB; ++k2) others = others || (k2 != kind && !e->list[k2].empty());
  if (others) G = (uint32_t)max_g;
  static const int gx_env = getenv("SDR_WB_GX") ? atoi(getenv("SDR_WB_GX")) : 0;  // exact, for sweeps
  if (gx_env) G = (uint32_t)gx_env;
  if (e->shape[kind].G) G = e->shape[kind].G;
  if (G > (uint32_t)T::MAX_WORKERS) G = T::MAX_WORKERS;
  static const bool mma_env = getenv("SDR_WB_MMA") && atoi(getenv("SDR_WB_MMA")) != 0;  // A/B switch
  const bool mma = e->wb_prefilter_mma || mma_env;
  const int smem = T::smem_bytes((int)G, mma);
  int rc_tab = SDR_OK;
  if (mma && (rc_tab = wb_tab_ready(e))) return rc_tab;
  LaunchParams p = {};
  p.iq = iq;
  p.ch_stride = ch_stride;
  p.n_samples = n_samples;
  p.fmt = fmt;
  p.chan_ids = e->d_list[kind];
  p.n_list = n_list;
  p.G = G;
  p.state = e->d_state[kind];
  p.state_stride = (uint32_t)WbTile::STATE_BYTES;
  p.scale = e->d_scale[kind];
  p.lsb = e->d_lsb;
  p.pcm = e->pass_pcm;
  p.pcm_stride = e->pcm_stride;
  p.lut = e->d_lut_wbfm_half;
  p.tab = e->d_wb_tab;
  p.counters = e->wb_count ? e->d_counters : nullptr;  // one atomic per tile: only when somebody asked
  static const int rec_env = getenv("SDR_WB_REC") ? atoi(getenv("SDR_WB_REC")) : -1;  // tuning override
  p.aux = (uint32_t)((rec_env >= 0 && rec_env <= (int)G) ? rec_env : std::min((int)G, (int)T::REC_WARP));
  p.scratch = nullptr;
  p.allowed = e->pass_allowed;
  const uint32_t grid = (n_list + G - 1) / G;
  if (mma) {
    SDR_CK(e, cudaFuncSetAttribute(wbfm_tile2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    wbfm_tile2_kernel<true><<<grid, 32 * T::warps_for((int)G), smem, stream>>>(p);
  } else {
    SDR_CK(e, cudaFuncSetAttribute(wbfm_tile2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    wbfm_tile2_kernel<false><<<grid, 32 * T::warps_for((int)G), smem, stream>>>(p);
  }
  SDR_CK(e, cudaGetLastError());
  e->launches++;
  return SDR_OK;
}

// wbfm_tile4_kernel: the pre-filter on the tcgen05 tensor cores; two channels per worker warp for banks that need more
// than one wave of one-channel-per-warp CTAs (as generation 3 against 2), else one
int launch_wbfm_tile4(sdr_engine *e, const uint8_t *iq, uint64_t ch_stride, uint32_t n_samples, int fmt,
                      cudaStream_t stream) {
  const int kind = SDR_KIND_WBFM;
  const uint32_t n_list = (uint32_t)e->list[kind].size();
  const int max_workers = WB4_MAX_WARPS - 2;
  static const int two_env = getenv("SDR_WB4_TWO") ? atoi(getenv("SDR_WB4_TWO")) : -1;  // tuning override
  const bool two = e->wb4_geometry ? e->wb4_geometry == 1
                   : two_env >= 0  ? two_env != 0
                                   : n_list > (uint32_t)(max_workers - 1) * (uint32_t)e->n_sm;
  static const int g_env = getenv("SDR_WB_G") ? atoi(getenv("SDR_WB_G")) : 0;  // tuning override
  const long max_g = g_env ? g_env : (two ? 2 : 1) * max_workers;
  const long slots = e->n_sm;
  const long W = ((long)n_list + slots * max_g - 1) / (slots * max_g);
  uint32_t G = (uint32_t)(((long)n_list + slots * W - 1) / (slots * W));
  static const int gx_env = getenv("SDR_WB_GX") ? atoi(getenv("SDR_WB_GX")) : 0;  // exact, for sweeps
  if (gx_env) G = (uint32_t)gx_env;
  if (e->shape[kind].G) G = e->shape[kind].G;
  if (two) G = (G + 1) & ~1u;
  if (G > (uint32_t)max_g) G = (uint32_t)max_g;
  if (G < (two ? 2u : 1u)) G = two ? 2 : 1;
  const int workers = two ? (int)G / 2 : (int)G;
  const int rec = std::min(workers, (int)WbTile2::REC_WARP);
  const int n_slots = rec < workers ? workers + 1 : workers;
  const int smem = two ? WbUmma::smem_bytes<true>(workers, n_slots) : WbUmma::smem_bytes<false>(workers, n_slots);
  if (!e->d_wb4_tab) {
    const std::vector<uint8_t> tab = wb_umma_table();
    SDR_CK(e, cudaMalloc(&e->d_wb4_tab, tab.size()));
    SDR_CK(e, cudaMemcpy(e->d_wb4_tab, tab.data(), tab.size(), cudaMemcpyHostToDevice));
  }
  LaunchParams p = {};
  p.iq = iq;
  p.ch_stride = ch_stride;
  p.n_samples = n_samples;
  p.fmt = fmt;
  p.chan_ids = e->d_list[kind];
  p.n_list = n_list;
  p.G = G;
  p.state = e->d_state[kind];
  p.state_stride = (uint32_t)WbTile::STATE_BYTES;
  p.scale = e->d_scale[kind];
  p.lsb = e->d_lsb;
  p.pcm = e->pass_pcm;
  p.pcm_stride = e->pcm_stride;
  p.lut = e->d_lut_wbfm_half;
  p.aux = (uint32_t)rec;
  p.tab = reinterpret_cast<const uint32_t *>(e->d_wb4_tab);
  p.counters = e->d_counters;
  p.call_id = e->wb_count ? 1 : 0;  // the per-tile diagnostic counters: one atomic per tile, only when somebody asked
  p.scratch = nullptr;
  p.allowed = e->pass_allowed;
  const uint32_t grid = (n_list + G - 1) / G;
  if (two) {
    SDR_CK(e, cudaFuncSetAttribute(wbfm_tile4_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    wbfm_tile4_kernel<true><<<grid, 32 * (workers + 2), smem, stream>>>(p);
  } else {
    SDR_CK(e, cudaFuncSetAttribute(wbfm_tile4_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    wbfm_tile4_kernel<false><<<grid, 32 * (workers + 2), smem, stream>>>(p);
  }
  SDR_CK(e, cudaGetLastError());
  // how many (half-)tiles clipping bytes kept off the tensor cores, for launch_wbfm_tile's choice of kernel: read by
  // a later call, whenever the copy has landed
  if (!e->h_wb_clip) {
    SDR_CK(e, cudaHostAlloc(&e->h_wb_clip, 16, cudaHostAllocDefault));
    *e->h_wb_clip = 0;  // what counters[3] starts from: a read before the first copy lands sees "nothing clipped"
  }
  SDR_CK(e, cudaMemcpyAsync((void *)e->h_wb_clip, e->d_counters + 3, 4, cudaMemcpyDeviceToHost, stream));
  e->wb4_units = (uint64_t)((n_list + (two ? 1 : 0)) / (two ? 2 : 1)) * ((n_samples + (two ? 511 : 1023)) / (two ? 512 : 1024));
  e->launches++;
  return SDR_OK;
}

int launch_wbfm_tile(sdr_engine *e, const uint8_t *iq, uint64_t ch_stride, uint32_t n_samples, int fmt,
                     cudaStream_t stream) {
  using T = WbTile;
  const int kind = SDR_KIND_WBFM;
  const uint32_t n_list = (uint32_t)e->list[kind].size();
  if (n_list == 0) return SDR_OK;
  // SDR_WB_KERNEL=1 .. 4 select a generation of the kernel (1: table gathered from global memory; 2: table in shared
  // memory, one channel per worker warp; 3: two channels per worker warp; 4: 3's or 2's geometry with the pre-filter
  // on the tcgen05 tensor cores). Default: 4 once a bank needs more than one wave of one-channel-per-warp CTAs --
  // two channels per warp halve the recurrence warp's chain per round and the round is worker-bound, which is where
  // taking the pre-filter off the CUDA cores pays (WBFM x8192: 0.785 -> 0.700 ms); below that (the WBFM share of a
  // mixed bank) the round is bound by the 1024-step chain whatever the workers do, and 2 has the least overhead.
  static const int gen_env = getenv("SDR_WB_KERNEL") ? atoi(getenv("SDR_WB_KERNEL")) : 0;
  int gen = e->wb_kernel ? e->wb_kernel : gen_env;
  const bool small_bank = n_list <= (uint32_t)(WbTile2::MAX_WORKERS - 1) * (uint32_t)e->n_sm;
  if (gen == 0) {
    gen = small_bank ? 2 : 4;
    // A bank whose input clips (raw bytes 0 where the rotation negates) gets nothing from generation 4 but its
    // overhead (+24 % when every tile falls back): if more than a quarter of the last observed launch fell back,
    // the next 64 calls take generation 3, then generation 4 is tried again.
    // input that is already signed and rotated never takes the tensor cores (the tap matrices are the u8 format's)
    if (gen == 4 && fmt != FMT_U8_OFFSET_ROTATE) gen = 3;
    if (gen == 4) {
      if (e->h_wb_clip) {
        const uint32_t seen = *e->h_wb_clip;
        if ((uint64_t)(seen - e->wb_clip_seen) * 4 > e->wb4_units) e->wb_clip_hold = 64;
        e->wb_clip_seen = seen;
      }
      if (e->wb_clip_hold > 0) {
        --e->wb_clip_hold;
        gen = 3;
      }
    }
  } else if (!e->wb_kernel && gen == 3 && small_bank) {
    gen = 2;
  }
  if (gen == 4 && e->d_lut_wbfm_half) return launch_wbfm_tile4(e, iq, ch_stride, n_samples, fmt, stream);
  if (gen == 3 && e->d_lut_wbfm_half) return launch_wbfm_tile3(e, iq, ch_stride, n_samples, fmt, stream);
  if (gen != 1 && e->d_lut_wbfm_half) return launch_wbfm_tile2(e, iq, ch_stride, n_samples, fmt, stream);
  // one CTA per SM (the rings fill shared memory): spread the channels evenly over the waves
  const long slots = e->n_sm;
  const long W = ((long)n_list + slots * T::MAX_WORKERS - 1) / (slots * T::MAX_WORKERS);
  uint32_t G = (uint32_t)(((long)n_list + slots * W - 1) / (slots * W));
  static const int g_env = getenv("SDR_WB_G") ? atoi(getenv("SDR_WB_G")) : 0;  // tuning override
  if (g_env) G = (uint32_t)g_env;
  if (e->shape[kind].G) G = e->shape[kind].G;
  if (G > (uint32_t)T::MAX_WORKERS) G = T::MAX_WORKERS;
  const int smem = T::smem_bytes((int)G);
  LaunchParams p = {};
  p.iq = iq;
  p.ch_stride = ch_stride;
  p.n_samples = n_samples;
  p.fmt = fmt;
  p.chan_ids = e->d_list[kind];
  p.n_list = n_list;
  p.G = G;
  p.state = e->d_state[kind];
  p.state_stride = (uint32_t)T::STATE_BYTES;
  p.scale = e->d_scale[kind];
  p.lsb = e->d_lsb;
  p.pcm = e->pass_pcm;
  p.pcm_stride = e->pcm_stride;
  p.lut = e->d_lut_wbfm;
  // workers allowed on the recurrence warp's scheduler (tunable: SDR_WB_S3)
  static const int s3_env = getenv("SDR_WB_S3") ? atoi(getenv("SDR_WB_S3")) : 4;
  p.aux = (uint32_t)s3_env;
  p.scratch = nullptr;
  p.allowed = e->pass_allowed;
  SDR_CK(e, cudaFuncSetAttribute(wbfm_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  const uint32_t grid = (n_list + G - 1) / G;
  wbfm_tile_kernel<<<grid, 32 * T::warps_for((int)G, s3_env), smem, stream>>>(p);
  SDR_CK(e, cudaGetLastError());
  e->launches++;
  return SDR_OK;
}

// Converts the block of every dumped channel into the dump buffer. Runs first in a call:
// the reference sends the dump whatever the squelch decides (IqDataProcessor.cc:753-760).
int run_iq_dump(sdr_engine *e, const uint8_t *iq, uint64_t ch_stride, uint64_t bytes, int fmt) {
  if (e->dump_dirty) {
    e->dump_list.clear();
    for (uint32_t ch = 0; ch < e->n; ++ch)
      if (e->dump_on[ch]) e->dump_list.push_back(ch);
    if (e->dump_list.size() > e->dump_rows) {
      SDR_CK(e, cudaStreamSynchronize(e->stream));
      if (e->dump_reader) SDR_CK(e, cudaStreamSynchronize(e->dump_reader));
      cudaFree(e->d_dump);
      cudaFree(e->d_dump_list);
      e->d_dump = nullptr;
      e->d_dump_list = nullptr;
      e->dump_rows = e->dump_list.size();
      SDR_CK(e, cudaMalloc(&e->d_dump, sdr_engine::RING_MAX * e->dump_rows * e->max_bytes));
      SDR_CK(e, cudaMalloc(&e->d_dump_list, e->dump_rows * 4));
    }
    if (!e->dump_list.empty()) {
      SDR_CK(e, cudaStreamSynchronize(e->stream));  // the list may be in use by a queued kernel
      SDR_CK(e, cudaMemcpy(e->d_dump_list, e->dump_list.data(), e->dump_list.size() * 4, cudaMemcpyHostToDevice));
    }
    e->dump_dirty = false;
  }
  e->dump_bytes = 0;
  if (e->dump_list.empty()) return SDR_OK;
  DumpParams d{};
  d.iq = iq;
  d.ch_stride = ch_stride;
  d.bytes = bytes;
  d.fmt = fmt;
  d.list = e->d_dump_list;
  d.n_list = (uint32_t)e->dump_list.size();
  // Ring entry seq % RING_MAX (so are the squelch's gate and magnitude, see run_squelch). A direct
  // caller reads entry seq - 1 on `stream`, in order. The ingest ring reads tick k's entry on its
  // d2h stream, after tick k's ev_comp and before its ev_done, and ingest_commit makes tick k+2's
  // work on `stream` wait for tick k's ev_done. Tick k+3, the next to write this entry, is queued on
  // `stream` after tick k+2, so its kernels start only once tick k's copies are over: three
  // entries are enough however deep the ingest ring is. A call gated in block passes changes
  // nothing here: its passes are all queued on `stream` (or wait on it) before tick k+1's work.
  d.out = e->dump_of(e->seq);
  d.out_stride = e->max_bytes;
  const uint64_t pieces = bytes / 16;
  uint32_t gx = (uint32_t)std::min<uint64_t>((pieces + 255) / 256, 64);
  iq_dump_kernel<<<dim3(gx, d.n_list), 256, 0, e->stream>>>(d);
  SDR_CK(e, cudaGetLastError());
  e->launches++;
  e->dump_bytes = bytes;
  return SDR_OK;
}

// Blocks the squelch judges in a call of `bytes` per channel at the current setting
uint32_t squelch_blocks(const sdr_engine *e, uint64_t bytes) {
  return e->squelch_block ? (uint32_t)((bytes + e->squelch_block - 1) / e->squelch_block) : 1;
}

// Samples channel ch produced in a call of `bytes` judged as n_blocks blocks of block_bytes
// (the last one shorter), given the call's gates [n_blocks][pitch]: its open blocks' samples.
uint32_t open_samples(const uint8_t *gate, uint64_t pitch, uint32_t ch, uint32_t n_blocks, uint64_t block_bytes,
                      uint64_t bytes) {
  uint64_t total = 0;
  for (uint32_t k = 0; k < n_blocks; ++k)
    if (gate[(size_t)k * pitch + ch]) total += (k + 1 == n_blocks ? bytes - (uint64_t)k * block_bytes : block_bytes) / 64;
  return (uint32_t)total;
}

// Runs the squelch kernel when a threshold that can close is set (the gate is then in force)
// or when signal reports are wanted. A channel whose threshold can never close
// (threshold <= -42 - gain: even magnitude 0 passes, DbfsCalculator.cc) needs no kernel.
int run_squelch(sdr_engine *e, const uint8_t *iq, uint64_t ch_stride, uint64_t bytes, int fmt) {
  e->last_gated = false;
  if (e->squelch_dirty) {
    bool armed = false;
    for (uint32_t ch = 0; ch < e->n && !armed; ++ch)
      armed = (int64_t)e->threshold[ch] > -42 - (int64_t)e->rx_gain_db[ch];
    if ((armed || e->signal_reports) && !e->d_tracking) {
      SDR_CK(e, cudaMalloc(&e->d_threshold, (size_t)e->n * 4));
      SDR_CK(e, cudaMalloc(&e->d_rx_gain, (size_t)e->n * 4));
      SDR_CK(e, cudaMalloc(&e->d_tracking, e->n));
      SDR_CK(e, cudaMalloc(&e->d_db_table, 128 * 4));
      // until now every block of every channel passed: the trackers are in `Tracking`
      // (SignalTracker.cc:104-145) if any block was seen, else in `NoSignal`
      SDR_CK(e, cudaMemsetAsync(e->d_tracking, e->seq > 0 ? 1 : 0, e->n, e->stream));
      int32_t table[128];
      for (int i = 1; i < 128; ++i) {  // DbfsCalculator.cc:60-68, host libm like the reference
        float db = 20 * log10f((float)i);
        table[i] = (int32_t)db;
      }
      table[0] = table[1];
      SDR_CK(e, cudaMemcpyAsync(e->d_db_table, table, sizeof table, cudaMemcpyHostToDevice, e->stream));
    }
    if (e->d_tracking) {
      int rc = join_streams(e);  // a recurrence kernel may still be reading its gate
      if (rc) return rc;
      SDR_CK(e, cudaMemcpyAsync(e->d_threshold, e->threshold.data(), (size_t)e->n * 4, cudaMemcpyHostToDevice, e->stream));
      SDR_CK(e, cudaMemcpyAsync(e->d_rx_gain, e->rx_gain_db.data(), (size_t)e->n * 4, cudaMemcpyHostToDevice, e->stream));
    }
    e->squelch_armed = armed;
    e->squelch_dirty = false;
  }
  if (!e->squelch_armed && !e->signal_reports) {
    if (e->d_tracking) e->tracking_stale = true;
    return SDR_OK;
  }
  if (e->tracking_stale) {
    SDR_CK(e, cudaMemsetAsync(e->d_tracking, 1, e->n, e->stream));
    e->tracking_stale = false;
  }
  // gate and magnitude entries: one row per block of the longest call the setting allows
  const uint32_t rows = std::max(e->sig_rows, squelch_blocks(e, e->max_bytes));
  if (!e->d_allowed || rows > e->sig_rows) {
    if (e->d_allowed) {  // queued recurrence kernels and read-back copies may still read the old entries
      int rc = join_streams(e);
      if (rc) return rc;
      SDR_CK(e, cudaStreamSynchronize(e->stream));
      if (e->dump_reader) SDR_CK(e, cudaStreamSynchronize(e->dump_reader));
      cudaFree(e->d_allowed);
      cudaFree(e->d_magnitude);
      e->d_allowed = nullptr;
      e->d_magnitude = nullptr;
    }
    e->sig_rows = rows;
    const size_t cells = sdr_engine::RING_MAX * (size_t)rows * e->n;
    SDR_CK(e, cudaMalloc(&e->d_allowed, cells));
    SDR_CK(e, cudaMalloc(&e->d_magnitude, cells * 4));
    SDR_CK(e, cudaMemsetAsync(e->d_magnitude, 0, cells * 4, e->stream));
  }
  SquelchParams q;
  q.iq = iq;
  q.ch_stride = ch_stride;
  q.n_bytes = bytes;
  q.block_bytes = e->squelch_block ? e->squelch_block : bytes;
  q.n_channels = e->n;
  q.fmt = fmt;
  q.threshold = e->d_threshold;
  q.gain_db = e->d_rx_gain;
  q.tracking = e->d_tracking;
  // ring entry seq % RING_MAX: why three entries suffice behind an ingest ring, see run_iq_dump
  q.allowed = e->allowed_of(e->seq);
  q.magnitude = e->magnitude_of(e->seq);
  q.db_table = e->d_db_table;
  squelch_kernel<<<e->n, 128, 0, e->stream>>>(q);
  SDR_CK(e, cudaGetLastError());
  e->launches++;
  e->last_gated = true;
  return SDR_OK;
}

int upload_tables(sdr_engine *e) {
  bool dirty = e->lists_dirty || e->lsb_dirty;
  for (int k = 1; k <= 4; ++k) dirty = dirty || e->scale_dirty[k];
  if (dirty) {  // a recurrence kernel may still be reading the tables
    int rc = join_streams(e);
    if (rc) return rc;
  }
  if (e->lists_dirty) {
    for (int k = 1; k <= 4; ++k) e->list[k].clear();
    for (uint32_t ch = 0; ch < e->n; ++ch) {
      const int k = kind_of_mode(e->mode[ch]);
      if (k) e->list[k].push_back(ch);
    }
    for (int k = 1; k <= 4; ++k)
      if (!e->list[k].empty())
        SDR_CK(e, cudaMemcpyAsync(e->d_list[k], e->list[k].data(), e->list[k].size() * 4,
                                  cudaMemcpyHostToDevice, e->stream));
    e->lists_dirty = false;
  }
  if (e->lsb_dirty) {
    SDR_CK(e, cudaMemcpyAsync(e->d_lsb, e->lsb.data(), e->n, cudaMemcpyHostToDevice, e->stream));
    e->lsb_dirty = false;
  }
  for (int k = 1; k <= 4; ++k) {
    if (!e->scale_dirty[k]) continue;
    for (uint32_t ch = 0; ch < e->n; ++ch) e->scale[k][ch] = scale_of(k, e->gain[k][ch], e->scaling);
    SDR_CK(e, cudaMemcpyAsync(e->d_scale[k], e->scale[k].data(), (size_t)e->n * 4, cudaMemcpyHostToDevice,
                              e->stream));
    e->scale_dirty[k] = false;
  }
  // the host vectors above must outlive the async copies from pageable memory;
  // cudaMemcpyAsync from pageable memory has returned only after staging them.
  return SDR_OK;
}

}  // namespace

extern "C" {

const char *sdr_version(void) { return "sdr_b200 0.1 (sm_100a)"; }

const char *sdr_last_error(const sdr_engine *e) { return e ? e->err.c_str() : g_create_error.c_str(); }

int sdr_state_bytes(int kind) { return state_bytes(kind); }

int sdr_engine_create(uint32_t n_channels, int device, uint64_t max_bytes_per_channel, sdr_engine **out) {
  if (!out) return SDR_E_ARG;
  *out = nullptr;
  if (n_channels == 0 || max_bytes_per_channel == 0 || max_bytes_per_channel % 64 ||
      max_bytes_per_channel / 2 > 0xffffffe0ull)
    return fail(nullptr, SDR_E_ARG, "n_channels and max_bytes_per_channel (multiple of 64) must be positive");
  int count = 0;
  cudaError_t ce = cudaGetDeviceCount(&count);
  if (ce != cudaSuccess || count == 0)
    return fail(nullptr, SDR_E_CUDA, "no CUDA device: this engine has no CPU path", ce);
  if (device < 0 || device >= count) return fail(nullptr, SDR_E_ARG, "device index out of range");
  sdr_engine *e = new (std::nothrow) sdr_engine();
  if (!e) return SDR_E_NOMEM;
  e->device = device;
  e->n = n_channels;
  e->max_bytes = max_bytes_per_channel;
#define SDR_CK_CREATE(call)                                                       \
  do {                                                                            \
    cudaError_t _ce = (call);                                                     \
    if (_ce != cudaSuccess) {                                                     \
      fail(nullptr, SDR_E_CUDA, #call, _ce);                                      \
      sdr_engine_destroy(e);                                                      \
      return _ce == cudaErrorMemoryAllocation ? SDR_E_NOMEM : SDR_E_CUDA;         \
    }                                                                             \
  } while (0)
  SDR_CK_CREATE(cudaSetDevice(device));
  SDR_CK_CREATE(cudaDeviceGetAttribute(&e->n_sm, cudaDevAttrMultiProcessorCount, device));
  SDR_CK_CREATE(cudaDeviceGetAttribute(&e->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
  SDR_CK_CREATE(cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking));
  {
    // the recurrence kernels are small and latency bound: highest priority, so their CTAs are
    // placed before the next call's FIR kernel floods the SMs
    int prio_lo = 0, prio_hi = 0;
    SDR_CK_CREATE(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    SDR_CK_CREATE(cudaStreamCreateWithPriority(&e->rec_stream, cudaStreamNonBlocking, prio_hi));
    SDR_CK_CREATE(cudaStreamCreateWithPriority(&e->wb_stream, cudaStreamNonBlocking, prio_hi));
    SDR_CK_CREATE(cudaEventCreateWithFlags(&e->ev_in, cudaEventDisableTiming));
    SDR_CK_CREATE(cudaEventCreateWithFlags(&e->ev_wb, cudaEventDisableTiming));
  }
  for (int i = 0; i < sdr_engine::RING_MAX; ++i) {
    SDR_CK_CREATE(cudaEventCreateWithFlags(&e->ev_fir[i], cudaEventDisableTiming));
    SDR_CK_CREATE(cudaEventCreateWithFlags(&e->ev_rec[i], cudaEventDisableTiming));
  }
  for (int i = 0; i < sdr_engine::PACE; ++i)
    SDR_CK_CREATE(cudaEventCreateWithFlags(&e->ev_pace[i], cudaEventDisableTiming));
  if (getenv("SDR_TRACE") && atoi(getenv("SDR_TRACE"))) {
    std::vector<unsigned long long> init(4 * sdr_engine::TRACE_CALLS);
    for (size_t i = 0; i < init.size(); ++i) init[i] = (i & 1) ? 0ull : ~0ull;
    SDR_CK_CREATE(cudaMalloc(&e->d_trace, init.size() * 8));
    SDR_CK_CREATE(cudaMemcpy(e->d_trace, init.data(), init.size() * 8, cudaMemcpyHostToDevice));
  }
  SDR_CK_CREATE(cudaMalloc(&e->d_counters, 16));
  SDR_CK_CREATE(cudaMemset(e->d_counters, 0, 16));
  e->stream = e->own_stream;

  e->dump_on.assign(n_channels, 0);           // IqDataProcessor.cc:62
  e->threshold.assign(n_channels, -200);      // IqDataProcessor.cc:41
  e->rx_gain_db.assign(n_channels, 0);
  e->mode.assign(n_channels, SDR_MODE_NONE);  // IqDataProcessor.cc:38
  e->lsb.assign(n_channels, 1);               // SsbDemodulator.cc:143
  for (int k = 1; k <= 4; ++k) {
    e->gain[k].assign(n_channels, default_gain(k, e->scaling));
    e->scale[k].assign(n_channels, 0.f);
    const size_t sb = (size_t)state_bytes(k) * n_channels;
    SDR_CK_CREATE(cudaMalloc(&e->d_state[k], sb));
    SDR_CK_CREATE(cudaMemsetAsync(e->d_state[k], 0, sb, e->stream));
    SDR_CK_CREATE(cudaMalloc(&e->d_scale[k], (size_t)n_channels * 4));
    SDR_CK_CREATE(cudaMalloc(&e->d_list[k], (size_t)n_channels * 4));
  }
  SDR_CK_CREATE(cudaMalloc(&e->d_lsb, n_channels));
  e->pcm_stride = (max_bytes_per_channel / 64 + 7) & ~7ull;  // rows stay 16-byte aligned
  for (int i = 0; i < 2; ++i) {
    SDR_CK_CREATE(cudaMalloc(&e->d_pcm2[i], (size_t)n_channels * e->pcm_stride * 2));
    SDR_CK_CREATE(cudaMemsetAsync(e->d_pcm2[i], 0, (size_t)n_channels * e->pcm_stride * 2, e->stream));
  }

  // atan2 tables, built with the host libm exactly as the reference builds its
  // WBFM table (WbFmDemodulator.cc:159-170). NBFM calls atan2 per sample on
  // tuner outputs that lie in [-140, 139] for 8-bit input (FmDemodulator.cc:476),
  // so a 280x280 table of (float)atan2((double)q,(double)i) is the same function.
  {
    std::vector<float> t((size_t)FM_LUT_DIM * FM_LUT_DIM);
    for (int q = 0; q < FM_LUT_DIM; ++q)
      for (int i = 0; i < FM_LUT_DIM; ++i)
        t[(size_t)q * FM_LUT_DIM + i] = (float)atan2((double)(q + FM_LUT_MIN), (double)(i + FM_LUT_MIN));
    SDR_CK_CREATE(cudaMalloc(&e->d_lut_fm, t.size() * 4));
    SDR_CK_CREATE(cudaMemcpy(e->d_lut_fm, t.data(), t.size() * 4, cudaMemcpyHostToDevice));
  }
  {
    std::vector<float> t(256 * 256);
    for (int y = 0; y < 256; ++y)
      for (int x = 0; x < 256; ++x) t[(size_t)y * 256 + x] = (float)atan2((double)y - 128, (double)x - 128);
    SDR_CK_CREATE(cudaMalloc(&e->d_lut_wbfm, t.size() * 4));
    SDR_CK_CREATE(cudaMemcpy(e->d_lut_wbfm, t.data(), t.size() * 4, cudaMemcpyHostToDevice));
    // wbfm_tile2_kernel keeps only the half plane q >= 0 (row |q|, column (uint8_t)i) and takes
    // theta(q < 0) = -theta(-q): true for this libm's atan2 on every entry, or the kernel is not used
    std::vector<float> h((size_t)WbTile2::LUT_ROWS * 256);
    bool odd = true;
    for (int q = 0; q <= 128; ++q)
      for (int c = 0; c < 256; ++c) {
        const int i = (int)(int8_t)c;
        const float v = (float)atan2((double)q, (double)i);
        h[(size_t)q * 256 + c] = v;
        if (q <= 127 && v != t[(size_t)(q + 128) * 256 + (i + 128)]) odd = false;
        if (q >= 1) {
          const float n = t[(size_t)(128 - q) * 256 + (i + 128)];  // the reference's entry for -q
          if (memcmp(&n, &v, 4) == 0 || n != -v) odd = false;
        }
      }
    if (odd) {
      SDR_CK_CREATE(cudaMalloc(&e->d_lut_wbfm_half, h.size() * 4));
      SDR_CK_CREATE(cudaMemcpy(e->d_lut_wbfm_half, h.data(), h.size() * 4, cudaMemcpyHostToDevice));
    }
  }
  SDR_CK_CREATE(cudaStreamSynchronize(e->stream));
#undef SDR_CK_CREATE
  *out = e;
  return SDR_OK;
}

int sdr_engine_destroy(sdr_engine *e) {
  if (!e) return SDR_E_ARG;
  cudaSetDevice(e->device);
  if (e->own_stream) cudaStreamSynchronize(e->own_stream);
  if (e->rec_stream) {
    cudaStreamSynchronize(e->rec_stream);
    cudaStreamDestroy(e->rec_stream);
  }
  if (e->wb_stream) {
    cudaStreamSynchronize(e->wb_stream);
    cudaStreamDestroy(e->wb_stream);
  }
  if (e->ev_in) cudaEventDestroy(e->ev_in);
  if (e->ev_wb) cudaEventDestroy(e->ev_wb);
  for (int i = 0; i < sdr_engine::RING_MAX; ++i) {
    if (e->ev_fir[i]) cudaEventDestroy(e->ev_fir[i]);
    if (e->ev_rec[i]) cudaEventDestroy(e->ev_rec[i]);
  }
  for (int i = 0; i < sdr_engine::PACE; ++i)
    if (e->ev_pace[i]) cudaEventDestroy(e->ev_pace[i]);
  for (int k = 1; k <= 4; ++k) {
    for (int i = 0; i < sdr_engine::RING_MAX; ++i) cudaFree(e->d_scratch[k][i]);
    cudaFree(e->d_state[k]);
    cudaFree(e->d_scale[k]);
    cudaFree(e->d_list[k]);
  }
  cudaFree(e->d_threshold);
  cudaFree(e->d_rx_gain);
  cudaFree(e->d_magnitude);
  cudaFree(e->d_tracking);
  cudaFree(e->d_dump);
  cudaFree(e->d_dump_list);
  cudaFree(e->d_allowed);
  cudaFree(e->d_db_table);
  cudaFree(e->d_lsb);
  cudaFree(e->d_lut_fm);
  cudaFree(e->d_fm_tab);
  cudaFree(e->d_wb_tab);
  cudaFree(e->d_wb4_tab);
  if (e->h_wb_clip) cudaFreeHost((void *)e->h_wb_clip);
  cudaFree(e->d_am_tab);
  cudaFree(e->d_lut_wbfm);
  cudaFree(e->d_lut_wbfm_half);
  cudaFree(e->d_trace);
  cudaFree(e->d_counters);
  cudaFree(e->d_iq);
  cudaFree(e->d_pcm2[0]);
  cudaFree(e->d_pcm2[1]);
  if (e->own_stream) cudaStreamDestroy(e->own_stream);
  delete e;
  return SDR_OK;
}

int sdr_set_stream(sdr_engine *e, void *cuda_stream) {
  if (!e) return SDR_E_ARG;
  SDR_CK(e, cudaStreamSynchronize(e->stream));
  SDR_CK(e, cudaStreamSynchronize(e->rec_stream));
  SDR_CK(e, cudaStreamSynchronize(e->wb_stream));
  e->rec_pending = false;
  e->wb_pending = false;
  e->stream = cuda_stream ? (cudaStream_t)cuda_stream : e->own_stream;
  return SDR_OK;
}

int sdr_set_scaling(sdr_engine *e, int scaling) {
  if (!e || (scaling != SDR_SCALING_RADIODIAGS && scaling != SDR_SCALING_RESEARCH)) return SDR_E_ARG;
  // the two trees also differ in the WBFM constructor gain; channels still at
  // the old default follow the tree
  const float old_def = default_gain(SDR_KIND_WBFM, e->scaling), new_def = default_gain(SDR_KIND_WBFM, scaling);
  for (auto &g : e->gain[SDR_KIND_WBFM])
    if (g == old_def) g = new_def;
  e->scaling = scaling;
  e->scale_dirty[SDR_KIND_FM] = e->scale_dirty[SDR_KIND_WBFM] = true;
  return SDR_OK;
}

int sdr_set_mode(sdr_engine *e, uint32_t ch, int mode) {
  if (!e || ch >= e->n || mode < SDR_MODE_NONE || mode > SDR_MODE_USB) return SDR_E_ARG;
  if (e->mode[ch] != mode) {
    e->mode[ch] = (uint8_t)mode;
    e->lists_dirty = true;
  }
  // IqDataProcessor.cc:247-258: selecting Lsb/Usb also flips the SSB object's sideband
  if (mode == SDR_MODE_LSB && !e->lsb[ch]) { e->lsb[ch] = 1; e->lsb_dirty = true; }
  if (mode == SDR_MODE_USB && e->lsb[ch]) { e->lsb[ch] = 0; e->lsb_dirty = true; }
  return SDR_OK;
}

int sdr_set_modes(sdr_engine *e, const uint8_t *modes) {
  if (!e || !modes) return SDR_E_ARG;
  for (uint32_t ch = 0; ch < e->n; ++ch)
    if (modes[ch] > SDR_MODE_USB) return SDR_E_ARG;
  for (uint32_t ch = 0; ch < e->n; ++ch) sdr_set_mode(e, ch, modes[ch]);
  return SDR_OK;
}

int sdr_set_gain(sdr_engine *e, uint32_t ch, int kind, float gain) {
  if (!e || ch >= e->n || kind < SDR_KIND_AM || kind > SDR_KIND_SSB) return SDR_E_ARG;
  e->gain[kind][ch] = gain;
  e->scale_dirty[kind] = true;
  return SDR_OK;
}

int sdr_set_gain_all(sdr_engine *e, int kind, float gain) {
  if (!e || kind < SDR_KIND_AM || kind > SDR_KIND_SSB) return SDR_E_ARG;
  e->gain[kind].assign(e->n, gain);
  e->scale_dirty[kind] = true;
  return SDR_OK;
}

int sdr_reset(sdr_engine *e, uint32_t ch, int kind) {
  if (!e || ch >= e->n || kind < SDR_KIND_AM || kind > SDR_KIND_SSB) return SDR_E_ARG;
  SDR_CK(e, cudaSetDevice(e->device));
  {
    int rc = join_streams(e);  // a recurrence kernel may still be updating this blob
    if (rc) return rc;
  }
  size_t sb = (size_t)state_bytes(kind), n = sb;
  // WbFmDemodulator::resetDemodulator leaves the de-emphasis IIR alone
  // (WbFmDemodulator.cc:304-320); its state is the last 16 bytes of the blob.
  if (kind == SDR_KIND_WBFM) n -= 16;
  SDR_CK(e, cudaMemsetAsync(e->d_state[kind] + sb * ch, 0, n, e->stream));
  return SDR_OK;
}

int sdr_set_launch_shape(sdr_engine *e, int kind, uint32_t G, uint32_t NT) {
  if (!e || kind < SDR_KIND_AM || kind > SDR_KIND_SSB || G > (uint32_t)MAX_G || NT > 1024 || NT % 32)
    return SDR_E_ARG;
  e->shape[kind].G = G;
  e->shape[kind].NT = NT;
  return SDR_OK;
}

uint64_t sdr_launch_count(const sdr_engine *e) { return e ? e->launches : 0; }

// Diagnostics (not part of include/sdr_b200.h): the launch timeline recorded under SDR_TRACE=1,
// [call % 4096][FIR start, FIR end, dc_block start, dc_block end] in globaltimer ns.
int sdr_debug_read_trace(sdr_engine *e, unsigned long long *out, uint64_t n_calls) {
  if (!e || !e->d_trace || !out || n_calls > sdr_engine::TRACE_CALLS) return SDR_E_ARG;
  SDR_CK(e, cudaSetDevice(e->device));
  SDR_CK(e, cudaDeviceSynchronize());
  SDR_CK(e, cudaMemcpy(out, e->d_trace, n_calls * 32, cudaMemcpyDeviceToHost));
  return SDR_OK;
}

// Diagnostics (not part of include/sdr_b200.h): dc_block_kernel's segmentation -- seg_count 0 =
// chosen per call, else a power of two <= 32; warm_rows = rows of 32 PCM samples a segment warms
// up on -- and how many segments it had to redo serially so far. Tests shrink the warm-up to
// force the redo path.
int sdr_debug_set_dc_shape(sdr_engine *e, uint32_t seg_count, uint32_t warm_rows) {
  if (!e || seg_count > 32 || (seg_count & (seg_count - 1))) return SDR_E_ARG;
  e->dc_seg_count = seg_count;
  e->dc_warm_rows = warm_rows;
  return SDR_OK;
}

// which generation of the WBFM kernel runs (0 = default); the three share the carry blob, so a test
// may switch between calls
// 4 = the pre-filter on the tcgen05 tensor cores (5, 6: with two / one channel(s) per worker warp whatever the
// bank's size); + 16: generations 2 and 3 with the pre-filter on the legacy mma.sync path (WbMma)
int sdr_debug_set_wbfm_kernel(sdr_engine *e, int generation) {
  if (!e || generation < 0 || (generation & ~16) > 6 || ((generation & 16) && (generation & ~16) > 3)) return SDR_E_ARG;
  // 5, 6: generation 4 with two / one channel(s) per worker warp whatever the bank's size
  e->wb4_geometry = (generation & ~16) > 4 ? (generation & ~16) - 4 : 0;
  e->wb_kernel = std::min(generation & ~16, 4);
  e->wb_prefilter_mma = (generation & 16) != 0;
  return SDR_OK;
}

// wb_umma_table() and the accumulator starts for the CPU-side check of the tcgen05 formulation
// (tests/test_wb_umma_table.py): 4096 bytes of tap matrices; starts[2 p + arm] for p = 0..3
int sdr_debug_wb_umma_table(uint8_t *taps_out, int32_t *starts_out) {
  if (!taps_out || !starts_out) return SDR_E_ARG;
  const std::vector<uint8_t> tab = wb_umma_table();
  memcpy(taps_out, tab.data(), tab.size());
  for (int pp = 0; pp < 4; ++pp)
    for (int arm = 0; arm < 2; ++arm) starts_out[2 * pp + arm] = WbUmma::start_of(pp, arm);
  return (int)tab.size();
}

// wb_mma_table() for the CPU-side check of the tensor-core formulation (tests/test_wb_mma_table.py)
int sdr_debug_wb_mma_table(uint32_t *out) {
  if (!out) return SDR_E_ARG;
  const std::vector<uint32_t> tab = wb_mma_table();
  memcpy(out, tab.data(), tab.size() * 4);
  return (int)tab.size();
}

// am_mma_table() for the CPU-side check of the tensor-core formulation (tests/test_am_mma_table.py):
// 2 formats x 32 lanes x 12 words
int sdr_debug_am_mma_table(uint32_t *out) {
  if (!out) return SDR_E_ARG;
  const std::vector<uint32_t> tab = am_mma_table();
  memcpy(out, tab.data(), tab.size() * 4);
  return (int)tab.size();
}

// how the AM/SSB FIR kernel fetches full tiles: 0 = cp.async with two slot buffers per warp,
// 2 / 3 / 4 = TMA with that many (1 = the default: TMA, two buffers); + 8 = stage 1 on the tensor
// cores (TMA loaders only; default: CUDA cores); + 16 = the 80-register build, six CTAs per SM
// (stage 1 on the CUDA cores only). For A/B runs and tests.
int sdr_debug_set_tile_loader(sdr_engine *e, int loader) {
  if (!e || loader < 0 || (loader & 7) > 4 || loader > 31) return SDR_E_ARG;
  e->stage1_mma = (loader & 8) != 0 && (loader & 7) != 0;
  e->fir_ctas_per_sm = (loader & 16) ? 6 : 5;
  loader &= 7;
  e->tile_loader = loader == 1 ? 2 : loader;
  return SDR_OK;
}

// (half-)tiles whose WBFM pre-filter ran on the tensor cores / on the CUDA cores since the first call of this
// function (which switches the counting on)
int sdr_debug_wb_prefilter_counts(sdr_engine *e, uint32_t *mma, uint32_t *simt) {
  if (!e || !mma || !simt) return SDR_E_ARG;
  e->wb_count = true;
  SDR_CK(e, cudaSetDevice(e->device));
  int rc = join_streams(e);
  if (rc) return rc;
  uint32_t c[4] = {};
  SDR_CK(e, cudaMemcpyAsync(c, e->d_counters, 16, cudaMemcpyDeviceToHost, e->stream));
  SDR_CK(e, cudaStreamSynchronize(e->stream));
  *mma = c[1];
  *simt = c[2];
  return SDR_OK;
}

int sdr_debug_dc_redo_count(sdr_engine *e, uint32_t *count) {
  if (!e || !count) return SDR_E_ARG;
  SDR_CK(e, cudaSetDevice(e->device));
  int rc = join_streams(e);
  if (rc) return rc;
  SDR_CK(e, cudaMemcpyAsync(count, e->d_counters, 4, cudaMemcpyDeviceToHost, e->stream));
  SDR_CK(e, cudaStreamSynchronize(e->stream));
  return SDR_OK;
}

}  // extern "C"

namespace {
int accept_iq(sdr_engine *e, const void *iq, uint64_t bytes, uint64_t ch_stride, uint32_t flags);
int wait_pass_slot(sdr_engine *e);
int demodulate_pass(sdr_engine *e, const uint8_t *iq, uint64_t stride, uint32_t n_samples, int fmt, bool have_rec);
int poisoned(sdr_engine *e) {
  e->err = "the engine is in a failed state after: " + e->poison_text;
  return SDR_E_CUDA;
}
}  // namespace

extern "C" {

int sdr_accept_iq(sdr_engine *e, const void *iq, uint64_t bytes, uint64_t ch_stride, uint32_t flags) {
  if (!e || !iq) return SDR_E_ARG;
  if (e->poisoned) return poisoned(e);
  const uint64_t launches_before = e->launches;
  const int rc = accept_iq(e, iq, bytes, ch_stride, flags);
  // an argument error queues nothing and leaves the engine usable; a failure after the first
  // launch leaves ring slots and events half used
  if (rc != SDR_OK && (rc == SDR_E_CUDA || e->launches != launches_before)) {
    e->poisoned = true;
    e->poison_text = e->err;
  }
  return rc;
}

}  // extern "C"

namespace {
int accept_iq(sdr_engine *e, const void *iq, uint64_t bytes, uint64_t ch_stride, uint32_t flags) {
  if (bytes == 0 || bytes % 64) return fail(e, SDR_E_ARG, "bytes_per_channel must be a positive multiple of 64");
  if (bytes > e->max_bytes) return fail(e, SDR_E_TOO_LONG, "bytes_per_channel exceeds max_bytes_per_channel");
  if (ch_stride < bytes || ch_stride % 16 || ((uintptr_t)iq & 15))
    return fail(e, SDR_E_ARG, "iq pointer and channel_stride must be multiples of 16, stride >= bytes");
  SDR_CK(e, cudaSetDevice(e->device));
  int rc = upload_tables(e);
  if (rc) return rc;
  // the previous call's WBFM kernel may still be reading the input buffer this call refills
  if (e->wb_pending) {
    SDR_CK(e, cudaStreamWaitEvent(e->stream, e->ev_wb, 0));
    e->wb_pending = false;
  }
  const uint8_t *dev_iq = (const uint8_t *)iq;
  uint64_t dev_stride = ch_stride;
  if (!(flags & SDR_IQ_DEVICE)) {
    if (!e->d_iq) SDR_CK(e, cudaMalloc(&e->d_iq, (size_t)e->n * e->max_bytes));
    SDR_CK(e, cudaMemcpy2DAsync(e->d_iq, bytes, iq, ch_stride, bytes, e->n, cudaMemcpyHostToDevice, e->stream));
    dev_iq = e->d_iq;
    dev_stride = bytes;
  }
  // Bounded run-ahead. With hundreds of calls queued the driver's launch queues fill up and the
  // GPU is fed in bursts (profiles/r01v7_pacing.txt); holding the caller once RUN_AHEAD calls are
  // in flight keeps the queues shallow.
  // (An event every fourth call: the bound is then RUN_AHEAD .. RUN_AHEAD + 3 calls, and three of
  // four calls queue one stream operation less.)
  const int slot = (int)((e->seq / 4) % (uint64_t)sdr_engine::PACE);
  if (e->seq % 4 == 0 && e->seq >= (uint64_t)sdr_engine::RUN_AHEAD)
    SDR_CK(e, cudaEventSynchronize(e->ev_pace[(int)(((e->seq - (uint64_t)sdr_engine::RUN_AHEAD) / 4) % (uint64_t)sdr_engine::PACE)]));
  const int fmt = (flags & SDR_IQ_S8_ROTATED) ? FMT_S8_ROTATED : FMT_U8_OFFSET_ROTATE;
  const bool have_rec = !e->list[SDR_KIND_AM].empty() || !e->list[SDR_KIND_SSB].empty();
  // scratch[par] was last read by the recurrence kernels RING passes ago, and the gate entry this
  // call's squelch writes by those of the call RING calls ago, whose passes are all at least RING
  // passes old (usually long over: then no wait is queued at all)
  if (have_rec || e->squelch_armed || e->signal_reports || e->squelch_dirty) {
    if ((rc = wait_pass_slot(e))) return rc;
  }
  if ((rc = run_iq_dump(e, dev_iq, dev_stride, bytes, fmt))) return rc;
  if ((rc = run_squelch(e, dev_iq, dev_stride, bytes, fmt))) return rc;
  const uint32_t n_blocks = squelch_blocks(e, bytes);
  e->last_blocks = n_blocks;
  e->last_block_bytes = e->squelch_block ? e->squelch_block : bytes;
  // While a gate is in force and the call holds several blocks, each block is its own pass: the
  // same launches as a call of that block alone, reading the block's bytes, gated by its row and
  // writing its PCM columns. Otherwise (reports only: every gate open) the call is one pass.
  const bool split = e->last_gated && e->squelch_armed && n_blocks > 1;
  const uint32_t passes = split ? n_blocks : 1;
  const uint64_t pass_bytes = split ? e->squelch_block : bytes;
  for (uint32_t k = 0; k < passes; ++k) {
    const uint64_t off = (uint64_t)k * pass_bytes;
    const uint64_t len = std::min(pass_bytes, bytes - off);
    if (k > 0 && have_rec && (rc = wait_pass_slot(e))) return rc;
    // Gate row k of this call's entry stays alive until its last reader, the recurrence kernel
    // of pass k, is over: the entry is rewritten by the squelch of call seq + RING, which is
    // queued after wait_pass_slot made `stream` wait for every pass at least RING passes old,
    // and every pass of this call is that old by then (each call has at least one pass).
    e->pass_allowed = e->last_gated ? e->allowed_of(e->seq) + (size_t)k * e->n : nullptr;
    e->pass_pcm = e->pcm_of(e->seq) + off / 64;
    if ((rc = demodulate_pass(e, dev_iq + off, dev_stride, (uint32_t)(len / 2), fmt, have_rec))) return rc;
  }
  if (split) {
    // the open blocks' PCM to the front of each row, once every pass has written its columns
    if ((rc = join_streams(e))) return rc;
    CompactParams c;
    c.pcm = e->pcm_of(e->seq);
    c.pcm_stride = e->pcm_stride;
    c.allowed = e->allowed_of(e->seq);
    c.n_channels = e->n;
    c.n_blocks = n_blocks;
    c.block_samples = (uint32_t)(e->squelch_block / 64);
    c.last_samples = (uint32_t)((bytes - (uint64_t)(n_blocks - 1) * e->squelch_block) / 64);
    pcm_compact_kernel<<<e->n, 256, 0, e->stream>>>(c);
    SDR_CK(e, cudaGetLastError());
    e->launches++;
  }
  if (e->seq % 4 == 0) SDR_CK(e, cudaEventRecord(e->ev_pace[slot], e->stream));
  e->seq++;
  e->last_samples = (uint32_t)(bytes / 64);
  return SDR_OK;
}

// `stream` waits for the recurrence kernels of the pass RING passes before the next one
int wait_pass_slot(sdr_engine *e) {
  const int par = (int)(e->pass % (uint64_t)e->ring);
  if (cudaEventQuery(e->ev_rec[par]) != cudaSuccess) {
    (void)cudaGetLastError();  // "not ready" is an answer, not an error to be found later
    SDR_CK(e, cudaStreamWaitEvent(e->stream, e->ev_rec[par], 0));
  }
  return SDR_OK;
}

// One demodulation pass over n_samples of every channel from iq, into e->pass_pcm, gated by
// e->pass_allowed.
int demodulate_pass(sdr_engine *e, const uint8_t *iq, uint64_t stride, uint32_t n_samples, int fmt, bool have_rec) {
  int rc;
  const int par = (int)(e->pass % (uint64_t)e->ring);
  // WBFM first, and beside the others when there are others: its CTAs (one per SM for the whole
  // launch) take their place on every SM, the short-lived CTAs of the other kinds flow around them
  static const int wb_split_env = getenv("SDR_WB_SPLIT") ? atoi(getenv("SDR_WB_SPLIT")) : 1;
  const bool wb_beside = wb_split_env && !e->list[SDR_KIND_WBFM].empty() &&
                         (have_rec || !e->list[SDR_KIND_FM].empty());
  if (wb_beside) {
    SDR_CK(e, cudaEventRecord(e->ev_in, e->stream));
    SDR_CK(e, cudaStreamWaitEvent(e->wb_stream, e->ev_in, 0));
    if ((rc = launch_wbfm_tile(e, iq, stride, n_samples, fmt, e->wb_stream))) return rc;
    SDR_CK(e, cudaEventRecord(e->ev_wb, e->wb_stream));
    e->wb_pending = true;
  }
  if ((rc = launch_amssb<false>(e, SDR_KIND_AM, iq, stride, n_samples, fmt))) return rc;
  if ((rc = launch_amssb<true>(e, SDR_KIND_SSB, iq, stride, n_samples, fmt))) return rc;
  if (have_rec) {
    SDR_CK(e, cudaEventRecord(e->ev_fir[par], e->stream));
    SDR_CK(e, cudaStreamWaitEvent(e->rec_stream, e->ev_fir[par], 0));
    if ((rc = launch_dc_block(e, SDR_KIND_AM, n_samples))) return rc;
    if ((rc = launch_dc_block(e, SDR_KIND_SSB, n_samples))) return rc;
  }
  // always recorded, so ev_rec[par] of the latest pass orders after everything on rec_stream
  SDR_CK(e, cudaEventRecord(e->ev_rec[par], e->rec_stream));
  e->rec_pending = true;
  if ((rc = launch_fm_tile(e, iq, stride, n_samples, fmt))) return rc;
  if (!wb_beside && (rc = launch_wbfm_tile(e, iq, stride, n_samples, fmt, e->stream))) return rc;
  e->pass++;
  return SDR_OK;
}
}  // namespace

extern "C" {

int sdr_get_pcm(sdr_engine *e, int16_t *pcm, uint32_t *counts) {
  if (!e) return SDR_E_ARG;
  if (e->poisoned) return poisoned(e);
  SDR_CK(e, cudaSetDevice(e->device));
  {
    int rc = join_streams(e);
    if (rc) return rc;
  }
  if (pcm && e->last_samples)
    SDR_CK(e, cudaMemcpy2DAsync(pcm, (size_t)e->last_samples * 2, e->pcm_of(e->seq - 1), e->pcm_stride * 2,
                                (size_t)e->last_samples * 2, e->n, cudaMemcpyDeviceToHost, e->stream));
  std::vector<uint8_t> gate;
  if (counts && e->last_gated && e->seq > 0) {
    gate.resize((size_t)e->last_blocks * e->n);
    SDR_CK(e, cudaMemcpyAsync(gate.data(), e->allowed_of(e->seq - 1), gate.size(), cudaMemcpyDeviceToHost, e->stream));
  }
  SDR_CK(e, cudaStreamSynchronize(e->stream));
  if (counts)
    for (uint32_t ch = 0; ch < e->n; ++ch)
      counts[ch] = e->mode[ch] == SDR_MODE_NONE ? 0
                   : gate.empty() ? e->last_samples
                                  : open_samples(gate.data(), e->n, ch, e->last_blocks, e->last_block_bytes,
                                                 (uint64_t)e->last_samples * 64);
  return SDR_OK;
}

int sdr_pcm_device(sdr_engine *e, int16_t **pcm, uint64_t *stride) {
  if (!e) return SDR_E_ARG;
  if (pcm) *pcm = e->pcm_of(e->seq ? e->seq - 1 : 0);  // the buffer of the last accept
  if (stride) *stride = e->pcm_stride;
  return SDR_OK;
}

int sdr_set_squelch_threshold(sdr_engine *e, uint32_t ch, int32_t threshold_dbfs) {
  if (!e || ch >= e->n) return SDR_E_ARG;
  e->threshold[ch] = threshold_dbfs;
  e->squelch_dirty = true;
  return SDR_OK;
}

int sdr_set_receive_gain_db(sdr_engine *e, uint32_t ch, uint32_t gain_db) {
  if (!e || ch >= e->n) return SDR_E_ARG;
  e->rx_gain_db[ch] = gain_db;
  e->squelch_dirty = true;
  return SDR_OK;
}

int sdr_enable_signal_reports(sdr_engine *e, int on) {
  if (!e) return SDR_E_ARG;
  e->signal_reports = on != 0;
  e->squelch_dirty = true;
  return SDR_OK;
}

int sdr_get_signal(sdr_engine *e, uint8_t *allowed, uint32_t *magnitude) {
  if (!e) return SDR_E_ARG;
  if (!e->last_gated || e->seq == 0) return fail(e, SDR_E_ARG, "no squelch result: set a threshold or enable signal reports first");
  SDR_CK(e, cudaSetDevice(e->device));
  const size_t last = (size_t)(e->last_blocks - 1) * e->n;  // the last block's row
  if (allowed)
    SDR_CK(e, cudaMemcpyAsync(allowed, e->allowed_of(e->seq - 1) + last, e->n, cudaMemcpyDeviceToHost, e->stream));
  if (magnitude)
    SDR_CK(e, cudaMemcpyAsync(magnitude, e->magnitude_of(e->seq - 1) + last, (size_t)e->n * 4, cudaMemcpyDeviceToHost, e->stream));
  SDR_CK(e, cudaStreamSynchronize(e->stream));
  return SDR_OK;
}

int sdr_set_squelch_block_bytes(sdr_engine *e, uint64_t block_bytes) {
  if (!e) return SDR_E_ARG;
  if (block_bytes % 2048 || block_bytes > e->max_bytes)
    return fail(e, SDR_E_ARG, "squelch block must be 0 or a multiple of 2048 within max_bytes_per_channel");
  e->squelch_block = block_bytes;
  return SDR_OK;
}

int sdr_get_signal_blocks(sdr_engine *e, uint8_t *allowed, uint32_t *magnitude, uint32_t *n_blocks) {
  if (!e) return SDR_E_ARG;
  if (!e->last_gated || e->seq == 0) return fail(e, SDR_E_ARG, "no squelch result: set a threshold or enable signal reports first");
  if (n_blocks) *n_blocks = e->last_blocks;
  if (!allowed && !magnitude) return SDR_OK;
  SDR_CK(e, cudaSetDevice(e->device));
  const size_t cells = (size_t)e->last_blocks * e->n;
  if (allowed) SDR_CK(e, cudaMemcpyAsync(allowed, e->allowed_of(e->seq - 1), cells, cudaMemcpyDeviceToHost, e->stream));
  if (magnitude)
    SDR_CK(e, cudaMemcpyAsync(magnitude, e->magnitude_of(e->seq - 1), cells * 4, cudaMemcpyDeviceToHost, e->stream));
  SDR_CK(e, cudaStreamSynchronize(e->stream));
  return SDR_OK;
}

int sdr_set_iq_dump(sdr_engine *e, uint32_t ch, int on) {
  if (!e || ch >= e->n) return SDR_E_ARG;
  if (e->dump_on[ch] != (uint8_t)(on != 0)) {
    e->dump_on[ch] = on != 0;
    if (on) e->dump_count++;
    else e->dump_count--;
    e->dump_dirty = true;
  }
  return SDR_OK;
}

int sdr_get_iq_dump(sdr_engine *e, uint32_t ch, int8_t *out, uint64_t capacity, uint64_t *n_bytes) {
  if (!e || ch >= e->n) return SDR_E_ARG;
  if (n_bytes) *n_bytes = 0;
  auto it = std::lower_bound(e->dump_list.begin(), e->dump_list.end(), ch);
  if (e->dump_dirty || it == e->dump_list.end() || *it != ch || e->dump_bytes == 0)
    return fail(e, SDR_E_ARG, "no IQ dump for this channel: enable it before the call whose block is wanted");
  if (out && capacity < e->dump_bytes) return fail(e, SDR_E_ARG, "IQ dump buffer too small");
  SDR_CK(e, cudaSetDevice(e->device));
  if (out) {
    SDR_CK(e, cudaMemcpyAsync(out, e->dump_of(e->seq - 1) + (size_t)(it - e->dump_list.begin()) * e->max_bytes, e->dump_bytes,
                              cudaMemcpyDeviceToHost, e->stream));
    SDR_CK(e, cudaStreamSynchronize(e->stream));
  }
  if (n_bytes) *n_bytes = e->dump_bytes;
  return SDR_OK;
}

int sdr_iq_dump_device(sdr_engine *e, int8_t **rows, uint64_t *row_stride, uint32_t *n_rows) {
  if (!e) return SDR_E_ARG;
  if (rows) *rows = e->d_dump ? e->dump_of(e->seq ? e->seq - 1 : 0) : nullptr;  // the entry of the last call
  if (row_stride) *row_stride = e->max_bytes;
  if (n_rows) *n_rows = e->dump_bytes ? (uint32_t)e->dump_list.size() : 0;
  return SDR_OK;
}

int sdr_join(sdr_engine *e) {
  if (!e) return SDR_E_ARG;
  return join_streams(e);
}

int sdr_sync(sdr_engine *e) {
  if (!e) return SDR_E_ARG;
  int rc = join_streams(e);
  if (rc) return rc;
  SDR_CK(e, cudaStreamSynchronize(e->stream));
  return SDR_OK;
}

// ---------------------------------------------------------------------------
// Ingest ring: the bank's DataConsumer (DataConsumer.cc:220-352). The reference copies each
// block into one of its message buffers and hands it to the consumer thread; here a block of
// every channel (a tick) is copied into a pinned slot, and the slot's host->device copy,
// demodulation and PCM device->host copy are queued on three streams, so the copy of tick
// k+1 overlaps the demodulation of tick k and the PCM read-back of tick k-1.
// ---------------------------------------------------------------------------
struct sdr_ingest {
  struct Slot {
    uint8_t *h_iq = nullptr, *d_iq = nullptr;
    int16_t *h_pcm = nullptr;
    uint8_t *h_gate = nullptr;
    uint32_t *h_magnitude = nullptr;
    int8_t *h_dump = nullptr;    // [dump_cap][block_bytes], grown at commit time
    uint32_t dump_cap = 0;
    uint32_t sig_cap = 1;        // block rows h_gate and h_magnitude hold, grown at commit time
    cudaEvent_t ev_h2d = nullptr, ev_comp = nullptr, ev_done = nullptr;
    bool own_host = true;        // false: h_iq belongs to a bank's shared tick array
    // where this tick's PCM, gate, magnitudes and dump rows were copied to: the slot's own arrays,
    // or a bank's shared ones
    int16_t *pcm_dst = nullptr;
    uint8_t *gate_dst = nullptr;
    uint32_t *mag_dst = nullptr;
    int8_t *dump_dst = nullptr;
    uint32_t timestamp = 0;
    uint64_t bytes = 0;
    // the tick's squelch blocks: n_blocks rows of gates and magnitudes, sig_pitch channels apart at
    // gate_dst / mag_dst, for blocks of sig_block bytes (the last one shorter)
    uint32_t n_blocks = 1;
    uint64_t sig_pitch = 0, sig_block = 0;
    bool gated = false, queued = false;  // gated: the squelch ran for this tick
    std::vector<uint8_t> mode;
    std::vector<uint32_t> counts;
    std::vector<uint32_t> dump_channels;  // the dumped channels, ascending; their rows are block_bytes apart
  };
  sdr_engine *e = nullptr;
  uint64_t block_bytes = 0;
  std::vector<Slot> slot;
  uint32_t head = 0, tail = 0, in_flight = 0;
  int prev = -1, prev2 = -1; // the slots of the last two ticks (see sdr_ingest_commit)
  int retired = -1;          // the slot of the last retired tick
  cudaStream_t h2d = nullptr, d2h = nullptr;
  uint32_t last_timestamp = 0, short_blocks = 0;
  uint64_t ticks = 0;
};

int sdr_ingest_destroy(sdr_ingest *q) {
  if (!q) return SDR_E_ARG;
  cudaSetDevice(q->e->device);
  if (q->h2d) cudaStreamSynchronize(q->h2d);
  cudaStreamSynchronize(q->e->stream);
  if (q->d2h) cudaStreamSynchronize(q->d2h);
  for (auto &s : q->slot) {
    if (s.own_host) cudaFreeHost(s.h_iq);
    cudaFreeHost(s.h_pcm);
    cudaFreeHost(s.h_gate);
    cudaFreeHost(s.h_magnitude);
    cudaFreeHost(s.h_dump);
    cudaFree(s.d_iq);
    if (s.ev_h2d) cudaEventDestroy(s.ev_h2d);
    if (s.ev_comp) cudaEventDestroy(s.ev_comp);
    if (s.ev_done) cudaEventDestroy(s.ev_done);
  }
  if (q->h2d) cudaStreamDestroy(q->h2d);
  if (q->d2h) {
    if (q->e->dump_reader == q->d2h) q->e->dump_reader = nullptr;
    cudaStreamDestroy(q->d2h);
  }
  delete q;
  return SDR_OK;
}

}  // extern "C"

namespace {
// host_iq: null, or n_slots pointers to pinned [n_channels][block_bytes] arrays the slots use instead
// of their own (a bank's shared tick arrays; then no per-slot PCM, gate, magnitude or dump array is
// allocated either)
int ingest_create(sdr_engine *e, uint32_t n_slots, uint64_t block_bytes, uint8_t *const *host_iq, sdr_ingest **out);
// pcm_dst, gate_dst, mag_dst, dump_dst: null (the slot's own arrays), or where a bank gathers this
// shard's PCM rows, gates, magnitudes and dump rows (block rows of gates and magnitudes sig_pitch
// channels apart, dump rows block_bytes apart)
int ingest_commit(sdr_ingest *q, uint32_t timestamp, uint64_t bytes, uint32_t flags, int16_t *pcm_dst,
                  uint8_t *gate_dst, uint32_t *mag_dst, uint64_t sig_pitch, int8_t *dump_dst);
}  // namespace

extern "C" {

int sdr_ingest_create(sdr_engine *e, uint32_t n_slots, uint64_t block_bytes, sdr_ingest **out) {
  return ingest_create(e, n_slots, block_bytes, nullptr, out);
}

}  // extern "C"

namespace {
int ingest_create(sdr_engine *e, uint32_t n_slots, uint64_t block_bytes, uint8_t *const *host_iq, sdr_ingest **out) {
  if (!e || !out || n_slots < 2 || n_slots > 64) return SDR_E_ARG;
  if (block_bytes == 0 || block_bytes % 64 || block_bytes > e->max_bytes)
    return fail(e, SDR_E_ARG, "ingest block_bytes must be a multiple of 64 within max_bytes_per_channel");
  SDR_CK(e, cudaSetDevice(e->device));
  sdr_ingest *q = new (std::nothrow) sdr_ingest();
  if (!q) return SDR_E_NOMEM;
  q->e = e;
  q->block_bytes = block_bytes;
  q->slot.resize(n_slots);
#define SDR_CK_Q(call)                                 \
  do {                                                 \
    cudaError_t _ce = (call);                          \
    if (_ce != cudaSuccess) {                          \
      fail(e, SDR_E_CUDA, #call, _ce);                 \
      sdr_ingest_destroy(q);                           \
      return SDR_E_CUDA;                               \
    }                                                  \
  } while (0)
  SDR_CK_Q(cudaStreamCreateWithFlags(&q->h2d, cudaStreamNonBlocking));
  SDR_CK_Q(cudaStreamCreateWithFlags(&q->d2h, cudaStreamNonBlocking));
  e->dump_reader = q->d2h;
  const size_t iq_bytes = (size_t)e->n * block_bytes, pcm_bytes = (size_t)e->n * (block_bytes / 64) * 2;
  for (uint32_t i = 0; i < n_slots; ++i) {
    sdr_ingest::Slot &s = q->slot[i];
    if (host_iq) {
      s.h_iq = host_iq[i];
      s.own_host = false;
    } else {
      SDR_CK_Q(cudaHostAlloc(&s.h_iq, iq_bytes, cudaHostAllocDefault));
      SDR_CK_Q(cudaHostAlloc(&s.h_pcm, pcm_bytes, cudaHostAllocDefault));
      SDR_CK_Q(cudaHostAlloc(&s.h_gate, e->n, cudaHostAllocDefault));
      SDR_CK_Q(cudaHostAlloc(&s.h_magnitude, (size_t)e->n * 4, cudaHostAllocDefault));
    }
    SDR_CK_Q(cudaMalloc(&s.d_iq, iq_bytes));
    SDR_CK_Q(cudaEventCreateWithFlags(&s.ev_h2d, cudaEventDisableTiming));
    SDR_CK_Q(cudaEventCreateWithFlags(&s.ev_comp, cudaEventDisableTiming));
    SDR_CK_Q(cudaEventCreateWithFlags(&s.ev_done, cudaEventDisableTiming));
    s.counts.assign(e->n, 0);
  }
#undef SDR_CK_Q
  *out = q;
  return SDR_OK;
}
}  // namespace

extern "C" {

int sdr_ingest_acquire(sdr_ingest *q, void **iq, uint64_t *channel_stride) {
  if (!q || !iq) return SDR_E_ARG;
  sdr_ingest::Slot &s = q->slot[q->head];
  if (s.queued) return fail(q->e, SDR_E_FULL, "ingest ring full: retire a tick first");
  *iq = s.h_iq;
  if (channel_stride) *channel_stride = q->block_bytes;
  return SDR_OK;
}

int sdr_ingest_commit(sdr_ingest *q, uint32_t timestamp, uint64_t bytes, uint32_t flags) {
  return ingest_commit(q, timestamp, bytes, flags, nullptr, nullptr, nullptr, 0, nullptr);
}

}  // extern "C"

namespace {
int ingest_commit(sdr_ingest *q, uint32_t timestamp, uint64_t bytes, uint32_t flags, int16_t *pcm_dst,
                  uint8_t *gate_dst, uint32_t *mag_dst, uint64_t sig_pitch, int8_t *dump_dst) {
  if (!q) return SDR_E_ARG;
  sdr_engine *e = q->e;
  sdr_ingest::Slot &s = q->slot[q->head];
  if (s.queued) return fail(e, SDR_E_FULL, "ingest ring full: retire a tick first");
  if (bytes == 0 || bytes % 64) return fail(e, SDR_E_ARG, "bytes_per_channel must be a positive multiple of 64");
  SDR_CK(e, cudaSetDevice(e->device));
  // the slot is free, so no copy of an earlier tick still lands in its dump array
  if (!dump_dst && e->dump_count > s.dump_cap) {
    cudaFreeHost(s.h_dump);
    s.h_dump = nullptr;
    s.dump_cap = 0;
    SDR_CK(e, cudaHostAlloc(&s.h_dump, (size_t)e->dump_count * q->block_bytes, cudaHostAllocDefault));
    s.dump_cap = e->dump_count;
  }
  const uint64_t take = bytes > q->block_bytes ? q->block_bytes : bytes;
  const uint32_t n_blocks = squelch_blocks(e, take);
  if (!gate_dst && n_blocks > s.sig_cap) {  // likewise for the gate and magnitude rows
    cudaFreeHost(s.h_gate);
    cudaFreeHost(s.h_magnitude);
    s.h_gate = nullptr;
    s.h_magnitude = nullptr;
    s.sig_cap = 0;
    SDR_CK(e, cudaHostAlloc(&s.h_gate, (size_t)n_blocks * e->n, cudaHostAllocDefault));
    SDR_CK(e, cudaHostAlloc(&s.h_magnitude, (size_t)n_blocks * e->n * 4, cudaHostAllocDefault));
    s.sig_cap = n_blocks;
  }
  // DataConsumer::acceptData, DataConsumer.cc:232-246: clip to the buffer, count short blocks
  q->last_timestamp = timestamp;
  if (bytes > q->block_bytes) bytes = q->block_bytes;
  else if (bytes < q->block_bytes) q->short_blocks++;
  if (bytes == q->block_bytes)
    SDR_CK(e, cudaMemcpyAsync(s.d_iq, s.h_iq, (size_t)e->n * bytes, cudaMemcpyHostToDevice, q->h2d));
  else
    SDR_CK(e, cudaMemcpy2DAsync(s.d_iq, q->block_bytes, s.h_iq, q->block_bytes, bytes, e->n,
                                cudaMemcpyHostToDevice, q->h2d));
  SDR_CK(e, cudaEventRecord(s.ev_h2d, q->h2d));
  SDR_CK(e, cudaStreamWaitEvent(e->stream, s.ev_h2d, 0));
  // the engine alternates between two PCM buffers: this tick writes the one the tick before the
  // previous one used, so that tick's read-back must be over (the previous tick's may still run)
  if (q->prev2 >= 0) SDR_CK(e, cudaStreamWaitEvent(e->stream, q->slot[q->prev2].ev_done, 0));
  int rc = sdr_accept_iq(e, s.d_iq, bytes, q->block_bytes, SDR_IQ_DEVICE | (flags & SDR_IQ_S8_ROTATED));
  if (rc) return rc;
  if ((rc = join_streams(e))) return rc;
  SDR_CK(e, cudaEventRecord(s.ev_comp, e->stream));
  SDR_CK(e, cudaStreamWaitEvent(q->d2h, s.ev_comp, 0));
  const size_t row = (size_t)(bytes / 64) * 2;
  s.pcm_dst = pcm_dst ? pcm_dst : s.h_pcm;
  SDR_CK(e, cudaMemcpy2DAsync(s.pcm_dst, row, e->pcm_of(e->seq - 1), e->pcm_stride * 2, row, e->n, cudaMemcpyDeviceToHost, q->d2h));
  // the tick's signal reports and IQ dump, from the engine's ring entries of this call (run_iq_dump
  // shows why they are not overwritten before these copies ran)
  s.gated = e->last_gated;
  s.gate_dst = gate_dst ? gate_dst : s.h_gate;
  s.mag_dst = mag_dst ? mag_dst : s.h_magnitude;
  s.sig_pitch = gate_dst ? sig_pitch : e->n;
  s.n_blocks = e->last_blocks;
  s.sig_block = e->last_block_bytes;
  if (s.gated) {  // every block row of the entry, one 2D copy each
    SDR_CK(e, cudaMemcpy2DAsync(s.gate_dst, s.sig_pitch, e->allowed_of(e->seq - 1), e->n, e->n, s.n_blocks,
                                cudaMemcpyDeviceToHost, q->d2h));
    SDR_CK(e, cudaMemcpy2DAsync(s.mag_dst, s.sig_pitch * 4, e->magnitude_of(e->seq - 1), (size_t)e->n * 4,
                                (size_t)e->n * 4, s.n_blocks, cudaMemcpyDeviceToHost, q->d2h));
  }
  s.dump_channels.clear();
  if (e->dump_bytes) s.dump_channels = e->dump_list;
  s.dump_dst = dump_dst ? dump_dst : s.h_dump;
  if (!s.dump_channels.empty())
    SDR_CK(e, cudaMemcpy2DAsync(s.dump_dst, q->block_bytes, e->dump_of(e->seq - 1), e->max_bytes, bytes,
                                s.dump_channels.size(), cudaMemcpyDeviceToHost, q->d2h));
  SDR_CK(e, cudaEventRecord(s.ev_done, q->d2h));
  s.timestamp = timestamp;
  s.bytes = bytes;
  s.mode = e->mode;
  s.queued = true;
  q->prev2 = q->prev;
  q->prev = (int)q->head;
  q->head = (q->head + 1) % (uint32_t)q->slot.size();
  q->in_flight++;
  q->ticks++;
  return SDR_OK;
}
}  // namespace

extern "C" {

int sdr_ingest_accept(sdr_ingest *q, uint32_t timestamp, const void *iq, uint64_t bytes, uint64_t channel_stride,
                      uint32_t flags) {
  if (!q || !iq) return SDR_E_ARG;
  void *dst = nullptr;
  int rc = sdr_ingest_acquire(q, &dst, nullptr);
  if (rc) return rc;
  const uint64_t take = bytes > q->block_bytes ? q->block_bytes : bytes;
  if (channel_stride < take) return fail(q->e, SDR_E_ARG, "channel_stride < bytes_per_channel");
  for (uint32_t ch = 0; ch < q->e->n; ++ch)  // the reference's memcpy into message[].buffer, DataConsumer.cc:251
    memcpy((uint8_t *)dst + (size_t)ch * q->block_bytes, (const uint8_t *)iq + (size_t)ch * channel_stride, take);
  return sdr_ingest_commit(q, timestamp, bytes, flags);
}

int sdr_ingest_retire(sdr_ingest *q, uint32_t *timestamp, const int16_t **pcm, uint32_t *samples_per_row,
                      const uint32_t **counts) {
  if (!q) return SDR_E_ARG;
  sdr_engine *e = q->e;
  sdr_ingest::Slot &s = q->slot[q->tail];
  if (!s.queued) return fail(e, SDR_E_EMPTY, "ingest ring empty: nothing to retire");
  SDR_CK(e, cudaSetDevice(e->device));
  SDR_CK(e, cudaEventSynchronize(s.ev_done));
  const uint32_t samples = (uint32_t)(s.bytes / 64);
  for (uint32_t ch = 0; ch < e->n; ++ch)
    s.counts[ch] = s.mode[ch] == SDR_MODE_NONE ? 0
                   : !s.gated ? samples
                              : open_samples(s.gate_dst, s.sig_pitch, ch, s.n_blocks, s.sig_block, s.bytes);
  if (timestamp) *timestamp = s.timestamp;
  if (pcm) *pcm = s.pcm_dst;
  if (samples_per_row) *samples_per_row = samples;
  if (counts) *counts = s.counts.data();
  s.queued = false;
  q->retired = (int)q->tail;
  q->tail = (q->tail + 1) % (uint32_t)q->slot.size();
  q->in_flight--;
  return SDR_OK;
}

// the slot of the last retired tick, or null if there is none (or its slot was committed again)
static const sdr_ingest::Slot *ingest_retired(const sdr_ingest *q) {
  if (q->retired < 0 || q->slot[q->retired].queued) return nullptr;
  return &q->slot[q->retired];
}

int sdr_ingest_retired_signal(const sdr_ingest *q, const uint8_t **allowed, const uint32_t **magnitude) {
  if (!q) return SDR_E_ARG;
  const sdr_ingest::Slot *s = ingest_retired(q);
  if (!s) return fail(q->e, SDR_E_EMPTY, "no retired tick: retire one first");
  if (!s->gated)
    return fail(q->e, SDR_E_ARG, "the retired tick ran no squelch: set a threshold or enable signal reports before its commit");
  const size_t last = (size_t)(s->n_blocks - 1) * s->sig_pitch;  // the last block's row
  if (allowed) *allowed = s->gate_dst + last;
  if (magnitude) *magnitude = s->mag_dst + last;
  return SDR_OK;
}

int sdr_ingest_retired_signal_blocks(const sdr_ingest *q, const uint8_t **allowed, const uint32_t **magnitude,
                                     uint32_t *n_blocks) {
  if (!q) return SDR_E_ARG;
  const sdr_ingest::Slot *s = ingest_retired(q);
  if (!s) return fail(q->e, SDR_E_EMPTY, "no retired tick: retire one first");
  if (!s->gated)
    return fail(q->e, SDR_E_ARG, "the retired tick ran no squelch: set a threshold or enable signal reports before its commit");
  if (allowed) *allowed = s->gate_dst;
  if (magnitude) *magnitude = s->mag_dst;
  if (n_blocks) *n_blocks = s->n_blocks;
  return SDR_OK;
}

int sdr_ingest_retired_iq_dump(const sdr_ingest *q, const int8_t **rows, uint64_t *row_stride, uint64_t *n_bytes,
                               const uint32_t **channels, uint32_t *n_rows) {
  if (!q) return SDR_E_ARG;
  const sdr_ingest::Slot *s = ingest_retired(q);
  if (!s) return fail(q->e, SDR_E_EMPTY, "no retired tick: retire one first");
  const bool any = !s->dump_channels.empty();
  if (rows) *rows = any ? s->dump_dst : nullptr;
  if (row_stride) *row_stride = q->block_bytes;
  if (n_bytes) *n_bytes = s->bytes;
  if (channels) *channels = any ? s->dump_channels.data() : nullptr;
  if (n_rows) *n_rows = (uint32_t)s->dump_channels.size();
  return SDR_OK;
}

int sdr_ingest_stats(const sdr_ingest *q, uint32_t *last_timestamp, uint32_t *short_block_count, uint64_t *ticks,
                     uint32_t *in_flight) {
  if (!q) return SDR_E_ARG;
  if (last_timestamp) *last_timestamp = q->last_timestamp;
  if (short_block_count) *short_block_count = q->short_blocks;
  if (ticks) *ticks = q->ticks;
  if (in_flight) *in_flight = q->in_flight;
  return SDR_OK;
}


// ---------------------------------------------------------------------------
// Multi-device bank (SURVEY.md section 8e): n_channels radios over the GPUs of one box.
// Channels are independent, so device g simply owns the contiguous range
// [n g / G, n (g + 1) / G): one engine and one ingest ring per device, no exchange between
// devices. What the devices share is host memory: ONE pinned tick array [n_channels][block_bytes]
// per slot that every device host->device-copies its slab out of, and ONE pinned PCM array
// [n_channels][bytes / 64] per slot that every device copies its slab into -- the "gather" is
// where the copies land. One host thread drives all devices: every call below only queues work.
// ---------------------------------------------------------------------------
struct sdr_bank {
  uint32_t n = 0;
  uint64_t block_bytes = 0;
  std::vector<int> device;
  std::vector<uint32_t> first;  // [n_devices + 1]
  std::vector<sdr_engine *> eng;
  std::vector<sdr_ingest *> ing;
  struct Slot {
    uint8_t *h_iq = nullptr;
    int16_t *h_pcm = nullptr;
    // [sig_cap][n_channels]: block row k of every shard's gates and magnitudes lands in its columns
    uint8_t *h_allowed = nullptr;
    uint32_t *h_magnitude = nullptr;
    uint32_t sig_cap = 1, n_blocks = 1;
    int8_t *h_dump = nullptr;       // [dump_cap][block_bytes]: every shard's dump rows, in global channel order
    uint32_t dump_cap = 0;
    std::vector<uint32_t> counts;
    std::vector<uint32_t> dump_channels;  // global indices of the rows of h_dump
    uint64_t bytes = 0;
    bool gated = false;  // every shard ran the squelch for this tick
    bool queued = false;
  };
  std::vector<Slot> slot;
  uint32_t head = 0, tail = 0;
  int retired = -1;  // the slot of the last retired tick
  std::string err;
};

static thread_local std::string g_bank_error;
static int bank_fail(sdr_bank *b, int code, const std::string &what) {
  if (b) b->err = what;
  else g_bank_error = what;
  return code;
}
// error of shard i's engine, with the shard named
static int bank_fail_shard(sdr_bank *b, int code, uint32_t i) {
  char head[64];
  snprintf(head, sizeof head, "device %d (shard %u): ", b->device[i], i);
  return bank_fail(b, code, std::string(head) + sdr_last_error(b->eng[i]));
}

const char *sdr_bank_last_error(const sdr_bank *b) { return b ? b->err.c_str() : g_bank_error.c_str(); }

int sdr_bank_destroy(sdr_bank *b) {
  if (!b) return SDR_E_ARG;
  for (size_t i = 0; i < b->eng.size(); ++i) {
    if (i < b->ing.size() && b->ing[i]) sdr_ingest_destroy(b->ing[i]);
    if (b->eng[i]) sdr_engine_destroy(b->eng[i]);
  }
  for (auto &s : b->slot) {
    cudaFreeHost(s.h_iq);
    cudaFreeHost(s.h_pcm);
    cudaFreeHost(s.h_allowed);
    cudaFreeHost(s.h_magnitude);
    cudaFreeHost(s.h_dump);
  }
  delete b;
  return SDR_OK;
}

int sdr_bank_create(uint32_t n_channels, const int *devices, uint32_t n_devices, uint64_t block_bytes,
                    uint32_t n_slots, sdr_bank **out) {
  if (!out) return SDR_E_ARG;
  *out = nullptr;
  if (!devices || n_devices == 0 || n_channels < n_devices || n_slots < 2 || n_slots > 64 || block_bytes == 0 ||
      block_bytes % 64)
    return bank_fail(nullptr, SDR_E_ARG, "sdr_bank_create: need 1..n_channels devices, 2..64 slots, block_bytes a multiple of 64");
  for (uint32_t i = 0; i < n_devices; ++i)
    for (uint32_t j = 0; j < i; ++j)
      if (devices[i] == devices[j]) return bank_fail(nullptr, SDR_E_ARG, "sdr_bank_create: a device is listed twice");
  sdr_bank *b = new (std::nothrow) sdr_bank();
  if (!b) return SDR_E_NOMEM;
  b->n = n_channels;
  b->block_bytes = block_bytes;
  b->device.assign(devices, devices + n_devices);
  b->first.resize(n_devices + 1);
  for (uint32_t i = 0; i <= n_devices; ++i) b->first[i] = (uint32_t)((uint64_t)n_channels * i / n_devices);
  b->eng.assign(n_devices, nullptr);
  b->ing.assign(n_devices, nullptr);
  b->slot.resize(n_slots);
  // the shared tick, PCM, gate and magnitude arrays: pinned for every device's context
  for (auto &s : b->slot) {
    cudaError_t ce = cudaHostAlloc(&s.h_iq, (size_t)n_channels * block_bytes, cudaHostAllocPortable);
    if (ce == cudaSuccess) ce = cudaHostAlloc(&s.h_pcm, (size_t)n_channels * (block_bytes / 64) * 2, cudaHostAllocPortable);
    if (ce == cudaSuccess) ce = cudaHostAlloc(&s.h_allowed, n_channels, cudaHostAllocPortable);
    if (ce == cudaSuccess) ce = cudaHostAlloc(&s.h_magnitude, (size_t)n_channels * 4, cudaHostAllocPortable);
    if (ce != cudaSuccess) {
      bank_fail(nullptr, SDR_E_NOMEM, std::string("sdr_bank_create: pinned host memory: ") + cudaGetErrorString(ce));
      sdr_bank_destroy(b);
      return ce == cudaErrorMemoryAllocation ? SDR_E_NOMEM : SDR_E_CUDA;
    }
    s.counts.assign(n_channels, 0);
  }
  for (uint32_t i = 0; i < n_devices; ++i) {
    const uint32_t n_i = b->first[i + 1] - b->first[i];
    int rc = sdr_engine_create(n_i, devices[i], block_bytes, &b->eng[i]);
    if (rc) {
      bank_fail(nullptr, rc, std::string("sdr_bank_create: ") + sdr_last_error(nullptr));
      sdr_bank_destroy(b);
      return rc;
    }
    std::vector<uint8_t *> slabs(n_slots);
    for (uint32_t k = 0; k < n_slots; ++k) slabs[k] = b->slot[k].h_iq + (size_t)b->first[i] * block_bytes;
    rc = ingest_create(b->eng[i], n_slots, block_bytes, slabs.data(), &b->ing[i]);
    if (rc) {
      bank_fail(nullptr, rc, std::string("sdr_bank_create: ") + sdr_last_error(b->eng[i]));
      sdr_bank_destroy(b);
      return rc;
    }
  }
  *out = b;
  return SDR_OK;
}

uint32_t sdr_bank_device_count(const sdr_bank *b) { return b ? (uint32_t)b->device.size() : 0; }

int sdr_bank_shard(const sdr_bank *b, uint32_t i, int *device, uint32_t *first_channel, uint32_t *n_channels,
                   sdr_engine **engine) {
  if (!b || i >= b->device.size()) return SDR_E_ARG;
  if (device) *device = b->device[i];
  if (first_channel) *first_channel = b->first[i];
  if (n_channels) *n_channels = b->first[i + 1] - b->first[i];
  if (engine) *engine = b->eng[i];
  return SDR_OK;
}

// shard of a channel: first[] is ascending
static uint32_t bank_shard_of(const sdr_bank *b, uint32_t ch) {
  return (uint32_t)(std::upper_bound(b->first.begin(), b->first.end(), ch) - b->first.begin()) - 1;
}

int sdr_bank_set_mode(sdr_bank *b, uint32_t channel, int mode) {
  if (!b || channel >= b->n) return SDR_E_ARG;
  const uint32_t i = bank_shard_of(b, channel);
  const int rc = sdr_set_mode(b->eng[i], channel - b->first[i], mode);
  return rc ? bank_fail(b, rc, "sdr_bank_set_mode: bad mode") : SDR_OK;
}

int sdr_bank_set_modes(sdr_bank *b, const uint8_t *modes) {
  if (!b || !modes) return SDR_E_ARG;
  for (size_t i = 0; i < b->eng.size(); ++i) {
    const int rc = sdr_set_modes(b->eng[i], modes + b->first[i]);
    if (rc) return bank_fail(b, rc, "sdr_bank_set_modes: bad mode");
  }
  return SDR_OK;
}

int sdr_bank_set_gain(sdr_bank *b, uint32_t channel, int kind, float gain) {
  if (!b || channel >= b->n) return SDR_E_ARG;
  const uint32_t i = bank_shard_of(b, channel);
  const int rc = sdr_set_gain(b->eng[i], channel - b->first[i], kind, gain);
  return rc ? bank_fail(b, rc, "sdr_bank_set_gain: bad kind") : SDR_OK;
}

int sdr_bank_reset(sdr_bank *b, uint32_t channel, int kind) {
  if (!b || channel >= b->n) return SDR_E_ARG;
  const uint32_t i = bank_shard_of(b, channel);
  const int rc = sdr_reset(b->eng[i], channel - b->first[i], kind);
  return rc ? bank_fail_shard(b, rc, i) : SDR_OK;
}

int sdr_bank_set_squelch_threshold(sdr_bank *b, uint32_t channel, int32_t threshold_dbfs) {
  if (!b || channel >= b->n) return SDR_E_ARG;
  const uint32_t i = bank_shard_of(b, channel);
  return sdr_set_squelch_threshold(b->eng[i], channel - b->first[i], threshold_dbfs);
}

int sdr_bank_set_receive_gain_db(sdr_bank *b, uint32_t channel, uint32_t gain_db) {
  if (!b || channel >= b->n) return SDR_E_ARG;
  const uint32_t i = bank_shard_of(b, channel);
  return sdr_set_receive_gain_db(b->eng[i], channel - b->first[i], gain_db);
}

int sdr_bank_enable_signal_reports(sdr_bank *b, int on) {
  if (!b) return SDR_E_ARG;
  for (size_t i = 0; i < b->eng.size(); ++i) sdr_enable_signal_reports(b->eng[i], on);
  return SDR_OK;
}

int sdr_bank_set_squelch_block_bytes(sdr_bank *b, uint64_t block_bytes) {
  if (!b) return SDR_E_ARG;
  for (size_t i = 0; i < b->eng.size(); ++i) {
    const int rc = sdr_set_squelch_block_bytes(b->eng[i], block_bytes);
    if (rc) return bank_fail_shard(b, rc, (uint32_t)i);
  }
  return SDR_OK;
}

int sdr_bank_set_iq_dump(sdr_bank *b, uint32_t channel, int on) {
  if (!b || channel >= b->n) return SDR_E_ARG;
  const uint32_t i = bank_shard_of(b, channel);
  return sdr_set_iq_dump(b->eng[i], channel - b->first[i], on);
}

int sdr_bank_acquire(sdr_bank *b, void **iq, uint64_t *channel_stride) {
  if (!b || !iq) return SDR_E_ARG;
  sdr_bank::Slot &s = b->slot[b->head];
  if (s.queued) return bank_fail(b, SDR_E_FULL, "bank ring full: retire a tick first");
  *iq = s.h_iq;
  if (channel_stride) *channel_stride = b->block_bytes;
  return SDR_OK;
}

int sdr_bank_commit(sdr_bank *b, uint32_t timestamp, uint64_t bytes, uint32_t flags) {
  if (!b) return SDR_E_ARG;
  sdr_bank::Slot &s = b->slot[b->head];
  if (s.queued) return bank_fail(b, SDR_E_FULL, "bank ring full: retire a tick first");
  if (bytes == 0 || bytes % 64) return bank_fail(b, SDR_E_ARG, "bytes_per_channel must be a positive multiple of 64");
  const uint64_t take = bytes > b->block_bytes ? b->block_bytes : bytes;  // clipped like DataConsumer.cc:232-246
  // the rows every shard will dump (its channels with the dump on); the slot is free, so nothing
  // still copies into its dump array
  uint64_t dump_total = 0;
  for (size_t i = 0; i < b->eng.size(); ++i) dump_total += b->eng[i]->dump_count;
  if (dump_total > s.dump_cap) {
    cudaFreeHost(s.h_dump);
    s.h_dump = nullptr;
    s.dump_cap = 0;
    const cudaError_t ce = cudaHostAlloc(&s.h_dump, dump_total * b->block_bytes, cudaHostAllocPortable);
    if (ce != cudaSuccess)
      return bank_fail(b, ce == cudaErrorMemoryAllocation ? SDR_E_NOMEM : SDR_E_CUDA,
                       std::string("sdr_bank_commit: pinned host memory: ") + cudaGetErrorString(ce));
    s.dump_cap = (uint32_t)dump_total;
  }
  // the squelch blocks of this tick, the same on every shard; the gate and magnitude rows grow like
  // the dump array
  const uint32_t n_blocks = squelch_blocks(b->eng[0], take);
  for (size_t i = 1; i < b->eng.size(); ++i)
    if (squelch_blocks(b->eng[i], take) != n_blocks)
      return bank_fail(b, SDR_E_ARG, "sdr_bank_commit: the shards' squelch blocks differ: set them with sdr_bank_set_squelch_block_bytes");
  if (n_blocks > s.sig_cap) {
    cudaFreeHost(s.h_allowed);
    cudaFreeHost(s.h_magnitude);
    s.h_allowed = nullptr;
    s.h_magnitude = nullptr;
    s.sig_cap = 0;
    cudaError_t ce = cudaHostAlloc(&s.h_allowed, (size_t)n_blocks * b->n, cudaHostAllocPortable);
    if (ce == cudaSuccess) ce = cudaHostAlloc(&s.h_magnitude, (size_t)n_blocks * b->n * 4, cudaHostAllocPortable);
    if (ce != cudaSuccess)
      return bank_fail(b, ce == cudaErrorMemoryAllocation ? SDR_E_NOMEM : SDR_E_CUDA,
                       std::string("sdr_bank_commit: pinned host memory: ") + cudaGetErrorString(ce));
    s.sig_cap = n_blocks;
  }
  s.n_blocks = n_blocks;
  s.gated = true;
  s.dump_channels.clear();
  for (size_t i = 0; i < b->eng.size(); ++i) {
    // this device's slabs of the shared arrays: PCM rows take / 64 samples apart, its gate and
    // magnitudes, and its dump rows after those of the devices before it
    int16_t *dst = s.h_pcm + (size_t)b->first[i] * (take / 64);
    int8_t *dump_dst = s.h_dump ? s.h_dump + s.dump_channels.size() * b->block_bytes : nullptr;
    const int rc = ingest_commit(b->ing[i], timestamp, bytes, flags, dst, s.h_allowed + b->first[i],
                                 s.h_magnitude + b->first[i], b->n, dump_dst);
    if (rc) return bank_fail_shard(b, rc, (uint32_t)i);
    const sdr_ingest::Slot &t = b->ing[i]->slot[b->ing[i]->prev];  // the slot just committed
    s.gated = s.gated && t.gated;
    for (uint32_t ch : t.dump_channels) s.dump_channels.push_back(ch + b->first[i]);
  }
  s.bytes = take;
  s.queued = true;
  b->head = (b->head + 1) % (uint32_t)b->slot.size();
  return SDR_OK;
}

int sdr_bank_retire(sdr_bank *b, uint32_t *timestamp, const int16_t **pcm, uint32_t *samples_per_row,
                    const uint32_t **counts) {
  if (!b) return SDR_E_ARG;
  sdr_bank::Slot &s = b->slot[b->tail];
  if (!s.queued) return bank_fail(b, SDR_E_EMPTY, "bank ring empty: nothing to retire");
  uint32_t ts = 0, samples = 0;
  for (size_t i = 0; i < b->eng.size(); ++i) {
    const uint32_t *c = nullptr;
    const int rc = sdr_ingest_retire(b->ing[i], &ts, nullptr, &samples, &c);
    if (rc) return bank_fail_shard(b, rc, (uint32_t)i);
    memcpy(s.counts.data() + b->first[i], c, (size_t)(b->first[i + 1] - b->first[i]) * 4);
  }
  if (timestamp) *timestamp = ts;
  if (pcm) *pcm = s.h_pcm;
  if (samples_per_row) *samples_per_row = samples;
  if (counts) *counts = s.counts.data();
  s.queued = false;
  b->retired = (int)b->tail;
  b->tail = (b->tail + 1) % (uint32_t)b->slot.size();
  return SDR_OK;
}

// the slot of the last retired tick, or null if there is none (or its slot was committed again)
static const sdr_bank::Slot *bank_retired(const sdr_bank *b) {
  if (b->retired < 0 || b->slot[b->retired].queued) return nullptr;
  return &b->slot[b->retired];
}

int sdr_bank_retired_signal(sdr_bank *b, const uint8_t **allowed, const uint32_t **magnitude) {
  if (!b) return SDR_E_ARG;
  const sdr_bank::Slot *s = bank_retired(b);
  if (!s) return bank_fail(b, SDR_E_EMPTY, "no retired tick: retire one first");
  if (!s->gated)
    return bank_fail(b, SDR_E_ARG, "the retired tick ran no squelch on every device: set a threshold or enable signal reports before its commit");
  const size_t last = (size_t)(s->n_blocks - 1) * b->n;  // the last block's row
  if (allowed) *allowed = s->h_allowed + last;
  if (magnitude) *magnitude = s->h_magnitude + last;
  return SDR_OK;
}

int sdr_bank_retired_signal_blocks(sdr_bank *b, const uint8_t **allowed, const uint32_t **magnitude,
                                   uint32_t *n_blocks) {
  if (!b) return SDR_E_ARG;
  const sdr_bank::Slot *s = bank_retired(b);
  if (!s) return bank_fail(b, SDR_E_EMPTY, "no retired tick: retire one first");
  if (!s->gated)
    return bank_fail(b, SDR_E_ARG, "the retired tick ran no squelch on every device: set a threshold or enable signal reports before its commit");
  if (allowed) *allowed = s->h_allowed;
  if (magnitude) *magnitude = s->h_magnitude;
  if (n_blocks) *n_blocks = s->n_blocks;
  return SDR_OK;
}

int sdr_bank_retired_iq_dump(sdr_bank *b, const int8_t **rows, uint64_t *row_stride, uint64_t *n_bytes,
                             const uint32_t **channels, uint32_t *n_rows) {
  if (!b) return SDR_E_ARG;
  const sdr_bank::Slot *s = bank_retired(b);
  if (!s) return bank_fail(b, SDR_E_EMPTY, "no retired tick: retire one first");
  const bool any = !s->dump_channels.empty();
  if (rows) *rows = any ? s->h_dump : nullptr;
  if (row_stride) *row_stride = b->block_bytes;
  if (n_bytes) *n_bytes = s->bytes;
  if (channels) *channels = any ? s->dump_channels.data() : nullptr;
  if (n_rows) *n_rows = (uint32_t)s->dump_channels.size();
  return SDR_OK;
}

}  // extern "C"
