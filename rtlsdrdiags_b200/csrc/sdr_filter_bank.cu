// Host side of the batched filter banks and their C ABI (include/sdr_b200.h, sdr_filter_bank_*).
// One bank = n_rows independent filter objects of one reference class with the same taps.
// No CPU path exists.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/sdr_b200.h"
#include "sdr_filter_bank.cuh"
#include "sdr_iir_bank.cuh"

using namespace sdr;

struct sdr_filter_bank {
  int device = 0, kind = 0;
  uint32_t rows = 0, N = 0, F = 1, q = 0, C = 0;
  uint32_t pending = 0;  // decimator: samples waiting in decimationBuffer (same for every row)
  int cur = 0;           // which carry buffer is current
  bool i16 = false, interp = false;
  size_t esize = 4;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  void *d_taps = nullptr, *d_carry[2] = {};
  std::vector<int16_t> q15;
  uint32_t sum_abs_q15 = 0;
  // staging for host callers
  void *d_in = nullptr, *d_out = nullptr;
  uint64_t cap_in = 0, cap_out = 0;
  uint64_t launches = 0;
  std::string err;
  // SDR_FILTER_IIR_F32: taps, the warm-up the taps need (~0u: the response does not decay, so no
  // segmentation), the diagnostic overrides (seg 0 / warm ~0u = automatic) and the redo counter
  std::vector<float> iir_b, iir_a;
  uint32_t iir_warm = 0, dbg_seg = 0, dbg_warm = ~0u;
  uint64_t resident_lanes = 0;
  uint32_t *d_redo = nullptr;
};

namespace {

thread_local std::string g_fb_create_error;

int fb_fail(sdr_filter_bank *b, int code, const char *what, cudaError_t ce = cudaSuccess) {
  char buf[512];
  if (ce != cudaSuccess) snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(ce));
  else snprintf(buf, sizeof buf, "%s", what);
  if (b) b->err = buf;
  else g_fb_create_error = buf;
  return code;
}

#define FB_CK(b, call)                                                   \
  do {                                                                   \
    cudaError_t _ce = (call);                                            \
    if (_ce != cudaSuccess) return fb_fail((b), SDR_E_CUDA, #call, _ce); \
  } while (0)

// Decimator_int16.cc:58-62 / Interpolator_int16.cc:274-279: float product, C round(), then the
// (int16_t) cast as x86 performs it (cvttss2si, low 16 bits: 32768.0 becomes -32768)
int16_t quantise_q15(float h) {
  float s = h * 32768;
  s = (float)round((double)s);
  if (!(fabsf(s) < 2147483648.0f)) return 0;
  return (int16_t)(uint16_t)(uint32_t)(int32_t)s;
}

constexpr uint32_t FB_SMEM_WORDS = 11 * 1024;  // 44 KB: under the 48 KB a kernel gets without opt-in

}  // namespace

// The launch plan of a bank: the tile (outputs per CTA), the staged span and the shared memory it
// takes. One function for sdr_filter_bank_create, which refuses taps / factor combinations that no
// tile can serve, and for sdr_filter_bank_run.
static size_t fb_plan(const sdr_filter_bank *b, FilterBankParams &p, uint32_t &tile) {
  // tile: as many outputs (<= 2048) as the staged span fits next to the taps
  const uint32_t M = b->interp ? 1 : b->F;
  const uint32_t budget = FB_SMEM_WORDS - b->N - 64;
  if (b->interp) {
    uint32_t ti = 2048 / b->F;
    if (ti < 1) ti = 1;
    while (ti > 1 && ti + b->q - 1 > budget) ti /= 2;
    tile = ti * b->F;
    p.span = ti + b->q - 1;
    p.pitch = p.span;
  } else {
    tile = 2048;
    while (tile > 32 && (uint64_t)M * (tile - 1) + b->N + 3 * 32 * M > budget) tile /= 2;
    p.span = M * (tile - 1) + b->N;
    // phases land in different banks when the staging loop writes 32 consecutive samples; the eight
    // extra words are what the 16-byte window loads of the float M = 2, 4 path may read past the data
    p.pitch = ((p.span + M - 1) / M + 8 + 31) / 32 * 32 + ((32 % M) == 0 && M > 1 ? 32 / M : (M > 1 ? 1 : 0));
  }
  // decimators with M = 2, 4: taps above the highest full block of four a-values (see the kernel)
  p.kp = 0;
  p.hoff = 0;
  if (!b->interp && (M == 2 || M == 4)) {
    const uint32_t a_top = (b->N - 1) / M, ph_top = (b->N - 1) % M;
    const int a_full = (ph_top == M - 1) ? (int)a_top : (int)a_top - 1;  // largest a with every phase present
    const int n_blocks = a_full >= 3 ? (a_full + 1) / 4 : 0;
    p.kp = b->N - (uint32_t)n_blocks * 4 * M;
    p.hoff = (4 - p.kp % 4) % 4;
  }
  p.np = (p.hoff + b->N + 3) / 4 * 4;
  p.tile_out = tile;
  const size_t smem = (size_t)4 * p.np + (size_t)(b->interp ? p.span : (size_t)M * p.pitch) * b->esize + 16;
  return smem;
}

// Warm-up of the IIR bank's segments: the zero-input recurrence in double, from each unit initial
// state, with IirFilter's tap order; W = the first step after which every response stays below
// 2^-64 (for a = {-0.95}: 865). Two states that differ by at most their own size then agree far
// below float resolution. A response that has not decayed within IIR_WARM_CAP steps (marginal or
// unstable filters, or very slow poles) returns ~0u: such banks run one segment per row.
static constexpr int IIR_WARM_CAP = 8192;
static uint32_t iir_warm_up(const float *a, uint32_t na) {
  const double tiny = ldexp(1.0, -64);
  int last = 0;  // last step (1-based) whose response was not below 2^-64
  for (uint32_t i = 0; i < na; ++i) {
    double h[IIR_MAX_NA] = {};  // h[0] = y[n-1]
    h[i] = 1.0;
    for (int n = 1; n <= 2 * IIR_WARM_CAP; ++n) {
      double r = 0.0 + (double)a[0] * h[na - 1];
      for (uint32_t k = 1; k < na; ++k) r = r + (double)a[k] * h[k - 1];
      const double y = 0.0 - r;
      for (uint32_t k = na - 1; k > 0; --k) h[k] = h[k - 1];
      h[0] = y;
      if (!(fabs(y) < tiny)) last = n;
    }
  }
  return last + 1 > IIR_WARM_CAP ? ~0u : (uint32_t)(last + 1);
}

typedef void (*IirKernel)(IirBankParams);
template <int NB>
static IirKernel iir_kernel_nb(uint32_t na) {
  switch (na) {
    case 1: return iir_bank_kernel<1, NB>;
    case 2: return iir_bank_kernel<2, NB>;
    case 3: return iir_bank_kernel<3, NB>;
    case 4: return iir_bank_kernel<4, NB>;
    case 5: return iir_bank_kernel<5, NB>;
    case 6: return iir_bank_kernel<6, NB>;
    case 7: return iir_bank_kernel<7, NB>;
    default: return iir_bank_kernel<8, NB>;
  }
}
static IirKernel iir_kernel(uint32_t nb, uint32_t na) {
  return nb == 1 ? iir_kernel_nb<1>(na) : nb == 2 ? iir_kernel_nb<2>(na) : iir_kernel_nb<0>(na);
}

// One IIR call: S segments per row (a power of two <= 32) so that rows x S lanes fill the GPU
// without a second wave, each at least four warm-ups long; no empty segments in the middle.
static int iir_run(sdr_filter_bank *b, const float *d_in, uint64_t istr, float *d_out, uint64_t ostr, uint32_t n) {
  const uint32_t blocks = (n + IIR_BLK - 1) / IIR_BLK;
  const uint32_t warm = b->dbg_warm != ~0u ? b->dbg_warm : b->iir_warm;
  const uint32_t warm_r = warm == ~0u ? ~0u : (warm + IIR_BLK - 1) / IIR_BLK * IIR_BLK;
  uint32_t S = 1;
  if (b->dbg_seg) {
    S = b->dbg_seg;
  } else if (warm_r != ~0u) {
    const uint32_t min_blocks = 4 * (warm_r / IIR_BLK > 0 ? warm_r / IIR_BLK : 1);
    while (S < 32 && (uint64_t)b->rows * 2 * S <= b->resident_lanes && blocks / (2 * S) >= min_blocks) S *= 2;
  }
  while (S > 1 && (blocks + S - 1) / S * (S - 1) >= blocks) S /= 2;
  IirBankParams p;
  p.in = d_in;
  p.out = d_out;
  p.carry_in = (const float *)b->d_carry[b->cur];
  p.carry_out = (float *)b->d_carry[b->cur ^ 1];
  p.redo = b->d_redo;
  p.in_stride = istr;
  p.out_stride = ostr;
  p.n = n;
  p.rows = b->rows;
  p.nb = (uint32_t)b->iir_b.size();
  p.na = (uint32_t)b->iir_a.size();
  p.C = b->C;
  p.seg_log2 = 0;
  while ((1u << p.seg_log2) < S) ++p.seg_log2;
  p.seg_len = (blocks + S - 1) / S * IIR_BLK;
  p.warm = S == 1 ? 0u : (warm_r == ~0u ? p.seg_len * S : warm_r);  // ~0u with a forced S: start at the head
  memset(p.b, 0, sizeof p.b);
  memset(p.a, 0, sizeof p.a);
  memcpy(p.b, b->iir_b.data(), 4 * (size_t)p.nb);
  memcpy(p.a, b->iir_a.data(), 4 * (size_t)p.na);
  const uint64_t lanes = (uint64_t)b->rows << p.seg_log2;
  iir_kernel(p.nb, p.na)<<<(unsigned)((lanes + 31) / 32), IIR_THREADS, 0, b->stream>>>(p);
  return SDR_OK;
}

extern "C" {

int sdr_filter_bank_create(int device, int kind, uint32_t n_rows, const float *taps, uint32_t n_taps,
                           uint32_t factor, sdr_filter_bank **out) {
  if (!out) return fb_fail(nullptr, SDR_E_ARG, "out is NULL");
  *out = nullptr;
  if (kind < SDR_FILTER_DECIMATOR_F32 || kind > SDR_FILTER_INTERPOLATOR_I16)
    return fb_fail(nullptr, SDR_E_ARG, "kind must be one of SDR_FILTER_*");
  if (!taps || n_taps == 0 || factor == 0 || n_rows == 0 || n_rows > 65535)
    return fb_fail(nullptr, SDR_E_ARG, "taps, n_taps, factor and n_rows (1..65535) must be set");
  const bool interp = kind == SDR_FILTER_INTERPOLATOR_F32 || kind == SDR_FILTER_INTERPOLATOR_I16;
  // Interpolator.h: "q = N/L must be an integer"
  if (interp && (n_taps % factor != 0)) return fb_fail(nullptr, SDR_E_ARG, "interpolator: n_taps must be a multiple of the factor");
  if (n_taps + 32 * factor + 64 > FB_SMEM_WORDS) return fb_fail(nullptr, SDR_E_ARG, "n_taps + 32 * factor exceeds the tile a CTA can stage");
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count)
    return fb_fail(nullptr, SDR_E_CUDA, "no usable CUDA device (there is no CPU fallback)");
  FB_CK(nullptr, cudaSetDevice(device));
  sdr_filter_bank *b = new sdr_filter_bank;
  b->device = device;
  b->kind = kind;
  b->rows = n_rows;
  b->N = n_taps;
  b->F = factor;
  b->interp = interp;
  b->i16 = kind == SDR_FILTER_DECIMATOR_I16 || kind == SDR_FILTER_INTERPOLATOR_I16;
  b->esize = b->i16 ? 2 : 4;
  b->q = interp ? n_taps / factor : n_taps;
  b->C = interp ? b->q - 1 : (n_taps - 1) + (factor - 1);
  {  // the plan sdr_filter_bank_run will use must fit the shared memory a kernel gets without opt-in
    FilterBankParams plan;
    uint32_t tile = 0;
    if (fb_plan(b, plan, tile) > 48 * 1024) {
      delete b;
      return fb_fail(nullptr, SDR_E_ARG, "n_taps and factor need a tile that does not fit in 48 KB of shared memory");
    }
  }
  cudaError_t ce = cudaStreamCreateWithFlags(&b->own_stream, cudaStreamNonBlocking);
  if (ce != cudaSuccess) { delete b; return fb_fail(nullptr, SDR_E_CUDA, "cudaStreamCreate", ce); }
  b->stream = b->own_stream;
  std::vector<int32_t> q32(n_taps);
  b->q15.resize(n_taps);
  for (uint32_t i = 0; i < n_taps; ++i) {
    b->q15[i] = quantise_q15(taps[i]);
    q32[i] = b->q15[i];
    b->sum_abs_q15 += (uint32_t)abs((int)b->q15[i]);
  }
  if (interp) {  // an output only meets the taps of its own phase: the largest phase sum bounds it
    b->sum_abs_q15 = 0;
    for (uint32_t ph = 0; ph < factor; ++ph) {
      uint32_t s = 0;
      for (uint32_t k = ph; k < n_taps; k += factor) s += (uint32_t)abs((int)b->q15[k]);
      b->sum_abs_q15 = s > b->sum_abs_q15 ? s : b->sum_abs_q15;
    }
  }
  const void *src = b->i16 ? (const void *)q32.data() : (const void *)taps;
  const size_t cbytes = (size_t)(b->C ? b->C : 1) * n_rows * b->esize;
  if ((ce = cudaMalloc(&b->d_taps, 4 * (size_t)n_taps)) != cudaSuccess ||
      (ce = cudaMalloc(&b->d_carry[0], cbytes)) != cudaSuccess ||
      (ce = cudaMalloc(&b->d_carry[1], cbytes)) != cudaSuccess ||
      (ce = cudaMemcpy(b->d_taps, src, 4 * (size_t)n_taps, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (ce = cudaMemset(b->d_carry[0], 0, cbytes)) != cudaSuccess ||
      (ce = cudaMemset(b->d_carry[1], 0, cbytes)) != cudaSuccess) {
    sdr_filter_bank_destroy(b);
    return fb_fail(nullptr, ce == cudaErrorMemoryAllocation ? SDR_E_NOMEM : SDR_E_CUDA, "filter bank allocation", ce);
  }
  *out = b;
  return SDR_OK;
}

/* IirFilter(nb, b, na, a) (Filters/IirFilter.cc) for every row */
int sdr_filter_bank_create_iir(int device, uint32_t n_rows, const float *b_taps, uint32_t nb, const float *a_taps,
                               uint32_t na, sdr_filter_bank **out) {
  if (!out) return fb_fail(nullptr, SDR_E_ARG, "out is NULL");
  *out = nullptr;
  if (!b_taps || !a_taps || nb < 1 || nb > IIR_MAX_NB || na < 1 || na > IIR_MAX_NA || n_rows == 0 || n_rows > 65535)
    return fb_fail(nullptr, SDR_E_ARG, "IIR bank: taps must be set, 1 <= nb <= 64, 1 <= na <= 8, 1 <= n_rows <= 65535");
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count)
    return fb_fail(nullptr, SDR_E_CUDA, "no usable CUDA device (there is no CPU fallback)");
  FB_CK(nullptr, cudaSetDevice(device));
  sdr_filter_bank *b = new sdr_filter_bank;
  b->device = device;
  b->kind = SDR_FILTER_IIR_F32;
  b->rows = n_rows;
  b->N = nb;
  b->F = 1;
  b->esize = 4;
  b->C = (nb - 1) + na;  // per row: the last nb - 1 inputs, then the last na outputs
  b->iir_b.assign(b_taps, b_taps + nb);
  b->iir_a.assign(a_taps, a_taps + na);
  b->iir_warm = iir_warm_up(a_taps, na);
  if (b->iir_warm != ~0u && b->iir_warm < na) b->iir_warm = na;  // the compared state must be made of computed outputs
  int per_sm = 0, sms = 0;
  cudaError_t ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, iir_kernel(nb, na), IIR_THREADS, 0);
  if (ce == cudaSuccess) ce = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  if (ce != cudaSuccess) { delete b; return fb_fail(nullptr, SDR_E_CUDA, "IIR bank: occupancy query", ce); }
  b->resident_lanes = (uint64_t)(per_sm > 0 ? per_sm : 1) * (uint64_t)sms * 32;
  ce = cudaStreamCreateWithFlags(&b->own_stream, cudaStreamNonBlocking);
  if (ce != cudaSuccess) { delete b; return fb_fail(nullptr, SDR_E_CUDA, "cudaStreamCreate", ce); }
  b->stream = b->own_stream;
  const size_t cbytes = (size_t)b->C * n_rows * 4;
  if ((ce = cudaMalloc(&b->d_carry[0], cbytes)) != cudaSuccess || (ce = cudaMalloc(&b->d_carry[1], cbytes)) != cudaSuccess ||
      (ce = cudaMalloc(&b->d_redo, 4)) != cudaSuccess || (ce = cudaMemset(b->d_carry[0], 0, cbytes)) != cudaSuccess ||
      (ce = cudaMemset(b->d_carry[1], 0, cbytes)) != cudaSuccess || (ce = cudaMemset(b->d_redo, 0, 4)) != cudaSuccess) {
    sdr_filter_bank_destroy(b);
    return fb_fail(nullptr, ce == cudaErrorMemoryAllocation ? SDR_E_NOMEM : SDR_E_CUDA, "filter bank allocation", ce);
  }
  *out = b;
  return SDR_OK;
}

int sdr_filter_bank_destroy(sdr_filter_bank *b) {
  if (!b) return SDR_E_ARG;
  cudaSetDevice(b->device);
  if (b->own_stream) cudaStreamSynchronize(b->own_stream);
  cudaFree(b->d_taps);
  cudaFree(b->d_carry[0]);
  cudaFree(b->d_carry[1]);
  cudaFree(b->d_in);
  cudaFree(b->d_out);
  cudaFree(b->d_redo);
  if (b->own_stream) cudaStreamDestroy(b->own_stream);
  delete b;
  return SDR_OK;
}

int sdr_filter_bank_set_stream(sdr_filter_bank *b, void *cuda_stream) {
  if (!b) return SDR_E_ARG;
  b->stream = cuda_stream ? (cudaStream_t)cuda_stream : b->own_stream;
  return SDR_OK;
}

/* resetFilterState() of every row (Decimator.cc:114-140, Interpolator.cc resetFilterState) */
int sdr_filter_bank_reset(sdr_filter_bank *b) {
  if (!b) return SDR_E_ARG;
  FB_CK(b, cudaSetDevice(b->device));
  const size_t cbytes = (size_t)(b->C ? b->C : 1) * b->rows * b->esize;
  FB_CK(b, cudaMemsetAsync(b->d_carry[b->cur], 0, cbytes, b->stream));
  // both decimator classes also drop the samples waiting in decimationBuffer
  // (Decimator.cc:137, Decimator_int16.cc:145)
  b->pending = 0;
  return SDR_OK;
}

uint64_t sdr_filter_bank_out_count(const sdr_filter_bank *b, uint64_t n_in) {
  if (!b) return 0;
  return b->interp ? n_in * b->F : (b->pending + n_in) / b->F;
}

int sdr_filter_bank_taps_q15(const sdr_filter_bank *b, int16_t *q) {
  if (!b || !q || b->kind == SDR_FILTER_IIR_F32) return SDR_E_ARG;  // there is no Q15 IirFilter
  memcpy(q, b->q15.data(), 2 * (size_t)b->N);
  return (int)b->N;
}

int sdr_filter_bank_run(sdr_filter_bank *b, const void *in, uint64_t in_stride, uint64_t n_in, void *out,
                        uint64_t out_stride, uint64_t *n_out_ret, uint32_t flags) {
  if (!b) return SDR_E_ARG;
  const uint64_t n_out = sdr_filter_bank_out_count(b, n_in);
  if (n_out_ret) *n_out_ret = n_out;
  if (n_in == 0) return SDR_OK;
  if (!in || (n_out && !out) || in_stride < n_in || out_stride < n_out) return fb_fail(b, SDR_E_ARG, "bad buffer, stride or count");
  if (n_in > (1ull << 40)) return fb_fail(b, SDR_E_TOO_LONG, "n_in too large");
  if (b->kind == SDR_FILTER_IIR_F32 && n_in >= (1ull << 31)) return fb_fail(b, SDR_E_TOO_LONG, "IIR bank: n_in must be below 2^31");
  FB_CK(b, cudaSetDevice(b->device));
  const bool host = !(flags & SDR_IQ_DEVICE);
  const void *d_in = in;
  void *d_out = out;
  uint64_t istr = in_stride, ostr = out_stride;
  if (host) {
    // dense staging rows; the copies are ordered on the bank's stream
    if (b->cap_in < n_in) {
      FB_CK(b, cudaStreamSynchronize(b->stream));
      cudaFree(b->d_in);
      b->d_in = nullptr;
      b->cap_in = 0;
      FB_CK(b, cudaMalloc(&b->d_in, n_in * b->rows * b->esize));
      b->cap_in = n_in;
    }
    if (b->cap_out < n_out) {
      FB_CK(b, cudaStreamSynchronize(b->stream));
      cudaFree(b->d_out);
      b->d_out = nullptr;
      b->cap_out = 0;
      FB_CK(b, cudaMalloc(&b->d_out, n_out * b->rows * b->esize));
      b->cap_out = n_out;
    }
    FB_CK(b, cudaMemcpy2DAsync(b->d_in, n_in * b->esize, in, in_stride * b->esize, n_in * b->esize, b->rows,
                               cudaMemcpyHostToDevice, b->stream));
    d_in = b->d_in;
    d_out = b->d_out;
    istr = n_in;
    ostr = n_out;
  }

  if (b->kind == SDR_FILTER_IIR_F32) {
    iir_run(b, (const float *)d_in, istr, (float *)d_out, ostr, (uint32_t)n_in);
  } else {
  FilterBankParams p;
  p.in = d_in;
  p.out = d_out;
  p.carry_in = b->d_carry[b->cur];
  p.carry_out = b->d_carry[b->cur ^ 1];
  p.taps = b->d_taps;
  p.in_stride = istr;
  p.out_stride = ostr;
  p.n_in = n_in;
  p.n_out = n_out;
  p.N = b->N;
  p.F = b->F;
  p.q = b->q;
  p.C = b->C;
  p.pending = b->pending;
  p.sum_abs_taps = b->sum_abs_q15;
  uint32_t tile;
  const size_t smem = fb_plan(b, p, tile);
  if (smem > 48 * 1024) return fb_fail(b, SDR_E_ARG, "tile does not fit in shared memory");
  const uint64_t tiles = n_out ? (n_out + tile - 1) / tile : 1;
  if (tiles > 0x7fffffffull) return fb_fail(b, SDR_E_TOO_LONG, "too many tiles");
  dim3 grid((unsigned)tiles, b->rows);
#define FB_LAUNCH(T, INTERP, MT) filter_bank_kernel<T, INTERP, MT><<<grid, FB_THREADS, smem, b->stream>>>(p)
#define FB_LAUNCH_DEC(T)                      \
  switch (b->F) {                             \
    case 1: FB_LAUNCH(T, false, 1); break;    \
    case 2: FB_LAUNCH(T, false, 2); break;    \
    case 4: FB_LAUNCH(T, false, 4); break;    \
    default: FB_LAUNCH(T, false, 0); break;   \
  }
#define FB_LAUNCH_INT(T)                      \
  switch (b->F) {                             \
    case 2: FB_LAUNCH(T, true, 2); break;     \
    case 3: FB_LAUNCH(T, true, 3); break;     \
    case 4: FB_LAUNCH(T, true, 4); break;     \
    case 8: FB_LAUNCH(T, true, 8); break;     \
    default: FB_LAUNCH(T, true, 0); break;    \
  }
  switch (b->kind) {
    case SDR_FILTER_DECIMATOR_F32: FB_LAUNCH_DEC(float); break;
    case SDR_FILTER_INTERPOLATOR_F32: FB_LAUNCH_INT(float); break;
    case SDR_FILTER_DECIMATOR_I16: FB_LAUNCH_DEC(int16_t); break;
    case SDR_FILTER_INTERPOLATOR_I16: FB_LAUNCH_INT(int16_t); break;
  }
#undef FB_LAUNCH_INT
#undef FB_LAUNCH_DEC
#undef FB_LAUNCH
  }
  FB_CK(b, cudaGetLastError());
  ++b->launches;
  b->cur ^= 1;
  if (!b->interp) b->pending = (uint32_t)((b->pending + n_in) % b->F);
  if (host) {
    if (n_out)
      FB_CK(b, cudaMemcpy2DAsync(out, out_stride * b->esize, b->d_out, n_out * b->esize, n_out * b->esize, b->rows,
                                 cudaMemcpyDeviceToHost, b->stream));
    FB_CK(b, cudaStreamSynchronize(b->stream));
  }
  return SDR_OK;
}

int sdr_filter_bank_sync(sdr_filter_bank *b) {
  if (!b) return SDR_E_ARG;
  FB_CK(b, cudaSetDevice(b->device));
  FB_CK(b, cudaStreamSynchronize(b->stream));
  return SDR_OK;
}

uint64_t sdr_filter_bank_launch_count(const sdr_filter_bank *b) { return b ? b->launches : 0; }

const char *sdr_filter_bank_last_error(const sdr_filter_bank *b) {
  return b ? b->err.c_str() : g_fb_create_error.c_str();
}

// Diagnostics (not part of include/sdr_b200.h): the IIR bank's segmentation -- seg_count 0 = chosen
// per call, else a power of two <= 32; warm = samples a segment s > 0 warms up on (rounded up to
// blocks of 32; ~0u = the bank's own) -- and how many segments were redone serially so far
// (synchronises). Tests shrink the warm-up to force the redo path.
int sdr_debug_filter_bank_set_iir_shape(sdr_filter_bank *b, uint32_t seg_count, uint32_t warm) {
  if (!b || b->kind != SDR_FILTER_IIR_F32 || seg_count > 32 || (seg_count & (seg_count - 1))) return SDR_E_ARG;
  b->dbg_seg = seg_count;
  b->dbg_warm = warm;
  return SDR_OK;
}

int sdr_debug_filter_bank_redo_count(sdr_filter_bank *b, uint32_t *count) {
  if (!b || !count || b->kind != SDR_FILTER_IIR_F32) return SDR_E_ARG;
  FB_CK(b, cudaSetDevice(b->device));
  FB_CK(b, cudaMemcpyAsync(count, b->d_redo, 4, cudaMemcpyDeviceToHost, b->stream));
  FB_CK(b, cudaStreamSynchronize(b->stream));
  return SDR_OK;
}

}  // extern "C"
