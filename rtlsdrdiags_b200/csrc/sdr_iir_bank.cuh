// Batched IirFilter (Filters/IirFilter.cc): n_rows independent Direct Form I filters with the same
// taps, as a segment-parallel recurrence (DESIGN section 4, "Segment-parallel recurrence").
//
// Arithmetic: the oracle's sdro_iir, one single-rounded operation at a time and in its order,
//   fir = 0;  fir = fir + b[k]*x[n-k]      k = 0 .. nb-1
//   r   = 0;  r = r + a[0]*y[n-na];  r = r + a[k]*y[n-k]   k = 1 .. na-1
//   y[n] = fir - r
// Signed zeros. `0 + p` turns a -0 product into +0, and fl(-0 - (+0)) = -0 while fl(-0 - (-0)) = +0.
// The numerator keeps its leading `0 +`: without it fir could be -0. With it, fir is never -0 (a
// round-to-nearest sum is -0 only if both terms are, and the sum starts at +0). The recurrence's
// leading `0 +` is dropped: r without it differs from r with it at most in the sign of a zero
// (adding +0 or -0 to a non-zero value gives that value), and fir - (+0) = fir - (-0) for every
// fir that is not -0. So y is the same bits, and the na = 1 chain is one multiply and one subtract
// per sample instead of three dependent operations. (NaN bit patterns are outside the contract.)
//
// Segmentation (dc_block_kernel's method, generalised to na states and any numerator). A call's
// rows are cut into S <= 32 segments of seg_len samples (a multiple of 32); every (row, segment)
// pair is a lane and a row's segments sit in one warp.
//   * segment 0 starts from the carried state;
//   * segment s > 0 starts `warm` samples early (or at the call's head, from the carried state,
//     if that is nearer) from y = 0. Its numerator reads the real input (and the carried inputs
//     before the call's head), so only the na y-values can differ from the serial run's;
//   * afterwards lane s compares the na y-values it entered its own samples with against lane
//     s - 1's final ones, bit for bit. Equal: by induction every output of segment s is the serial
//     one. Different (not merged yet, or never: a y stuck on a denormal): the first such segment of
//     each row is redone from the true state and the comparison is repeated.
// Correctness never depends on `warm`; the host picks it so that a redo is rare.
//
// One CTA = two warps over 32 lanes, in steps of one BLOCK of 32 samples per lane.
//   warp 0, the CHAIN: the recurrence and nothing else, its na states in registers. It turns the
//     numerators of block c into outputs in place (a 144-byte run per lane in shared memory).
//   warp 1, the FEEDER: stages every lane's input IIR_AHEAD blocks ahead through 4-byte cp.async
//     (the warp copies one lane's 32 samples per instruction, so any element offset and any row
//     stride coalesce into whole lines), computes block c + 1's numerators in tap order from that
//     ring, and writes block c - 1's outputs back, again one lane's 32 samples per instruction.
// One CTA barrier per block.
#pragma once
#include "sdr_platform.h"

namespace sdr {

constexpr int IIR_MAX_NB = 64, IIR_MAX_NA = 8;
constexpr int IIR_THREADS = 64;
constexpr int IIR_BLK = 32;                     // samples per lane and step
constexpr int IIR_RING = 8;                     // input blocks per lane in shared memory
constexpr int IIR_AHEAD = IIR_RING - 3;         // in flight beyond the block being filtered and its two predecessors (nb - 1 <= 63)
constexpr int IIR_XP = IIR_RING * IIR_BLK + 1;  // words per lane of the input ring: odd, so lane-per-thread reads are conflict-free
constexpr int IIR_FP = IIR_BLK + 4;             // words per lane of a numerator / output block (144 bytes: 128-bit accesses conflict-free)

struct IirBankParams {
  const float *in;         // [rows][in_stride]
  float *out;              // [rows][out_stride]
  const float *carry_in;   // [rows][C]: x[-(nb-1)] .. x[-1], then y[-1], y[-2], .. y[-na]
  float *carry_out;        // [rows][C], the same after this call
  uint32_t *redo;          // segments redone serially (diagnostics)
  uint64_t in_stride, out_stride;
  uint32_t n;              // samples per row, this call (< 2^31)
  uint32_t rows, nb, na, C;
  uint32_t seg_log2;       // S = 1 << seg_log2 segments per row
  uint32_t seg_len;        // samples per segment (multiple of IIR_BLK)
  uint32_t warm;           // warm-up samples of a segment s > 0 (multiple of IIR_BLK)
  float b[IIR_MAX_NB], a[IIR_MAX_NA];
};

__device__ __forceinline__ void iir_cp4(float *smem, const float *gmem) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void iir_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void iir_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// What the feeder needs of every lane in one pass (written by the feeder thread of that lane): one
// 16-byte record per lane and direction, so the per-lane loops below read it with one shared load.
struct __align__(16) IirRun {
  const float *p;  // input (or output) row + the lane's first sample of the pass
  uint32_t len;    // samples the lane runs this pass (0: it sits the pass out)
  uint32_t skip;   // store - begin: warm-up samples whose outputs are dropped
};
struct IirLanes {
  IirRun in[32], out[32];
  const float *hist[32];  // carry row + nb - 1: hist[g] = x[g] for -(nb-1) <= g < 0
  int32_t begin[32];      // first sample of the pass
};

// feeder: block c of every lane into the ring (c < 0: the history before the lane's first sample).
// Samples past a lane's run are never filtered, so they are not fetched.
__device__ __forceinline__ void iir_fill(const IirBankParams &p, const IirLanes &L, float *s_x, int c, int t) {
  float *slot = s_x + ((c + 2) & (IIR_RING - 1)) * IIR_BLK + t;
  const int o = c * IIR_BLK + t;
  if (c >= 0) {
#pragma unroll 8
    for (int j = 0; j < 32; ++j) {
      const IirRun r = L.in[j];
      if ((uint32_t)o < r.len) iir_cp4(slot + j * IIR_XP, r.p + o);
    }
  } else {
    for (int j = 0; j < 32; ++j) {
      if (L.in[j].len == 0) continue;
      const int g = L.begin[j] + o;
      if (g >= 0) iir_cp4(slot + j * IIR_XP, L.in[j].p + o);
      else if (g >= -(int)(p.nb - 1)) iir_cp4(slot + j * IIR_XP, L.hist[j] + g);
      // older samples meet no tap
    }
  }
}

// feeder: the numerators of block c of this thread's lane, in tap order, into its run of f
template <int NB>
__device__ __forceinline__ void iir_numerator(const IirBankParams &p, const float *xr, float *f, int c) {
  const int base = ((c + 2) & (IIR_RING - 1)) * IIR_BLK;
  constexpr int RM = IIR_RING * IIR_BLK - 1;
  if constexpr (NB == 1 || NB == 2) {
    // the reference's own shapes: a sliding window in registers, one shared load per sample
    const float b0 = p.b[0], b1 = NB == 2 ? p.b[1] : 0.f;
    float prev = NB == 2 ? xr[(base - 1) & RM] : 0.f;
#pragma unroll
    for (int q = 0; q < IIR_BLK / 4; ++q) {
      float v[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float x = xr[base + 4 * q + i];
        float acc = fadd(0.f, fmul(b0, x));
        if (NB == 2) acc = fadd(acc, fmul(b1, prev));
        prev = x;
        v[i] = acc;
      }
      sts_u4(f + 4 * q, u32x4{f2u(v[0]), f2u(v[1]), f2u(v[2]), f2u(v[3])});
    }
  } else {
    for (int q = 0; q < IIR_BLK / 4; ++q) {
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      for (uint32_t k = 0; k < p.nb; ++k) {
        const float bk = p.b[k];
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = fadd(v[i], fmul(bk, xr[(base + 4 * q + i - (int)k) & RM]));
      }
      sts_u4(f + 4 * q, u32x4{f2u(v[0]), f2u(v[1]), f2u(v[2]), f2u(v[3])});
    }
  }
}

// chain: one sample of the recurrence; h[0] = y[n-1] .. h[NA-1] = y[n-NA]. r starts at the product
// itself rather than at 0 + product: the same y, see the top of this file.
template <int NA>
__device__ __forceinline__ float iir_step(const float (&a)[NA], float (&h)[NA], float fir) {
  float r = fmul(a[0], h[NA - 1]);
#pragma unroll
  for (int k = 1; k < NA; ++k) r = fadd(r, fmul(a[k], h[k - 1]));
  const float y = fsub(fir, r);
#pragma unroll
  for (int k = NA - 1; k > 0; --k) h[k] = h[k - 1];
  h[0] = y;
  return y;
}

// NA = denominator taps; NB = 1 or 2 (numerator window in registers) or 0 (any nb, from the ring)
template <int NA, int NB>
__global__ void __launch_bounds__(IIR_THREADS) iir_bank_kernel(const __grid_constant__ IirBankParams p) {
  __shared__ float s_x[32 * IIR_XP];
  __shared__ __align__(16) float s_f[3 * 32 * IIR_FP];
  __shared__ __align__(16) IirLanes s_lanes;
  __shared__ uint32_t s_begin[32];  // per pass: first sample the lane runs, ~0u if it sits the pass out
  __shared__ uint32_t s_more;

  const int lane = threadIdx.x & 31;
  const bool chain = threadIdx.x < 32;
  const uint32_t S = 1u << p.seg_log2;
  const uint32_t idx = blockIdx.x * 32u + (uint32_t)lane;
  const uint32_t row = idx >> p.seg_log2, s = idx & (S - 1);
  const uint32_t store = s * p.seg_len;  // the lane's own samples are [store, end)
  const bool valid = row < p.rows && store < p.n;
  const uint32_t end = valid ? min(store + p.seg_len, p.n) : 0u;
  const uint64_t r64 = valid ? row : 0;
  const float *in_row = p.in + r64 * p.in_stride;
  const float *carry_row = p.carry_in + r64 * p.C;

  float a[NA], h[NA], y_in[NA], y_end[NA];
  uint32_t begin = store > p.warm ? store - p.warm : 0u;
  bool exact = begin == 0;  // starts from the carried state: nothing to verify
#pragma unroll
  for (int k = 0; k < NA; ++k) {
    a[k] = p.a[k];
    h[k] = valid && exact ? carry_row[p.nb - 1 + k] : 0.f;
    y_in[k] = y_end[k] = h[k];
  }
  bool todo = valid, redo = false;

  for (;;) {
    // ---- both warps learn which lanes run this pass and from which sample ----
    if (chain) s_begin[lane] = todo ? begin : ~0u;
    __syncthreads();
    const uint32_t my_begin = s_begin[lane];
    const bool on = my_begin != ~0u;
    const uint32_t len = on ? end - my_begin : 0u;
    const uint32_t trips = __reduce_max_sync(0xffffffffu, (len + IIR_BLK - 1) / IIR_BLK);

    if (!chain) {
      const uint32_t skip = on ? store - my_begin : 0u;
      s_lanes.in[lane] = IirRun{in_row + (on ? my_begin : 0u), len, skip};
      s_lanes.out[lane] = IirRun{p.out + r64 * p.out_stride + (on ? my_begin : 0u), len, skip};
      s_lanes.hist[lane] = carry_row + (p.nb - 1);
      s_lanes.begin[lane] = (int32_t)(on ? my_begin : 0u);
      __syncwarp();
      for (int c = -2; c < IIR_AHEAD; ++c) {
        iir_fill(p, s_lanes, s_x, c, lane);
        iir_commit();
      }
    }

    // iteration it: the feeder fills block it + AHEAD, filters block it and writes block it - 2
    // back; the chain runs block it - 1
    for (uint32_t it = 0; it <= trips + 1; ++it) {
      if (chain) {
        if (it >= 1 && it <= trips) {
          const uint32_t c = it - 1;
          const uint32_t g0 = my_begin + c * IIR_BLK;
          const bool act = on && g0 < end;
          float *fp = s_f + (c % 3) * 32 * IIR_FP + lane * IIR_FP;
          float f[IIR_BLK];
#pragma unroll
          for (int q = 0; q < IIR_BLK / 4; ++q) {
            const u32x4 v = lds_u4(fp + 4 * q);
            f[4 * q] = u2f(v.x); f[4 * q + 1] = u2f(v.y); f[4 * q + 2] = u2f(v.z); f[4 * q + 3] = u2f(v.w);
          }
          if (act && g0 == store) {
#pragma unroll
            for (int k = 0; k < NA; ++k) y_in[k] = h[k];
          }
          const uint32_t r = act ? min(end - g0, (uint32_t)IIR_BLK) : 0u;
          if (__any_sync(0xffffffffu, act && r < (uint32_t)IIR_BLK)) {
#pragma unroll
            for (int t = 0; t < IIR_BLK; ++t)
              if ((uint32_t)t < r) f[t] = iir_step<NA>(a, h, f[t]);
          } else if (act) {
#pragma unroll
            for (int t = 0; t < IIR_BLK; ++t) f[t] = iir_step<NA>(a, h, f[t]);
          }
          if (act) {
#pragma unroll
            for (int q = 0; q < IIR_BLK / 4; ++q)
              sts_u4(fp + 4 * q, u32x4{f2u(f[4 * q]), f2u(f[4 * q + 1]), f2u(f[4 * q + 2]), f2u(f[4 * q + 3])});
          }
        }
      } else {
        if (it < trips) {
          iir_fill(p, s_lanes, s_x, (int)it + IIR_AHEAD, lane);
          iir_commit();
          iir_wait<IIR_AHEAD>();  // block `it` of every lane has landed
          __syncwarp();
          if (it * IIR_BLK < len) iir_numerator<NB>(p, s_x + lane * IIR_XP, s_f + (it % 3) * 32 * IIR_FP + lane * IIR_FP, (int)it);
        }
        if (it >= 2) {  // outputs of block c, one lane's run per instruction
          const uint32_t c = it - 2, o = c * IIR_BLK;
          const float *fb = s_f + (c % 3) * 32 * IIR_FP + lane;
#pragma unroll 8
          for (int j = 0; j < 32; ++j) {
            const IirRun r = s_lanes.out[j];
            const float v = fb[j * IIR_FP];
            if (o >= r.skip && o + (uint32_t)lane < r.len) const_cast<float *>(r.p)[o + lane] = v;
          }
        }
      }
      __syncthreads();
    }
    if (!chain) iir_wait<0>();

    // ---- the chain verifies: lane s entered its samples in the state lane s - 1 left them in ----
    if (chain) {
      if (todo) {
#pragma unroll
        for (int k = 0; k < NA; ++k) y_end[k] = h[k];
        exact = exact || redo;  // a redo starts from its predecessor's final state
      }
      float prev[NA];
      bool differs = false;
#pragma unroll
      for (int k = 0; k < NA; ++k) {
        prev[k] = __shfl_up_sync(0xffffffffu, y_end[k], 1);
        differs = differs || f2u(prev[k]) != f2u(y_in[k]);
      }
      const bool bad = valid && !exact && differs;
      const uint32_t bad_mask = __ballot_sync(0xffffffffu, bad);
      // The first bad segment of each row is redone from its predecessor's state, which is final
      // (every segment before it verified). Later bad ones wait: their predecessors may change.
      const uint32_t row_lanes = S >= 32 ? 0xffffffffu : ((1u << S) - 1u) << ((uint32_t)lane & ~(S - 1));
      const bool first = bad && (bad_mask & row_lanes & ((1u << lane) - 1u)) == 0;
      if (first && p.redo) atomicAdd(p.redo, 1u);
      todo = redo = first;
      if (first) {
        begin = store;
#pragma unroll
        for (int k = 0; k < NA; ++k) h[k] = y_in[k] = prev[k];
      }
      if (lane == 0) s_more = bad_mask;
    }
    __syncthreads();
    if (s_more == 0) break;
  }

  // ---- the row's next carry: its last nb - 1 inputs and na outputs ----
  if (valid && end == p.n) {
    float *co = p.carry_out + r64 * p.C;
    if (chain) {
#pragma unroll
      for (int k = 0; k < NA; ++k) co[p.nb - 1 + k] = y_end[k];
    } else {
      for (uint32_t i = 0; i + 1 < p.nb; ++i) {
        const int g = (int)p.n - (int)(p.nb - 1) + (int)i;
        co[i] = g >= 0 ? in_row[g] : carry_row[(int)(p.nb - 1) + g];
      }
    }
  }
}

}  // namespace sdr
