// Warp-tile kernels (device only).
//
// One WORKER WARP owns one channel and walks its stream in tiles of 1024 complex
// samples (2048 input bytes). Lane l owns the tile's samples [32 l, 32 l + 32):
// exactly the input of one 8 kS/s PCM sample, because the reference's three
// decimators divide by 4 * 4 * 2 = 32. Every FIR stage therefore runs in
// registers; the few older samples a stage needs come from the lanes below by
// warp shuffle, and lanes near 0 reach into the PREVIOUS tile, whose registers the
// warp keeps (shfl_prev). No shared-memory staging of stage data, no CTA barrier
// between stages.
//
// Input arrives by cp.async (LDGSTS, 16 B per lane, fully coalesced) into a
// double-buffered, XOR-swizzled 2 KB slot per warp, so the tile after the current
// one is in flight while the current one is computed and both the global reads
// and the per-lane 64-byte shared reads are conflict free.
//
// The strictly sequential recurrences (IirFilter.cc:161-176) run with lane == channel:
// for AM/SSB in a second, tiny kernel over the numerators the FIR kernel leaves in HBM/L2
// (it overlaps the next call's FIR kernel on another stream); for WBFM, whose recurrence
// runs at the full 256 kS/s, in one extra warp per CTA one tile behind the workers, with a
// single CTA barrier per tile round.
#pragma once
#include "sdr_device.cuh"

#if SDR_DEVICE_BUILD
#include <cuda.h>  // CUtensorMap
#ifndef SDR_FIR_UNROLL
// Tiles per trip of the AM / SSB FIR loop. Two: the "previous tile" registers need no copying (the
// roles alternate) and stage 1 of one tile overlaps the shuffle chains of the other: AM x1024
// 0.1238 -> 0.1190 ms per step, SSB x8192 0.1453 -> 0.1374 (profiles/r02_am_fir_variants.txt).
#define SDR_FIR_UNROLL 2
#endif
#ifndef SDR_FM_UNROLL
#define SDR_FM_UNROLL 1  // tiles per trip of the NBFM loop (A/B builds)
#endif
namespace sdr { constexpr int FIR_UNROLL = SDR_FIR_UNROLL, FM_UNROLL = SDR_FM_UNROLL; }
namespace sdr {

constexpr int TILE = 1024;             // complex samples per tile
constexpr int TILE_BYTES = 2 * TILE;   // input bytes per tile
constexpr unsigned FULL = 0xffffffffu;

// value of "virtual lane (lane - j)": lanes below j read the previous tile's register
template <class T>
__device__ __forceinline__ T shfl_prev(T cur, T prev, int j, int lane) {
  return __shfl_sync(FULL, lane >= 32 - j ? prev : cur, (lane - j) & 31);
}
// after a tile with r valid lanes (1..32): the registers of the last 32 lanes of the stream
template <class T>
__device__ __forceinline__ T roll_prev(T cur, T prev, int r, int lane) {
  return __shfl_sync(FULL, lane >= r ? prev : cur, (lane + r) & 31);
}

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// 16-byte chunk q of a tile lives in slot q ^ ((q >> 3) & 3): conflict-free both for
// the coalesced fill (lane writes chunk 32 j + lane) and for the per-lane read of
// four consecutive chunks (lane reads chunks 4 lane + j).
__device__ __forceinline__ int tile_slot(int q) { return q ^ ((q >> 3) & 3); }

__device__ __forceinline__ void tile_fill(char *slot_base, const uint8_t *src, int lane, int valid_chunks) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int q = 32 * j + lane;
    if (q < valid_chunks) cp_async16(slot_base + 16 * tile_slot(q), src + 16 * q);
  }
}
__device__ __forceinline__ void tile_read(const char *slot_base, int lane, uint32_t (&w)[16]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const u32x4 v = lds_u4(slot_base + 16 * tile_slot(4 * lane + j));
    w[4 * j] = v.x; w[4 * j + 1] = v.y; w[4 * j + 2] = v.z; w[4 * j + 3] = v.w;
  }
}

// The same fill and read for FULL tiles with every address computed once per warp: the lane's
// shared addresses are loop invariants and the chunk offsets are immediates, so a tile costs
// four LDGSTS and four LDS.128 plus a handful of integer instructions (the generic versions
// above re-derive the swizzle and the shared window per tile: ~80 instructions).
//   fill: chunk 32 j + lane lands in slot 32 j + (lane ^ ((lane >> 3) & 3))
//   read: chunk 4 lane + j sits in slot 4 lane + (j ^ ((lane >> 1) & 3))
struct TileIo {
  uint32_t fill;    // shared address of the lane's chunk-0 destination in slot buffer 0
  uint32_t rd[4];   // shared addresses of the lane's four chunks in slot buffer 0
  __device__ __forceinline__ void init(const char *slots, int lane) {
    const uint32_t base = (uint32_t)__cvta_generic_to_shared(slots);
    fill = base + 16u * (uint32_t)(lane ^ ((lane >> 3) & 3));
    const uint32_t x = (uint32_t)(lane >> 1) & 3u;
#pragma unroll
    for (uint32_t j = 0; j < 4; ++j) rd[j] = base + 64u * (uint32_t)lane + 16u * (j ^ x);
  }
  // g = the tile's first byte + 16 * lane; buf = 0 or TILE_BYTES
  __device__ __forceinline__ void fill_full(uint32_t buf, const uint8_t *g) const {
    const uint32_t s = fill + buf;
    asm volatile(
        "cp.async.cg.shared.global [%0], [%1], 16;\n\t"
        "cp.async.cg.shared.global [%0+512], [%1+512], 16;\n\t"
        "cp.async.cg.shared.global [%0+1024], [%1+1024], 16;\n\t"
        "cp.async.cg.shared.global [%0+1536], [%1+1536], 16;" ::"r"(s), "l"(g)
        : "memory");
  }
  __device__ __forceinline__ void read(uint32_t buf, uint32_t (&w)[16]) const {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];"
                   : "=r"(w[4 * j]), "=r"(w[4 * j + 1]), "=r"(w[4 * j + 2]), "=r"(w[4 * j + 3])
                   : "r"(rd[j] + buf)
                   : "memory");
  }
};

// ---------------------------------------------------------------------------
// TMA tile loader. A full tile (2048 contiguous bytes of one channel) is a box of 16 rows x 128
// bytes of the 3-D view [channel][row of 128 B][128] of the caller's IQ array; ONE lane issues
// one cp.async.bulk.tensor per tile and the copy engine lands it in the warp's slot with the
// hardware's 128-byte swizzle (16-byte chunk c of row r sits at chunk c ^ (r & 7)), which makes
// the per-lane read of 64 consecutive bytes bank-conflict free exactly like the hand swizzle of
// TileIo: lanes 2r and 2r+1 share row r, and a quarter-warp's eight 16-byte reads fall on eight
// different chunk columns. Completion is an mbarrier per slot buffer (expect_tx = 2048 bytes).
// ---------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(bar), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_tile(uint32_t dst, const CUtensorMap *map, uint32_t row, uint32_t ch, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(0), "r"(row), "r"(ch), "r"(bar)
      : "memory");
}
// one lane of the (converged) warp, chosen by the hardware: the TMA issue path then has
// warp-uniform operands and needs no per-lane predicate
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}"
      : "=r"(pred));
  return pred != 0;
}
struct TmaIo {
  uint32_t slot;    // shared address of slot buffer 0 (1024-byte aligned); buffer b follows at + b * TILE_BYTES
  uint32_t bar;     // shared address of the buffers' mbarriers (8 bytes each)
  uint32_t rd[4];   // shared addresses of the lane's four 16-byte chunks in buffer 0
  uint32_t phase;   // bit b = parity the next wait on buffer b's barrier expects
  __device__ __forceinline__ void init(const char *slots, uint64_t *bars, int lane, int n_buffers) {
    slot = (uint32_t)__cvta_generic_to_shared(slots);
    bar = (uint32_t)__cvta_generic_to_shared(bars);
    const uint32_t r = (uint32_t)lane >> 1, c0 = 4u * ((uint32_t)lane & 1u);
#pragma unroll
    for (uint32_t j = 0; j < 4; ++j) rd[j] = slot + 128u * r + 16u * ((c0 + j) ^ (r & 7u));
    phase = 0;
    if (lane == 0) {
      for (int b = 0; b < n_buffers; ++b) mbar_init(bar + 8 * b, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
  }
  // one lane: arm buffer b's barrier and start the copy of tile `t` of channel `ch`
  __device__ __forceinline__ void issue(uint32_t b, const CUtensorMap *map, uint32_t t, uint32_t ch) const {
    mbar_expect_tx(bar + 8 * b, TILE_BYTES);
    tma_load_tile(slot + b * TILE_BYTES, map, t * (TILE_BYTES / 128), ch, bar + 8 * b);
  }
  __device__ __forceinline__ void wait(uint32_t b) {
    mbar_wait(bar + 8 * b, (phase >> b) & 1u);
    phase ^= 1u << b;
  }
  __device__ __forceinline__ void read(uint32_t b, uint32_t (&w)[16]) const {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];"
                   : "=r"(w[4 * j]), "=r"(w[4 * j + 1]), "=r"(w[4 * j + 2]), "=r"(w[4 * j + 3])
                   : "r"(rd[j] + b * TILE_BYTES)
                   : "memory");
  }
};

// two (int16_t)float conversions with x86 wrap semantics, packed
__device__ __forceinline__ uint32_t f2i16x2_wrap(float v0, float v1) {
  int r0 = f2i_rz(v0), r1 = f2i_rz(v1);
  if (!(fabsf(v0) < 2147483648.0f)) r0 = 0;
  if (!(fabsf(v1) < 2147483648.0f)) r1 = 0;
  return __byte_perm((uint32_t)r0, (uint32_t)r1, 0x5410);
}

// ---------------------------------------------------------------------------
// AM / SSB
// ---------------------------------------------------------------------------
// registers a worker carries from tile to tile (per lane)
template <bool SSB>
struct AmSsbCarry {
  uint32_t a7, b7;            // last rotation period of the lane, in front_end_ab's grouping
  uint32_t s1a0, s1a1, s1b0, s1b1;  // the lane's eight stage-1 outputs per arm (int8 x 4)
  uint32_t p;                 // stage-2 outputs: I pair in bytes 0-1, Q pair in bytes 2-3
  int dem;                    // the lane's demodulated value (AM magnitude / SSB phased sum): a small integer
  int y3a, y3b;               // SSB: stage-3 outputs (delay line and Hilbert history)
};

// A filter with every tap doubled: with the rounding constant doubled too, acc' = 2 acc
// exactly, so acc >> 15 is acc' >> 16 and an int8 result is simply byte 2 of acc' -- four
// results pack with three PRMTs instead of four shifts and three logic ops.
template <class F>
struct Doubled {
  static constexpr int N = F::N;
  SDR_HD static constexpr int tap(int k) { return 2 * F::tap(k); }
};
static_assert(2 * 6419 < 32768 && 2 * 5914 < 32768, "doubled AM stage-1/2 taps must fit int16");
// bytes 2 of four accumulators -> one word of four int8
__device__ __forceinline__ uint32_t pack_b2x4(int a0, int a1, int a2, int a3) {
  return __byte_perm(__byte_perm((uint32_t)a0, (uint32_t)a1, 0x7762), __byte_perm((uint32_t)a2, (uint32_t)a3, 0x7762),
                     0x5410);
}

template <bool SSB>
struct AmSsbTile {
  static constexpr int NREG = SSB ? 10 : 8;
  // state blob: two carry buffers of NREG words per lane, then a 16-byte tail: word 1 = y[n-1] of the
  // DC-removal IIR (dc_block_kernel's), word 2 = the VERSION word that says which carry buffer is
  // current: bit 31 = buffer index, bits 0-30 = id of the call that wrote it. The FIR kernel
  // reads a channel's carry and writes its new carry from different warps at unrelated times
  // of one launch, so the new carry goes to the OTHER buffer; a reader that already finds this
  // call's id in the version word takes the buffer the word does not name. All-zero = fresh.
  static constexpr int CARRY_WORDS = NREG * 32;
  static constexpr int TAIL_OFFSET = 2 * NREG * 128;
  static constexpr int STATE_BYTES = TAIL_OFFSET + 16;
  static constexpr int WARMUP_TILES = SSB ? 2 : 1;  // see amssb_fir_kernel

  __device__ __forceinline__ static void load_carry(AmSsbCarry<SSB> &c, const uint32_t *blob, int lane) {
    c.a7 = blob[0 * 32 + lane]; c.b7 = blob[1 * 32 + lane];
    c.s1a0 = blob[2 * 32 + lane]; c.s1a1 = blob[3 * 32 + lane];
    c.s1b0 = blob[4 * 32 + lane]; c.s1b1 = blob[5 * 32 + lane];
    c.p = blob[6 * 32 + lane];
    c.dem = (int)blob[7 * 32 + lane];
    if constexpr (SSB) { c.y3a = (int)blob[8 * 32 + lane]; c.y3b = (int)blob[9 * 32 + lane]; }
    else { c.y3a = 0; c.y3b = 0; }
  }
  __device__ __forceinline__ static void store_carry(const AmSsbCarry<SSB> &c, uint32_t *blob, int lane) {
    blob[0 * 32 + lane] = c.a7; blob[1 * 32 + lane] = c.b7;
    blob[2 * 32 + lane] = c.s1a0; blob[3 * 32 + lane] = c.s1a1;
    blob[4 * 32 + lane] = c.s1b0; blob[5 * 32 + lane] = c.s1b1;
    blob[6 * 32 + lane] = c.p;
    blob[7 * 32 + lane] = (uint32_t)c.dem;
    if constexpr (SSB) { blob[8 * 32 + lane] = (uint32_t)c.y3a; blob[9 * 32 + lane] = (uint32_t)c.y3b; }
  }

  // One tile of one channel. `w` = the lane's 64 input bytes. Returns what the
  // recurrence kernel consumes for this lane's PCM sample: the numerator of the DC-removal
  // filter, fl(x[n] - x[n-1]), where x is the AM magnitude estimate or the SSB phased sum. Both
  // are small integers (AM |x| <= 271, SSB <= 553 for 8-bit input: stage gains 113/128, 122/114,
  // 181/122, Hilbert 372/181), so the float difference is exact and travels as an int16.
  // Updates the carry to this tile's registers rolled by r valid lanes.
  // FULL_TILE: r == 32 is known at compile time (the hot loop); otherwise 1 <= r <= 32.
  template <bool FULL_TILE = false>
  __device__ __forceinline__ static int tile(const uint32_t (&w)[16], int fmt, bool lsb, AmSsbCarry<SSB> &pv, int lane, int r,
                                             uint32_t hring) {
    AmSsbCarry<SSB> cu;
    stage1_simt(w, fmt, pv, cu, lane);
    return rest<FULL_TILE>(cu, lsb, pv, lane, r, hring);
  }

  // stage 1 on the CUDA cores: front end, then 8 taps 4:1 on each arm (AmDemodulator.cc:349-374
  // through Decimator_int16). Leaves the lane's eight outputs per arm (int8 x 4 per word) and its
  // last rotation group in `cu`.
  __device__ __forceinline__ static void stage1_simt(const uint32_t (&w)[16], int fmt, const AmSsbCarry<SSB> &pv,
                                                     AmSsbCarry<SSB> &cu, int lane) {
    // a[g], b[g]: rotation period g in front_end_ab's grouping (I' in the low halves, Q' in the high halves)
    uint32_t a[8], b[8];
#pragma unroll
    for (int g = 0; g < 8; ++g) front_end_ab(fmt, w[2 * g], w[2 * g + 1], a[g], b[g]);
    cu.a7 = a[7];
    cu.b7 = b[7];
    const uint32_t am1 = shfl_prev(a[7], pv.a7, 1, lane), bm1 = shfl_prev(b[7], pv.b7, 1, lane);
    // output m: taps 7..4 meet period m - 1's samples s0..s3, taps 3..0 period m's (Decimator_int16.cc:310-351)
    using D = Doubled<taps::AM1>;
    constexpr uint32_t ti0 = pack16(D::tap(7), D::tap(4)), ti1 = pack16(D::tap(6), D::tap(5));  // I': (a.b0, a.b1), (b.b0, b.b1)
    constexpr uint32_t ti2 = pack16(D::tap(3), D::tap(0)), ti3 = pack16(D::tap(2), D::tap(1));
    constexpr uint32_t tq0 = pack16(D::tap(7), D::tap(6)), tq1 = pack16(D::tap(5), D::tap(4));  // Q': (a.b2, a.b3), (b.b2, b.b3)
    constexpr uint32_t tq2 = pack16(D::tap(3), D::tap(2)), tq3 = pack16(D::tap(1), D::tap(0));
    int ya[8], yb[8];
#pragma unroll
    for (int m = 0; m < 8; ++m) {
      const uint32_t pa = m == 0 ? am1 : a[m == 0 ? 0 : m - 1], pb = m == 0 ? bm1 : b[m == 0 ? 0 : m - 1];
      // the int8 result is byte 2 of the doubled accumulator
      ya[m] = dp2a_lo_ss(ti3, b[m], dp2a_lo_ss(ti2, a[m], dp2a_lo_ss(ti1, pb, dp2a_lo_ss(ti0, pa, 1 << 15))));
      yb[m] = dp2a_hi_ss(tq3, b[m], dp2a_hi_ss(tq2, a[m], dp2a_hi_ss(tq1, pb, dp2a_hi_ss(tq0, pa, 1 << 15))));
    }
    cu.s1a0 = pack_b2x4(ya[0], ya[1], ya[2], ya[3]);
    cu.s1a1 = pack_b2x4(ya[4], ya[5], ya[6], ya[7]);
    cu.s1b0 = pack_b2x4(yb[0], yb[1], yb[2], yb[3]);
    cu.s1b1 = pack_b2x4(yb[4], yb[5], yb[6], yb[7]);
  }

  // Everything after stage 1, from cu.s1a0..s1b1 (cu.a7 / cu.b7 are carried along untouched).
  // hring = shared address of the warp's window rings. A ring is 64 words: [0, 32) = the value of
  // the 32 lanes before the tile (the carry), [32, 64) = this tile's, so "the lane j below" is a load at an immediate
  // offset instead of a select, a lane index and a shuffle. Words 0-63: stage 3's window (pv.p / cu.p); words 64-127
  // (SSB): the Hilbert transformer's (y3b). The caller sets both carries at a piece's start (ring_init).
  template <bool FULL_TILE = false>
  __device__ __forceinline__ static int rest(AmSsbCarry<SSB> &cu, bool lsb, AmSsbCarry<SSB> &pv, int lane, int r,
                                             uint32_t hring) {
    // stage 2: 12 taps, 4:1
    const uint32_t pa0 = shfl_prev(cu.s1a0, pv.s1a0, 1, lane), pa1 = shfl_prev(cu.s1a1, pv.s1a1, 1, lane);
    const uint32_t pb0 = shfl_prev(cu.s1b0, pv.s1b0, 1, lane), pb1 = shfl_prev(cu.s1b1, pv.s1b1, 1, lane);
    int za0, za1, zb0, zb1;
    {
      const uint32_t w0[3] = {pa0, pa1, cu.s1a0}, w1[3] = {pa1, cu.s1a0, cu.s1a1};
      za0 = fir_s8<Doubled<taps::AM2>, 11, 3>(w0, 1 << 15);
      za1 = fir_s8<Doubled<taps::AM2>, 11, 3>(w1, 1 << 15);
      const uint32_t v0[3] = {pb0, pb1, cu.s1b0}, v1[3] = {pb1, cu.s1b0, cu.s1b1};
      zb0 = fir_s8<Doubled<taps::AM2>, 11, 3>(v0, 1 << 15);
      zb1 = fir_s8<Doubled<taps::AM2>, 11, 3>(v1, 1 << 15);
    }
    cu.p = pack_b2x4(za0, za1, zb0, zb1);

    // stage 3: 16 taps, 2:1. Window word i holds stage-2 samples at positions 2i, 2i+1
    // (I in bytes 0-1, Q in bytes 2-3); position pos meets tap 15 - pos.
    uint32_t q[8];
    q[7] = cu.p;
    {
      const uint32_t at = hring + 128u + 4u * lane;
      asm volatile("st.shared.u32 [%0], %1;" ::"r"(at), "r"(cu.p) : "memory");
      __syncwarp();
      window_ring<1>(q, at);
    }
    int acc_i = 1 << 14, acc_q = 1 << 14;
    stage3<0>(q, acc_i, acc_q);
    cu.y3a = (int)(int16_t)(acc_i >> 15);
    cu.y3b = (int)(int16_t)(acc_q >> 15);

    if constexpr (!SSB) {
      // magnitude estimate, tie -> q branch (AmDemodulator.cc:441-458)
      // |y3| <= 128 * 48394 / 32768 < 190 for 8-bit input, so none of the reference's int16 casts
      // can bite and max + min/2 is the same whichever branch a tie takes
      const int im = iabs(cu.y3a), qm = iabs(cu.y3b);
      cu.dem = max(im, qm) + (min(im, qm) >> 1);
    } else {
      // phasing network (SsbDemodulator.cc:569-590): delay line {0 x15, -32768}, Hilbert 31 taps
      const int x15 = shfl_prev(cu.y3a, pv.y3a, 15, lane);
      int acc = (1 << 14) + taps::SSB_DELAY::tap(15) * x15;
      acc = acc > 0x3fffffff ? 0x3fffffff : acc;
      acc = acc < -0x40000000 ? -0x40000000 : acc;
      const int i_delayed = (int)(int16_t)(acc >> 15);
      int h = (1 << 14) + taps::SSB_HILBERT::tap(0) * cu.y3b;
      // the 15 even lanes below through the ring: a store, a warp barrier and 15 loads at immediate offsets
      // instead of 15 select-and-shuffle pairs
      asm volatile("st.shared.u32 [%0], %1;" ::"r"(hring + 256u + 128u + 4u * lane), "r"(cu.y3b) : "memory");
      __syncwarp();
      hilbert_ring<2>(h, hring + 256u + 128u + 4u * lane);
      const int q_shifted = (int)(int16_t)(h >> 15);
      cu.dem = lsb ? i_delayed - q_shifted : i_delayed + q_shifted;
    }
    // numerator of the DC-removal IIR, b = {1, -1}: fl(1*x[n] + (-1)*x[n-1]) (IirFilter.cc:164). x is a
    // small integer, so the float products and the sum are exact: the difference is taken in int
    const int out = cu.dem - shfl_prev(cu.dem, pv.dem, 1, lane);

    // the last 32 lanes of the stream become the next tile's "previous" registers
    if (FULL_TILE || r == 32) {
      pv = cu;
    } else {
      pv.a7 = roll_prev(cu.a7, pv.a7, r, lane); pv.b7 = roll_prev(cu.b7, pv.b7, r, lane);
      pv.s1a0 = roll_prev(cu.s1a0, pv.s1a0, r, lane); pv.s1a1 = roll_prev(cu.s1a1, pv.s1a1, r, lane);
      pv.s1b0 = roll_prev(cu.s1b0, pv.s1b0, r, lane); pv.s1b1 = roll_prev(cu.s1b1, pv.s1b1, r, lane);
      pv.p = roll_prev(cu.p, pv.p, r, lane);
      pv.dem = roll_prev(cu.dem, pv.dem, r, lane);
      if constexpr (SSB) {
        pv.y3a = roll_prev(cu.y3a, pv.y3a, r, lane);
        pv.y3b = roll_prev(cu.y3b, pv.y3b, r, lane);
      }
    }
    {
      __syncwarp();  // every lane has read its windows
      asm volatile("st.shared.u32 [%0], %1;" ::"r"(hring + 4u * lane), "r"(pv.p) : "memory");
      if constexpr (SSB) asm volatile("st.shared.u32 [%0], %1;" ::"r"(hring + 256u + 4u * lane), "r"(pv.y3b) : "memory");
    }
    return out;
  }
  // the rings' carries at a piece's start
  __device__ __forceinline__ static void ring_init(uint32_t hring, const AmSsbCarry<SSB> &pv, int lane) {
    __syncwarp();  // the previous piece's last reads of the rings are done
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(hring + 4u * lane), "r"(pv.p) : "memory");
    if constexpr (SSB) asm volatile("st.shared.u32 [%0], %1;" ::"r"(hring + 256u + 4u * lane), "r"((uint32_t)pv.y3b) : "memory");
  }

  // ---- stage 1 on the tensor cores (slots in the TMA layout) ----
  // The two 8-tap 4:1 decimators as a warp-private int8 GEMM on the RAW bytes, mma.sync m16n8k32:
  //   D[16 x 8] += A[16 x 32] * B[32 x 8], twice per K (64 bytes) and per tap half
  //   A row h = the 64 raw bytes that end with half-window h's own 32 (a half-window = 16 samples =
  //     four outputs per arm; the 32 bytes before it hold the 4 samples of history the first output
  //     needs), fetched with ldmatrix straight from the swizzled slot -- no de-interleave, no
  //     offset, no rotation: those are in where the taps sit in B and which sign they carry;
  //   B column n: taps of I' output n (n < 4) or Q' output n - 4 of the half-window, split as
  //     256 * hi + lo (two int8 matrices); the u8 offset and the rounding constant are in the
  //     accumulator start. Table: am_mma_table() in the engine.
  // A lane ends up with two neighbouring outputs of one arm for eight half-windows; they go through
  // a 512-byte shared buffer into the layout stage 2 wants (lane = window, four packed words).
  // 8 LDSM + 16 IMMA + the transpose replace the packed-byte front end and 64 IDP.2A.
  // As in the NBFM tuner one thing is not linear: int8 negation leaves -128 alone
  // (IqDataProcessor.cc:594-607), so a raw byte 0 where the rotation negates makes the tile (and the
  // one after it, whose history it is) take the exact CUDA-core path.
  struct Mma {
    uint32_t b[8];      // taps fragments [hi / lo][k-step][b0, b1]
    int c[4];           // accumulator starts: hi column 2tq, hi 2tq+1, lo 2tq, lo 2tq+1
    // Byte offset in the slot of this lane's ldmatrix row, per k-step, for M-tiles 0 / 2 (`even`, + 1024
    // for M-tile 2) and 1 / 3 (`odd`, + 1024 for M-tile 3): an M-tile is 512 bytes further on, and the
    // 128-byte swizzle (chunk ^ (128-byte row & 7)) repeats every 1024 bytes.
    uint32_t even[2], odd[2];
    uint32_t hist_s;    // shared address of the warp's 32 bytes of raw history (bytes before the tile)
    uint32_t hist_row;  // lanes 0 and 16: their row of (M-tile 0, k-step 0) is the history; else 0
    uint32_t zmask;     // which bytes of this lane's fragment words sit where the rotation negates
    uint32_t xst, xld;  // transpose buffer: the lane's store base and its 16-byte read address
    __device__ __forceinline__ static uint32_t chunk_offset(int q) {  // 16-byte chunk q of the tile, q >= 0
      return (uint32_t)((q >> 3) * 128 + (((q & 7) ^ ((q >> 3) & 7)) * 16));
    }
    __device__ __forceinline__ void init(const uint32_t *tab, int fmt, uint32_t hist, uint32_t xbuf, int lane) {
      const uint32_t *t = tab + ((fmt == FMT_U8_OFFSET_ROTATE ? 0 : 32) + lane) * 12;
#pragma unroll
      for (int i = 0; i < 8; ++i) b[i] = t[i];
#pragma unroll
      for (int i = 0; i < 4; ++i) c[i] = (int)t[8 + i];
      const int r8 = (lane & 7) + 8 * ((lane >> 3) & 1);
#pragma unroll
      for (int kk = 0; kk < 2; ++kk) {
        // chunk of M-tile m: 2 * (16 m + r8) + 2 * (kk - 1) + (lane >> 4); M-tile 2's minus 1024 bytes
        // serves M-tile 0 as well (whose row 0, k-step 0 is the history: hist_row)
        const int q0 = 2 * r8 + 2 * (kk - 1) + (lane >> 4);
        even[kk] = chunk_offset(64 + q0) - 1024u;
        odd[kk] = chunk_offset(32 + q0);
      }
      hist_s = hist;
      hist_row = r8 == 0 ? hist + 16u * (uint32_t)(lane >> 4) : 0u;
      zmask = (lane & 1) ? 0x00808080u : 0x80000000u;  // odd tq: bytes 4, 5, 6 of a rotation group; even: byte 3
      const int g = lane >> 2, tq = lane & 3;
      xst = xbuf + (uint32_t)((g >> 1) * 16 + (tq >> 1) * 8 + (g & 1) * 4 + (tq & 1) * 2);
      xld = xbuf + 16u * (uint32_t)lane;
    }
  };
  template <bool U8>
  __device__ __forceinline__ static void imma_data(int (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    if constexpr (U8)
      asm("mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
          : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3])
          : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
    else
      asm("mma.sync.aligned.m16n8k32.row.col.s32.s8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
          : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3])
          : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
  template <int IMM>
  __device__ __forceinline__ static void ldsm4(uint32_t addr, uint32_t (&r)[4]) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4+%5];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(addr), "n"(IMM)
                 : "memory");
  }
  // slot_s = shared address of the tile. Fills cu.s1a0 .. cu.s1b1; returns false, with cu
  // untouched, if a raw byte 0 sits where the rotation negates.
  template <bool U8>
  __device__ __forceinline__ static bool stage1_mma(uint32_t slot_s, const Mma &mm, AmSsbCarry<SSB> &cu) {
    uint32_t z = 0;
    const uint32_t e0 = slot_s + mm.even[0], e1 = slot_s + mm.even[1], o0 = slot_s + mm.odd[0], o1 = slot_s + mm.odd[1];
#pragma unroll
    for (int half = 0; half < 2; ++half) {  // M-tiles 2 half, 2 half + 1 together: their IMMA chains interleave
      uint32_t a[2][2][4];
      if (half == 0) {
        ldsm4<0>(mm.hist_row ? mm.hist_row : e0, a[0][0]);
        ldsm4<0>(e1, a[0][1]);
        ldsm4<0>(o0, a[1][0]);
        ldsm4<0>(o1, a[1][1]);
      } else {
        ldsm4<1024>(e0, a[0][0]);
        ldsm4<1024>(e1, a[0][1]);
        ldsm4<1024>(o0, a[1][0]);
        ldsm4<1024>(o1, a[1][1]);
      }
      int hi[2][4], lo[2][4];
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        hi[m][0] = hi[m][2] = mm.c[0]; hi[m][1] = hi[m][3] = mm.c[1];
        lo[m][0] = lo[m][2] = mm.c[2]; lo[m][1] = lo[m][3] = mm.c[3];
      }
#pragma unroll
      for (int kk = 0; kk < 2; ++kk)
#pragma unroll
        for (int m = 0; m < 2; ++m) {
          imma_data<U8>(hi[m], a[m][kk], mm.b[2 * kk], mm.b[2 * kk + 1]);
          imma_data<U8>(lo[m], a[m][kk], mm.b[4 + 2 * kk], mm.b[4 + 2 * kk + 1]);
        }
      if constexpr (U8) {  // the tile's own bytes are the k-step 1 fragments
#pragma unroll
        for (int m = 0; m < 2; ++m)
#pragma unroll
          for (int i = 0; i < 4; ++i) z |= (a[m][1][i] - 0x01010101u) & ~a[m][1][i];
      }
      // rows g (e = 0) and g + 8 (e = 1) of M-tile mt: two neighbouring outputs of half-window
      // 16 mt + g + 8 e; the int8 result is byte 2 of the doubled accumulator (see Doubled)
#pragma unroll
      for (int m = 0; m < 2; ++m)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const uint32_t acc0 = (uint32_t)((hi[m][2 * e] << 8) + lo[m][2 * e]);
          const uint32_t acc1 = (uint32_t)((hi[m][2 * e + 1] << 8) + lo[m][2 * e + 1]);
          const uint32_t pair = __byte_perm(acc0, acc1, 0x0062);
          asm volatile("st.shared.u16 [%0], %1;" ::"r"(mm.xst + 128 * (2 * half + m) + 64 * e), "h"((uint16_t)pair) : "memory");
        }
    }
    if constexpr (U8) {
      if (__any_sync(FULL, (z & mm.zmask) != 0)) return false;
    }
    __syncwarp();
    uint32_t x[4];
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(x[0]), "=r"(x[1]), "=r"(x[2]), "=r"(x[3]) : "r"(mm.xld) : "memory");
    cu.s1a0 = x[0]; cu.s1a1 = x[1]; cu.s1b0 = x[2]; cu.s1b1 = x[3];
    return true;
  }
  // The last rotation group before the tile, as the planes stage1_simt's lane 0 reads: from the
  // raw history's last eight bytes. (Every lane gets the same words; lane 31's are what counts.)
  __device__ __forceinline__ static void planes_from_history(uint32_t hist_s, int fmt, AmSsbCarry<SSB> &pv) {
    uint32_t w0, w1;
    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(w0), "=r"(w1) : "r"(hist_s + 24) : "memory");
    front_end_ab(fmt, w0, w1, pv.a7, pv.b7);
  }
  // and back: the raw bytes of a rotation group from its planes (front_end_group's inverse;
  // wrapping int8 negation is its own inverse)
  __device__ __forceinline__ static void raw_from_planes(uint32_t a, uint32_t b, int fmt, uint32_t &w0, uint32_t &w1) {
    raw_from_ab(fmt, a, b, w0, w1);
  }

  template <int I>
  __device__ __forceinline__ static void stage3(const uint32_t (&q)[8], int &acc_i, int &acc_q) {
    if constexpr (I < 8) {
      constexpr uint32_t t = pack16(taps::AM3::tap(15 - 2 * I), taps::AM3::tap(14 - 2 * I));
      acc_i = dp2a_lo_ss(t, q[I], acc_i);
      acc_q = dp2a_hi_ss(t, q[I], acc_q);
      stage3<I + 1>(q, acc_i, acc_q);
    }
  }
  // stage 3's window from the ring: q[7 - j] = the word of the lane j below, j = 1..7
  template <int J>
  __device__ __forceinline__ static void window_ring(uint32_t (&q)[8], uint32_t at) {
    if constexpr (J < 8) {
      asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(q[7 - J]) : "r"(at), "n"(-4 * J) : "memory");
      window_ring<J + 1>(q, at);
    }
  }
  // the Hilbert transformer's window from its ring: even taps only (odd taps are zero); |x| <= 179 so the per-tap
  // clamp cannot fire. `at` = shared address of the lane's own word in [32, 64)
  template <int K>
  __device__ __forceinline__ static void hilbert_ring(int &h, uint32_t at) {
    if constexpr (K <= 30) {
      int v;
      asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(at), "n"(-4 * K) : "memory");
      h += taps::SSB_HILBERT::tap(K) * v;
      hilbert_ring<K + 2>(h, at);
    }
  }
};

// AM / SSB run as two kernels.
//
// amssb_fir_kernel: barrier-free worker warps. Everything up to the numerator of the
// DC-removal filter is finite-memory, so a channel's block can be cut anywhere in time: a
// warp that does not start at tile 0 first runs WARMUP tiles from an all-zero carry and
// discards their outputs, after which every register the next tile reads from the carry is
// exact (AM: the carry of tile t is a function of tile t's own lanes >= 22; SSB: the Hilbert
// history of lane 2 reaches five lanes into the tile before, hence two tiles). The launch is
// therefore treated as ONE sequence of tiles, cut into as many equal shares as the GPU holds
// worker warps in a single wave: the load balance is exact for any bank size (1024 channels
// or 8192) and there is no tail wave.
//
// dc_block_kernel: the sequential recurrence, lane == channel, over the numerators the FIR
// kernel left in `scratch`. The engine launches it on a second stream, so it overlaps the
// next call's FIR kernel.
// TMA = true: full tiles arrive by cp.async.bulk.tensor (TmaIo), one instruction of one lane per
// tile; false: by four cp.async per lane (TileIo). A partial last tile takes cp.async either way.
// NST = slot buffers per warp: NST - 1 tiles are in flight while one is computed.
// MMA (with TMA only): stage 1 on the tensor cores (AmSsbTile::stage1_mma).
// MINB = CTAs resident per SM the register budget is cut for (5: up to 96 registers, 6: 80; since the window rings the
// kernel needs 78-80 either way and six CTAs are resident).
template <bool SSB, bool TMA, int NST, bool MMA, int MINB = 5>
__global__ void __launch_bounds__(128, MINB) amssb_fir_kernel(const __grid_constant__ LaunchParams p,
                                                           const __grid_constant__ CUtensorMap tmap) {
  using T = AmSsbTile<SSB>;
  constexpr uint32_t WARMUP = T::WARMUP_TILES;
  static_assert(!MMA || TMA, "the tensor-core stage 1 reads the TMA slot layout");
  extern __shared__ __align__(1024) uint4 smem_raw[];
  __shared__ uint64_t s_bar[4][NST];
  __shared__ uint4 s_mma[MMA ? 4 : 1][34];  // per warp: 32 bytes of raw history, 512 bytes of transpose buffer
  __shared__ uint32_t s_ring[4][SSB ? 128 : 64];  // per warp: the window rings of AmSsbTile::rest
  // the warp index through a shuffle: the compiler then knows that everything derived from it (the
  // warp's share, its slot and barrier addresses, the TMA coordinates) is warp-uniform
  const int lane = threadIdx.x & 31, warp = __shfl_sync(FULL, (int)(threadIdx.x >> 5), 0);
  const uint32_t n_warps = p.aux;  // worker warps of the whole grid
  const uint32_t gw = blockIdx.x * (blockDim.x >> 5) + warp;
  trace_begin(p);
  if (gw >= n_warps) return;
  const uint32_t n_tiles = (p.n_samples + TILE - 1) / TILE;
  // The launch is one sequence of n_list * n_tiles tiles (channel-major); warp gw takes the
  // gw-th of n_warps equal shares of it, whatever channel boundaries fall inside.
  const uint64_t total = (uint64_t)p.n_list * n_tiles;
  uint64_t g0 = total * gw / n_warps;
  const uint64_t g1 = total * (gw + 1) / n_warps;

  char *slots = reinterpret_cast<char *>(smem_raw) + warp * NST * TILE_BYTES;
  TileIo io;
  TmaIo tio;
  if constexpr (TMA) tio.init(slots, s_bar[warp], lane, NST);
  else io.init(slots, lane);
  const int fmt = p.fmt;
  typename T::Mma mm;
  if constexpr (MMA) {
    const uint32_t ms = (uint32_t)__cvta_generic_to_shared(s_mma[warp]);
    mm.init(p.tab, fmt, ms, ms + 32, lane);
  }

  while (g0 < g1) {
    // the piece of one channel: tiles [t0, t1) of list entry li
    const uint32_t li = (uint32_t)(g0 / n_tiles);
    const uint32_t t0 = (uint32_t)(g0 - (uint64_t)li * n_tiles);
    const uint32_t t1 = (uint32_t)min((uint64_t)n_tiles, t0 + (g1 - g0));
    g0 += t1 - t0;
    const uint32_t ch = __shfl_sync(FULL, p.chan_ids[li], 0);
    if (p.allowed && !p.allowed[ch]) continue;  // squelched: the demodulator is not called, its state stays
    const uint8_t *src = p.iq + (uint64_t)ch * p.ch_stride;
    uint32_t *blob = reinterpret_cast<uint32_t *>(p.state + (uint64_t)ch * p.state_stride);
    // a piece that starts within WARMUP tiles of the block's head starts AT the head, from the
    // carried state; any other starts WARMUP tiles early from an all-zero carry
    const uint32_t tw = t0 <= WARMUP ? 0 : t0 - WARMUP;
    AmSsbCarry<SSB> pv;
    uint32_t *version = blob + T::TAIL_OFFSET / 4 + 2;  // tail words 0-1 belong to dc_block_kernel
    if (tw == 0) {
      const uint32_t v = *reinterpret_cast<volatile uint32_t *>(version);
      const uint32_t cur = (v & 0x7fffffffu) == p.call_id ? (v >> 31) ^ 1u : v >> 31;
      T::load_carry(pv, blob + cur * T::CARRY_WORDS, lane);
    } else {
      pv.a7 = pv.b7 = pv.s1a0 = pv.s1a1 = pv.s1b0 = pv.s1b1 = pv.p = 0;
      pv.dem = 0;
      pv.y3a = pv.y3b = 0;
    }
    const bool lsb = SSB && p.lsb[ch] != 0;
    const uint32_t hring = (uint32_t)__cvta_generic_to_shared(s_ring[warp]);
    T::ring_init(hring, pv, lane);
    // tensor-core stage 1: the raw bytes before the piece's first tile. force_simt: they (or,
    // later, the tile before) hold a byte the GEMM cannot represent. planes_ok: pv.a7 / pv.b7
    // hold the last rotation group (they do not after a tensor-core tile).
    bool force_simt = false, planes_ok = true;
    if constexpr (MMA) {
      __syncwarp();  // the previous piece's last reads of the history are done
      uint32_t w0, w1;
      T::raw_from_planes(pv.a7, pv.b7, fmt, w0, w1);  // all-zero carry -> 0x80 bytes: "no signal"
      if (lane < 6) asm volatile("st.shared.u32 [%0], %1;" ::"r"(mm.hist_s + 4 * lane), "r"(0x80808080u) : "memory");
      if (lane == 31) asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(mm.hist_s + 24), "r"(w0), "r"(w1) : "memory");
      if (fmt == FMT_U8_OFFSET_ROTATE)
        force_simt = __any_sync(FULL, lane == 31 && ((w0 & 0xff000000u) == 0 || (((w1 | 0xff000000u) - 0x01010101u) & ~(w1 | 0xff000000u) & 0x80808080u) != 0));
      __syncwarp();
    }

    // Full tiles [tw, tf) go through the lean loop; a partial last tile of the block (any
    // multiple of 32 samples) takes the generic path once.
    const uint32_t partial = (t1 == n_tiles && (p.n_samples & (TILE - 1))) ? 1u : 0u;
    const uint32_t tf = t1 - partial;
    const uint8_t *g = src + 16 * lane;  // the lane's chunk 0 of tile 0
    // the scratch row of tile tw ([list entry][row][32] int16); rows of warm-up tiles are walked
    // over but not written
    int16_t *sp = p.scratch + ((uint64_t)li * n_tiles + tw) * 32 + lane;
    // tile `tt` goes to slot buffer `b`: TMA or cp.async for a full tile, cp.async for the partial one
    auto fetch = [&](uint32_t tt, uint32_t b) {
      if (tt < tf) {
        if constexpr (TMA) { if (elect_one()) tio.issue(b, &tmap, tt, ch); }
        else io.fill_full(b * TILE_BYTES, g + (uint64_t)tt * TILE_BYTES);
      } else if (tt == tf && partial) {
        tile_fill(slots + b * TILE_BYTES, src + (uint64_t)tt * TILE_BYTES, lane, (int)(p.n_samples - tt * TILE) >> 3);
      }
    };
    __syncwarp();  // the previous piece's last reads of the slot buffers are done
#pragma unroll
    for (uint32_t k = 0; k < NST - 1; ++k) {
      fetch(tw + k, k);
      cp_async_commit();
    }
    uint32_t buf = 0;  // slot buffer of the tile being computed
#pragma unroll FIR_UNROLL
    for (uint32_t t = tw; t < tf; ++t) {
      fetch(t + NST - 1, buf == 0 ? NST - 1 : buf - 1);  // where tile t - 1 was; every lane has read it
      cp_async_commit();
      uint32_t w[16];
      int d;
      if constexpr (MMA) {
        tio.wait(buf);
        const uint32_t slot_s = tio.slot + buf * TILE_BYTES;
        AmSsbCarry<SSB> cu;
        cu.a7 = cu.b7 = 0;
        bool ok = false;
        if (!force_simt)
          ok = fmt == FMT_U8_OFFSET_ROTATE ? T::template stage1_mma<true>(slot_s, mm, cu) : T::template stage1_mma<false>(slot_s, mm, cu);
        if (!ok) {  // a clipping byte in this tile or right before it: the exact path
          tio.read(buf, w);
          if (!planes_ok) T::planes_from_history(mm.hist_s, fmt, pv);
          T::stage1_simt(w, fmt, pv, cu, lane);
        }
        planes_ok = !ok;
        force_simt = !ok && fmt == FMT_U8_OFFSET_ROTATE;
        // the tile's last 32 bytes (chunks 126, 127 sit at 121, 120 under the swizzle) become the history
        __syncwarp();
        if (lane < 8) {
          uint32_t hv;
          asm volatile("ld.shared.u32 %0, [%1];" : "=r"(hv) : "r"(slot_s + (lane < 4 ? 121u * 16u : 120u * 16u) + 4u * (lane & 3)) : "memory");
          asm volatile("st.shared.u32 [%0], %1;" ::"r"(mm.hist_s + 4 * lane), "r"(hv) : "memory");
        }
        __syncwarp();  // the slot may be refilled, the history read
        d = T::template rest<true>(cu, lsb, pv, lane, 32, hring);
      } else {
        if constexpr (TMA) {
          tio.wait(buf);
          tio.read(buf, w);
        } else {
          cp_async_wait<NST - 1>();
          __syncwarp();
          io.read(buf * TILE_BYTES, w);
        }
        __syncwarp();  // this buffer may be refilled once every lane has read it
        d = T::template tile<true>(w, fmt, lsb, pv, lane, 32, hring);
      }
      if (t >= t0) *sp = (int16_t)d;
      sp += 32;
      buf = buf + 1 == NST ? 0 : buf + 1;
    }
    if constexpr (MMA) {
      if (!planes_ok) T::planes_from_history(mm.hist_s, fmt, pv);  // the partial tile and the carry need them
    }
    if (partial) {
      cp_async_wait<0>();
      __syncwarp();
      uint32_t w[16];
      tile_read(slots + buf * TILE_BYTES, lane, w);
      const int r = (int)(p.n_samples - tf * TILE) >> 5;
      const int d = T::template tile<false>(w, fmt, lsb, pv, lane, r, hring);
      if (lane < r) *sp = (int16_t)d;  // tf >= t0 always
    }
    // Only the piece that ends the block leaves the channel's state: into the carry buffer
    // that is not current, then it publishes the switch. Pieces that read the carry later in
    // this launch recognise the call id and keep reading the old buffer.
    if (t1 == n_tiles) {
      const uint32_t nxt = (*reinterpret_cast<volatile uint32_t *>(version) >> 31) ^ 1u;
      T::store_carry(pv, blob + nxt * T::CARRY_WORDS, lane);
      __syncwarp();
      if (lane == 0) *reinterpret_cast<volatile uint32_t *>(version) = (nxt << 31) | p.call_id;
    }
  }
  if (p.trace && lane == 0) atomicMax(p.trace + 1, trace_now());
}

// y[n] = fl(d[n] - fl(-0.95f * y[n-1])), pcm[n] = (int16_t)(gain * y[n])
// (IirFilter.cc:161-176 with a = {-0.95}; AmDemodulator.cc:461-467, SsbDemodulator.cc:587-594).
//
// The recurrence is strictly sequential and bit-exactness forbids re-association, but it
// CONTRACTS: two trajectories fed the same numerators from different start states differ by
// 0.95^n times the initial difference until the difference drops below the rounding step, and a
// few steps later they are bit-identical for good (200,000 random starts per input class: median
// 360-500 steps, latest 717-807 depending on the run; tools/iir_merge.py,
// profiles/r02_iir_merge.txt). So a call's rows (a row = 32 PCM samples = one FIR tile) are cut
// into up to 32 SEGMENTS per channel and every (channel, segment) pair gets a lane:
//   * segment 0 starts from the carried y[n-1];
//   * segment s > 0 starts `warm_rows` rows early from y = 0 (or at row 0 from the carried state if
//     that is nearer), discards the outputs of the warm-up rows, and keeps the state it had when
//     it entered its own rows;
//   * afterwards lane s compares that state with the FINAL state of lane s - 1, bit for bit.
//     Equal: by induction every sample of segment s is what the serial loop computes. Different
//     (the trajectories had not merged yet; or never do: a y stuck on a denormal under
//     all-zero numerators): the first such segment of the channel is redone from the true state,
//     then the comparison is repeated -- the serial order, paid only where it is needed.
// The chain per call is warm_rows + seg_rows rows long instead of all rows.
//
// One CTA = TWO warps over the same 32 lanes. Warp 0 is the CHAIN warp: a row of numerators is 64
// contiguous bytes per lane (int16, [list entry][row][32]), fetched DC_PF rows ahead by cp.async into
// the lane's own ring in shared memory (an L2 round trip is several rows of chain long), then the 32
// dependent FMUL -> FSUB pairs, and the row's 32 y into a double-buffered row in shared memory --
// nothing else, because whatever else the warp issued would sit between the chain's dependent
// instructions (the first version converted and stored in the same warp: 1500 cycles per row against
// ~350, the float -> int conversions queue on the quarter-rate XU pipe; profiles/r02_dc_block_ncu.txt).
// Warp 1 is the CONVERTER, one row behind: gain, (int16_t) and the row's 64 bytes of PCM. One
// CTA barrier per row. At 64 threads x 64 registers a CTA fits beside the resident CTAs of the
// next call's FIR kernel without taking one's place.
constexpr int DC_PF = 8;             // rows in flight per lane
constexpr int DC_LANE_PITCH = 80;    // 64 + 16: lane-per-row 128-bit reads are bank-conflict free
constexpr int DC_STAGE_BYTES = 32 * DC_LANE_PITCH;
constexpr int DC_Y_PITCH = 144;      // 128 + 16, ditto
constexpr int DC_Y_BYTES = 32 * DC_Y_PITCH;

struct DcRows {
  uint32_t begin, store, end;  // rows [begin, end) are run, PCM is kept from row `store` on
};

// the lane's 64 bytes of row `g` into its place in ring stage `stage_s` (shared address)
__device__ __forceinline__ void dc_fetch_row(uint32_t stage_s, const int16_t *g) {
  asm volatile(
      "cp.async.cg.shared.global [%0], [%1], 16;\n\t"
      "cp.async.cg.shared.global [%0+16], [%1+16], 16;\n\t"
      "cp.async.cg.shared.global [%0+32], [%1+32], 16;\n\t"
      "cp.async.cg.shared.global [%0+48], [%1+48], 16;" ::"r"(stage_s), "l"(g)
      : "memory");
}

__global__ void __launch_bounds__(64, 16) dc_block_kernel(const __grid_constant__ LaunchParams p) {
  trace_begin(p);
  const int lane = threadIdx.x & 31;
  const bool chain = threadIdx.x < 32;
  const uint32_t S = p.seg_count, Lr = p.seg_rows;       // S: power of two <= 32
  const uint32_t idx = blockIdx.x * 32u + (uint32_t)lane;
  const uint32_t li = idx / S, s = idx & (S - 1);
  const uint32_t n_rows = (p.n_samples + TILE - 1) / TILE;
  const uint32_t n_pcm = p.n_samples >> 5;
  const float a1 = (float)(-0.95);

  bool valid = li < p.n_list && s * Lr < n_rows;
  const uint32_t ch = valid ? p.chan_ids[li] : 0;
  if (valid && p.allowed && !p.allowed[ch]) valid = false;  // squelched: the demodulator is not called
  float *tail = reinterpret_cast<float *>(p.state + (uint64_t)ch * p.state_stride + p.aux);
  const float carried = valid ? tail[1] : 0.f;
  const float gain = valid ? p.scale[ch] : 0.f;
  int16_t *out = p.pcm + (uint64_t)ch * p.pcm_stride;
  const int16_t *src = p.scratch + (uint64_t)(valid ? li : 0) * n_rows * 32;
  // |y| <= max(|y[-1]|, 20 |d|max) and |d| < 2^15: with |gain| < 500 and |y[-1]| < 2e6 no
  // gain * y can reach 2^31, where cvt.rzi saturates but x86 cvttss2si wraps
  const bool no_patch = __all_sync(FULL, !valid || (fabsf(gain) < 500.f && fabsf(carried) < 2e6f));

  __shared__ uint4 s_ring[DC_PF * DC_STAGE_BYTES / 16];
  __shared__ uint4 s_y[2 * DC_Y_BYTES / 16];
  __shared__ uint32_t s_begin[32];  // per pass: row the lane starts at, or ~0u if it sits the pass out
  __shared__ uint32_t s_more;       // another pass follows
  const uint32_t ring_s = (uint32_t)__cvta_generic_to_shared(s_ring) + (uint32_t)lane * DC_LANE_PITCH;
  char *ybuf = reinterpret_cast<char *>(s_y) + lane * DC_Y_PITCH;

  DcRows rw;
  rw.store = s * Lr;
  rw.end = min(rw.store + Lr, n_rows);
  rw.begin = rw.store > p.warm_rows ? rw.store - p.warm_rows : 0u;
  float y = rw.begin == 0 ? carried : 0.f;
  bool exact = rw.begin == 0;  // started from the true state: nothing to verify
  bool todo = valid, redo = false;
  float y_in = y, y_end = y;   // state on entering row `store`; state after row end - 1

  for (;;) {
    // ---- both warps learn which lanes run this pass and from which row ----
    if (chain) s_begin[lane] = todo ? rw.begin : ~0u;
    __syncthreads();
    const uint32_t begin = s_begin[lane];
    const bool on = begin != ~0u;
    const uint32_t trips = __reduce_max_sync(FULL, on ? rw.end - begin : 0u);

    if (chain) {
#pragma unroll
      for (int k = 0; k < DC_PF - 1; ++k) {
        if (on && begin + k < rw.end) dc_fetch_row(ring_s + k * DC_STAGE_BYTES, src + (uint64_t)(begin + k) * 32);
        cp_async_commit();
      }
    }
    uint32_t stage = 0;  // ring stage of the row being run
    // iteration `it`: the chain warp runs row begin + it, the converter row begin + it - 1
    for (uint32_t it = 0; it <= trips; ++it) {
      if (chain) {
        const uint32_t row = begin + it;
        const bool act = on && row < rw.end;
        if (it < trips) {
          {  // row + DC_PF - 1 goes where row - 1 was
            const uint32_t ahead = stage == 0 ? DC_PF - 1 : stage - 1;
            if (on && row + DC_PF - 1 < rw.end)
              dc_fetch_row(ring_s + ahead * DC_STAGE_BYTES, src + (uint64_t)(row + DC_PF - 1) * 32);
            cp_async_commit();
          }
          cp_async_wait<DC_PF - 1>();  // this lane's copy of `row` has landed
          uint32_t w[16];
#pragma unroll
          for (int j = 0; j < 4; ++j)
            asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];"
                         : "=r"(w[4 * j]), "=r"(w[4 * j + 1]), "=r"(w[4 * j + 2]), "=r"(w[4 * j + 3])
                         : "r"(ring_s + stage * DC_STAGE_BYTES + 16 * j)
                         : "memory");
          stage = stage + 1 == DC_PF ? 0 : stage + 1;
          if (act && row == rw.store) y_in = y;
          const bool keep = act && row >= rw.store;
          const uint32_t left = n_pcm - row * 32u;  // the call's last row may hold fewer than 32 samples
          const uint32_t r = act ? min(left, 32u) : 0u;
          char *yrow = ybuf + (it & 1) * DC_Y_BYTES;
          if (__any_sync(FULL, act && r < 32u)) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int dd[2] = {(int)(int16_t)(w[j] & 0xffffu), (int)w[j] >> 16};
#pragma unroll
              for (int i = 0; i < 2; ++i) {
                if ((uint32_t)(2 * j + i) < r) y = fsub(i2f(dd[i]), fmul(a1, y));
                if (keep) sts<float>(yrow + 4 * (2 * j + i), y);
              }
            }
          } else if (act) {
            const bool any_keep = keep;  // the converter reads the row only where it keeps it
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float d0 = i2f((int)(int16_t)(w[2 * j] & 0xffffu)), d1 = i2f((int)w[2 * j] >> 16);
              const float d2 = i2f((int)(int16_t)(w[2 * j + 1] & 0xffffu)), d3 = i2f((int)w[2 * j + 1] >> 16);
              const float y0 = fsub(d0, fmul(a1, y));
              const float y2 = fsub(d1, fmul(a1, y0));
              const float y3 = fsub(d2, fmul(a1, y2));
              y = fsub(d3, fmul(a1, y3));
              if (any_keep) sts_u4(yrow + 16 * j, u32x4{f2u(y0), f2u(y2), f2u(y3), f2u(y)});
            }
          }
        }
      } else if (it >= 1) {
        const uint32_t row = begin + it - 1;
        const bool keep = on && row < rw.end && row >= rw.store;
        if (keep) {
          const uint32_t r = min(n_pcm - row * 32u, 32u);
          const char *yrow = ybuf + ((it - 1) & 1) * DC_Y_BYTES;
          int16_t *dst = out + (uint64_t)row * 32;
          u32x4 v[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = lds_u4(yrow + 16 * j);
          uint32_t o[16];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float g0 = fmul(gain, u2f(v[j].x)), g1 = fmul(gain, u2f(v[j].y));
            const float g2 = fmul(gain, u2f(v[j].z)), g3 = fmul(gain, u2f(v[j].w));
            if (no_patch) {
              o[2 * j] = __byte_perm((uint32_t)f2i_rz(g0), (uint32_t)f2i_rz(g1), 0x5410);
              o[2 * j + 1] = __byte_perm((uint32_t)f2i_rz(g2), (uint32_t)f2i_rz(g3), 0x5410);
            } else {
              o[2 * j] = f2i16x2_wrap(g0, g1);
              o[2 * j + 1] = f2i16x2_wrap(g2, g3);
            }
          }
          if (r == 32u) {
#pragma unroll
            for (int j = 0; j < 4; ++j) stg_u4(dst + 8 * j, u32x4{o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]});
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if ((uint32_t)j < r) dst[j] = (int16_t)(o[j >> 1] >> (16 * (j & 1)));
          }
        }
      }
      __syncthreads();
    }
    if (chain) cp_async_wait<0>();

    // ---- the chain warp verifies: lane s entered its rows in the state lane s - 1 left them in ----
    if (chain) {
      if (todo) {
        y_end = y;
        exact = exact || redo;  // a redo starts from its predecessor's final state
      }
      const float prev_end = __shfl_up_sync(FULL, y_end, 1);
      const bool bad = valid && !exact && f2u(y_in) != f2u(prev_end);
      const uint32_t bad_mask = __ballot_sync(FULL, bad);
      // The first bad segment of each channel is redone from its predecessor's state, which is
      // final (every segment before it verified). Later bad ones wait: their predecessors may change.
      const uint32_t ch_lanes = S >= 32 ? 0xffffffffu : ((1u << S) - 1u) << ((uint32_t)lane & ~(S - 1));
      const bool first = bad && (bad_mask & ch_lanes & ((1u << lane) - 1u)) == 0;
      if (first && p.counters) atomicAdd(p.counters, 1u);
      todo = redo = first;
      if (first) {
        rw.begin = rw.store;
        y = prev_end;
        y_in = prev_end;
      }
      if (lane == 0) s_more = bad_mask;
    }
    __syncthreads();
    if (s_more == 0) break;
  }
  if (chain && valid && rw.end == n_rows) tail[1] = y_end;
  trace_end(p);
}


// ---------------------------------------------------------------------------
// Narrow-band FM (FmDemodulator.cc): no recurrence anywhere, so a worker warp runs the whole
// chain for its share of the launch's tiles and stores PCM itself; the CTA never synchronises.
//
// The 32-tap 4:1 tuner decimators (two thirds of the chain's multiply-adds) run on the tensor
// cores as a warp-private Toeplitz GEMM, mma.sync m16n8k32 int8 (IMMA.16832):
//   D[16 x 8] = A[16 x 128] * B[128 x 8]
//   B column n = the 128 RAW input bytes that end with window n's own 64 (a window = one
//     lane's 32 samples; the 64 bytes before it are the filter's history), fetched straight
//     from the cp.async tile buffer with ldmatrix -- no de-interleave, no offset, no rotation;
//   A row p (p < 8) = the taps that turn those bytes into I' output p of the window, row 8 + p
//     the same for Q': the Fs/4 rotation, the I/Q de-interleave and the decimation are all in
//     where the taps sit and which sign they carry. int16 taps = 256 * hi + lo, two int8
//     matrices; the u8 offset (u = s + 128) is a per-row constant folded into the accumulator
//     start together with the rounding constant 1 << 14. Tables: fm_mma_table() in the engine.
// 32 IMMA replace 256 IDP.2A + the packed-byte front end + the window shuffles. One thing is
// not linear: int8 negation leaves -128 alone (IqDataProcessor.cc:594-607), so a raw byte 0 in
// a position the rotation negates would come out as +128. Such bytes (a clipping ADC) are
// detected on the fragments already in registers and the tile takes the exact SIMT path.
// ---------------------------------------------------------------------------
struct FmCarry {
  float th[4];          // theta of the lane's last four 64 kS/s samples
  uint32_t dw[4];       // the lane's eight discriminator outputs (int16 x 2 per word)
  uint32_t ew;          // the lane's two 16 kS/s samples (int16 x 2)
  uint32_t hist;        // lanes 0-15: the last 64 raw input bytes (tuner history, logical order);
                        // lanes 16, 17: the sticky clamp-path flags
};

constexpr int FM_HIST_BYTES = 64;                          // raw bytes of tuner history before a tile
constexpr int FM_BUF_STRIDE = FM_HIST_BYTES + TILE_BYTES;  // [history | tile] twice per warp
constexpr int FM_TH_STRIDE = 12;                           // words per window row of the theta transpose
constexpr int FM_WARP_SMEM = 2 * FM_BUF_STRIDE + 32 * FM_TH_STRIDE * 4 + 64 * 4;  // + the audio ring
// fm_mma_table(): per format nine entries of [lane][4 words]: the A fragments [hi/lo][k-step]
// and the accumulator starts
constexpr int FM_TAB_WORDS_PER_FMT = 9 * 32 * 4;

struct FmTile {
  static constexpr int NREG = 10;
  // state blob: two carry buffers of NREG words per lane (versioned like AM/SSB, see
  // AmSsbTile), then a 16-byte tail whose word 2 is the version
  static constexpr int CARRY_WORDS = NREG * 32;
  static constexpr int TAIL_OFFSET = 2 * NREG * 128;
  static constexpr int STATE_BYTES = TAIL_OFFSET + 16;
  static constexpr int WARMUP_TILES = 1;

  __device__ __forceinline__ static void load_carry(FmCarry &c, const uint32_t *blob, int lane) {
#pragma unroll
    for (int i = 0; i < 4; ++i) { c.th[i] = u2f(blob[i * 32 + lane]); c.dw[i] = blob[(4 + i) * 32 + lane]; }
    c.ew = blob[8 * 32 + lane];
    c.hist = blob[9 * 32 + lane];
  }
  __device__ __forceinline__ static void store_carry(const FmCarry &c, uint32_t *blob, int lane) {
#pragma unroll
    for (int i = 0; i < 4; ++i) { blob[i * 32 + lane] = f2u(c.th[i]); blob[(4 + i) * 32 + lane] = c.dw[i]; }
    blob[8 * 32 + lane] = c.ew;
    blob[9 * 32 + lane] = c.hist;
  }

  // The raw history travels between calls in the format-independent form of the IQ dump
  // (signed, rotated, interleaved), so all-zero means "no signal yet" as in a fresh reference
  // object and a caller may change the input format between calls. Word `even` = bytes 0-3 of
  // a rotation group (I0 Q0 I1 Q1), else bytes 4-7 (I2 Q2 I3 Q3). Wrapping int8 negation is
  // its own inverse, so the round trip is exact.
  __device__ __forceinline__ static uint32_t hist_to_state(uint32_t raw, int fmt, bool even) {
    if (fmt != FMT_U8_OFFSET_ROTATE) return raw;
    return even ? offset_and_negate(byte_perm(raw, 0u, 0x2310), 0x00ff0000u, 0x00010000u)    // I0 Q0 -Q1 I1
                : offset_and_negate(byte_perm(raw, 0u, 0x2310), 0xff00ffffu, 0x01000101u);   // -I2 -Q2 Q3 -I3
  }
  __device__ __forceinline__ static uint32_t hist_from_state(uint32_t st, int fmt, bool even) {
    if (fmt != FMT_U8_OFFSET_ROTATE) return st;
    return even ? offset_and_negate(byte_perm(st, 0u, 0x2310), 0xff000000u, 0x01000000u)
                : offset_and_negate(byte_perm(st, 0u, 0x2310), 0x00ffffffu, 0x00010101u);
  }

  // ---- exact SIMT tuner (tiles with a clipping byte, and the reference for the GEMM) ----
  template <int M>
  __device__ __forceinline__ static int tuner_one(const uint32_t (&ext)[15]) {
    const uint32_t w[8] = {ext[M], ext[M + 1], ext[M + 2], ext[M + 3], ext[M + 4], ext[M + 5], ext[M + 6], ext[M + 7]};
    return (int)(int16_t)(fir_s8<taps::FM_TUNER, 31, 8>(w) >> 15);
  }
  template <int M>
  __device__ __forceinline__ static void tuner_all(const uint32_t (&ea)[15], const uint32_t (&eb)[15], const float *lut,
                                                   float (&th)[8]) {
    if constexpr (M < 8) {
      const int yi = tuner_one<M>(ea), yq = tuner_one<M>(eb);
      // theta = (float)atan2((double)q, (double)i), FmDemodulator.cc:476 (table, see sdr_engine.cu)
      th[M] = ld_lut(lut + (yq - FM_LUT_MIN) * FM_LUT_DIM + (yi - FM_LUT_MIN));
      tuner_all<M + 1>(ea, eb, lut, th);
    }
  }
  // window `win` (-1 = the history) of the tile buffer: its 64 raw bytes in logical order
  __device__ __forceinline__ static void read_window(const char *buf, int win, uint32_t (&w)[16]) {
    const int x = (win >> 1) & 3;  // -1 -> 3: the history is kept in window 31's physical order
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const u32x4 v = lds_u4(buf + 64 * win + 16 * (j ^ x));
      w[4 * j] = v.x; w[4 * j + 1] = v.y; w[4 * j + 2] = v.z; w[4 * j + 3] = v.w;
    }
  }
  __device__ __noinline__ static void theta_simt(const char *buf, int fmt, const float *lut, int lane, float (&th)[8]) {
    uint32_t w[16], a[8], b[8], ea[15], eb[15];
    read_window(buf, lane - 1, w);
#pragma unroll
    for (int g = 1; g < 8; ++g) front_end_group(fmt, w[2 * g], w[2 * g + 1], ea[g - 1], eb[g - 1]);
    read_window(buf, lane, w);
#pragma unroll
    for (int g = 0; g < 8; ++g) front_end_group(fmt, w[2 * g], w[2 * g + 1], a[g], b[g]);
#pragma unroll
    for (int i = 0; i < 8; ++i) { ea[7 + i] = a[i]; eb[7 + i] = b[i]; }
    tuner_all<0>(ea, eb, lut, th);
  }

  // ---- tensor-core tuner ----
  // Per-lane constants. The A fragments (32 words per lane) stay in shared memory, one
  // LDS.128 per fragment and use, so that six CTAs fit an SM: the chain is latency bound
  // (table gathers, shared-memory hand-overs, votes) and lives on occupancy.
  struct Mma {
    uint32_t tab_s;       // shared address of this lane's first A fragment ([hi/lo][k-step] 512 B apart)
    uint32_t rel0, rel1;  // ldmatrix row address of this lane for K bytes 0-63 / 64-127 of N-tile 0
    uint32_t zmask;       // which bytes of this lane's B words sit in negated positions
    __device__ __forceinline__ void init(const uint32_t *tab_smem, int lane) {
      tab_s = (uint32_t)__cvta_generic_to_shared(tab_smem) + 16u * (uint32_t)lane;
      const int row = lane & 7, i = lane >> 3;
      rel1 = (uint32_t)(64 * row + 16 * (i ^ ((row >> 1) & 3)));
      rel0 = (uint32_t)(64 * (row - 1) + 16 * (i ^ (((row - 1) >> 1) & 3)));  // row 0: the window before
      zmask = (lane & 1) ? 0x00808080u : 0x80000000u;  // tq odd: group bytes 4,5,6; even: byte 3
    }
  };
  __device__ __forceinline__ static void lds128(uint32_t addr, uint32_t (&r)[4]) {
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
  }
  template <bool U8>
  __device__ __forceinline__ static void imma(int (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    if constexpr (U8)
      asm("mma.sync.aligned.m16n8k32.row.col.s32.s8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
          : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3])
          : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
    else
      asm("mma.sync.aligned.m16n8k32.row.col.s32.s8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
          : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3])
          : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
  __device__ __forceinline__ static void ldmatrix4(uint32_t addr, uint32_t (&r)[4]) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(addr)
                 : "memory");
  }
  // theta of the tile's 256 tuner outputs, left in `thbuf` (row = window, FM_TH_STRIDE words).
  // buf_s = shared address of the tile buffer (its history sits in the 64 bytes before it).
  // Returns false, with nothing written, if a raw byte 0 sits where the rotation negates.
  template <bool U8>
  __device__ __forceinline__ static bool theta_mma(uint32_t buf_s, const Mma &m, const float *lut, float *thbuf, int lane) {
    const int g = lane >> 2, tq = lane & 3;
    uint32_t z = 0;
    float th[4][2];
    uint32_t c0[4];  // accumulator starts: hi row g, hi row g+8, lo row g, lo row g+8
    lds128(m.tab_s + 8 * 512, c0);
#pragma unroll
    for (int half = 0; half < 2; ++half) {  // two N-tiles (8 windows each) at a time: their MMA chains interleave
      uint32_t b[2][2][4];
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        ldmatrix4(buf_s + m.rel0 + 512 * (2 * half + cc), b[cc][0]);
        ldmatrix4(buf_s + m.rel1 + 512 * (2 * half + cc), b[cc][1]);
      }
      if constexpr (U8) {  // zero-byte test: every window's own bytes, and the history before window 0
#pragma unroll
        for (int cc = 0; cc < 2; ++cc)
#pragma unroll
          for (int i = 0; i < 4; ++i) z |= (b[cc][1][i] - 0x01010101u) & ~b[cc][1][i];
        if (half == 0) {
#pragma unroll
          for (int i = 0; i < 4; ++i) z |= (b[0][0][i] - 0x01010101u) & ~b[0][0][i];
        }
      }
      int hi[2][4], lo[2][4];
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        hi[cc][0] = hi[cc][1] = (int)c0[0]; hi[cc][2] = hi[cc][3] = (int)c0[1];
        lo[cc][0] = lo[cc][1] = (int)c0[2]; lo[cc][2] = lo[cc][3] = (int)c0[3];
      }
#pragma unroll
      for (int s = 0; s < 4; ++s) {
        uint32_t ahi[4], alo[4];
        lds128(m.tab_s + s * 512, ahi);
        lds128(m.tab_s + (4 + s) * 512, alo);
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          imma<U8>(hi[cc], ahi, b[cc][s >> 1][2 * (s & 1)], b[cc][s >> 1][2 * (s & 1) + 1]);
          imma<U8>(lo[cc], alo, b[cc][s >> 1][2 * (s & 1)], b[cc][s >> 1][2 * (s & 1) + 1]);
        }
      }
      // (int16_t)(acc >> 15), acc = 256 hi + lo: I' of windows 8c+2tq, +1 in [0],[1]; Q' in [2],[3]
#pragma unroll
      for (int cc = 0; cc < 2; ++cc)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int yi = (256 * hi[cc][e] + lo[cc][e]) >> 15, yq = (256 * hi[cc][2 + e] + lo[cc][2 + e]) >> 15;
          th[2 * half + cc][e] = ld_lut(lut + (yq - FM_LUT_MIN) * FM_LUT_DIM + (yi - FM_LUT_MIN));
        }
    }
    if constexpr (U8) {
      if (__any_sync(FULL, (z & m.zmask) != 0)) return false;
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      thbuf[(8 * c + 2 * tq) * FM_TH_STRIDE + g] = th[c][0];
      thbuf[(8 * c + 2 * tq + 1) * FM_TH_STRIDE + g] = th[c][1];
    }
    return true;
  }

  template <int J>
  __device__ __forceinline__ static void gather_e(uint32_t (&e)[20], uint32_t cur, uint32_t prev, int lane) {
    if constexpr (J <= 19) {
      e[19 - J] = shfl_prev(cur, prev, J, lane);
      gather_e<J + 1>(e, cur, prev, lane);
    }
  }

  // Everything after the tuner, from the lane's eight theta. big_a / big_b: sticky "clamp
  // reachable" flags of the previous tile (in) and of this tile (out). Returns the lane's PCM.
  __device__ __forceinline__ static int tile(const float (&th)[8], float k, FmCarry &pv, int lane, int r, bool &big_a,
                                             bool &big_b, uint32_t *ering) {
    FmCarry cu;
#pragma unroll
    for (int i = 0; i < 4; ++i) cu.th[i] = th[4 + i];

    // discriminator: taps {0,0,1,0,-1,0,0} -> theta[n-2] - theta[n-4]; wrap; * k; (int16_t)
    float te[12];
#pragma unroll
    for (int i = 0; i < 4; ++i) te[i] = shfl_prev(cu.th[i], pv.th[i], 1, lane);
#pragma unroll
    for (int i = 0; i < 8; ++i) te[4 + i] = th[i];
    // A quiet channel (a carrier that deviates a few kHz) never leaves (-pi, pi), and with the
    // default gains k * pi stays far below 2^31: both the FP64 wrap and the conversion's range
    // patch are skipped unless some lane of the warp needs them (one vote per tile).
    float df[8];
    float dmax = 0.f;
#pragma unroll
    for (int m = 0; m < 8; ++m) {
      df[m] = fsub(te[m + 2], te[m]);
      dmax = fmaxf(dmax, fabsf(df[m]));
    }
    const bool wraps = __any_sync(FULL, dmax >= 3.14159274101257324f);
    const bool patch = !(fabsf(k) < 3.0e8f);  // |k * dtheta| <= |k| * 2 pi < 2^31: cvt.rzi cannot saturate
    int d[8];
    if (wraps || patch) {  // warp-uniform: a real branch, so the quiet path executes none of it
#pragma unroll
      for (int m = 0; m < 8; ++m) d[m] = f2i16_wrap(fmul(k, wrap_pi_table(df[m])));  // df: a difference of two table values
    } else {
#pragma unroll
      for (int m = 0; m < 8; ++m) d[m] = (int)(int16_t)f2i_rz(fmul(k, df[m]));
    }
    int dabs = 0;
#pragma unroll
    for (int m = 0; m < 8; ++m) dabs = max(dabs, iabs(d[m]));
    const bool big = dabs > taps::FM_POST::SAFE;
#pragma unroll
    for (int i = 0; i < 4; ++i) cu.dw[i] = pack_i16x2(d[2 * i], d[2 * i + 1]);
    const bool cur_a = __any_sync(FULL, big && lane < r);
    const bool exact_a = cur_a || big_a;

    // post-demodulation decimator: 12 taps, 4:1 on int16
    uint32_t de[8];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      de[i] = shfl_prev(cu.dw[i], pv.dw[i], 1, lane);
      de[4 + i] = cu.dw[i];
    }
    int e0, e1;
    {
      const uint32_t w0[6] = {de[0], de[1], de[2], de[3], de[4], de[5]};
      const uint32_t w1[6] = {de[2], de[3], de[4], de[5], de[6], de[7]};
      e0 = (int)(int16_t)(fir_s16<taps::FM_POST, 11, 6>(w0, exact_a) >> 15);
      e1 = (int)(int16_t)(fir_s16<taps::FM_POST, 11, 6>(w1, exact_a) >> 15);
    }
    cu.ew = pack_i16x2(e0, e1);
    const bool cur_b =
        __any_sync(FULL, (iabs(e0) > taps::AUDIO40::SAFE || iabs(e1) > taps::AUDIO40::SAFE) && lane < r);
    const bool exact_b = cur_b || big_b;

    // audio decimator: 40 taps, 2:1: the lane's two samples and the 19 lanes below, through the
    // warp's 64-word ring in shared memory (previous tile's 32 words, then this tile's): one
    // store and twenty conflict-free loads instead of nineteen select-and-shuffle pairs
    ering[32 + lane] = cu.ew;
    __syncwarp();
    uint32_t ee[20];
#pragma unroll
    for (int i = 0; i < 20; ++i) ee[i] = ering[13 + lane + i];
    int acc;
    if (!exact_b) {
      acc = fir_s16_fast<taps::AUDIO40, 39, 20>(ee);
    } else {
      // middle taps first without the clamp; only if some lane's prefix sums left the clamp range
      // does the warp redo them in the reference's clamped order
      bool clean;
      acc = fir_s16_guard_mid_plain<taps::AUDIO40, 39, 20>(ee, clean);
      if (__any_sync(FULL, !clean)) acc = fir_s16_guard_mid<taps::AUDIO40, 39, 20>(ee);
      const bool clamped = __any_sync(FULL, !fir_s16_guard_tail_is_free<taps::AUDIO40>(acc));
      acc = fir_s16_guard_tail<taps::AUDIO40, 39, 20>(ee, acc, clamped);
    }
    const int pcm = (int)(int16_t)(acc >> 15);

    big_a = cur_a || (r < 32 && big_a);
    big_b = cur_b || (r < 32 && big_b);
    if (r == 32) {
#pragma unroll
      for (int i = 0; i < 4; ++i) { pv.th[i] = cu.th[i]; pv.dw[i] = cu.dw[i]; }
      pv.ew = cu.ew;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        pv.th[i] = roll_prev(cu.th[i], pv.th[i], r, lane);
        pv.dw[i] = roll_prev(cu.dw[i], pv.dw[i], r, lane);
      }
      pv.ew = roll_prev(cu.ew, pv.ew, r, lane);
    }
    __syncwarp();
    ering[lane] = pv.ew;  // the next tile's "previous" words
    return pcm;
  }
};

// Every warp is a worker. As in amssb_fir_kernel the launch is one channel-major sequence of
// tiles dealt out in equal shares: the chain has finite memory (the 40-tap audio decimator
// looks 20 lanes back, everything before it less), so a share that starts inside a block warms
// up on the tile before it; a share that starts within a tile of the head starts at the head.
template <int MIN_CTAS>
__global__ void __launch_bounds__(128, MIN_CTAS) fm_tile_kernel(const __grid_constant__ LaunchParams p) {
  extern __shared__ uint4 smem_raw[];
  __shared__ uint4 s_tab[FM_TAB_WORDS_PER_FMT / 4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  {
    const uint4 *src4 = reinterpret_cast<const uint4 *>(p.tab + (p.fmt == FMT_U8_OFFSET_ROTATE ? 0 : FM_TAB_WORDS_PER_FMT));
    for (int i = threadIdx.x; i < FM_TAB_WORDS_PER_FMT / 4; i += blockDim.x) s_tab[i] = src4[i];
  }
  __syncthreads();
  const uint32_t n_warps = p.aux;
  const uint32_t gw = blockIdx.x * (blockDim.x >> 5) + warp;
  if (gw >= n_warps) return;
  const uint32_t n_tiles = (p.n_samples + TILE - 1) / TILE;
  const uint64_t total = (uint64_t)p.n_list * n_tiles;
  uint64_t g0 = total * gw / n_warps;
  const uint64_t g1 = total * (gw + 1) / n_warps;

  char *wbase = reinterpret_cast<char *>(smem_raw) + warp * FM_WARP_SMEM;
  char *buf0 = wbase + FM_HIST_BYTES;  // tile buffers at buf0 and buf0 + FM_BUF_STRIDE
  float *thbuf = reinterpret_cast<float *>(wbase + 2 * FM_BUF_STRIDE);
  uint32_t *ering = reinterpret_cast<uint32_t *>(wbase + 2 * FM_BUF_STRIDE + 32 * FM_TH_STRIDE * 4);
  TileIo io;
  io.init(buf0, lane);
  const uint32_t buf0_s = (uint32_t)__cvta_generic_to_shared(buf0);
  const int fmt = p.fmt;
  FmTile::Mma mm;
  mm.init(reinterpret_cast<const uint32_t *>(s_tab), lane);
  constexpr uint32_t WARMUP = FmTile::WARMUP_TILES;

  while (g0 < g1) {
    const uint32_t li = (uint32_t)(g0 / n_tiles);
    const uint32_t t0 = (uint32_t)(g0 - (uint64_t)li * n_tiles);
    const uint32_t t1 = (uint32_t)min((uint64_t)n_tiles, t0 + (g1 - g0));
    g0 += t1 - t0;
    const uint32_t ch = p.chan_ids[li];
    if (p.allowed && !p.allowed[ch]) continue;  // squelched
    const uint8_t *src = p.iq + (uint64_t)ch * p.ch_stride;
    uint32_t *blob = reinterpret_cast<uint32_t *>(p.state + (uint64_t)ch * p.state_stride);
    uint32_t *tail = blob + FmTile::TAIL_OFFSET / 4;
    const uint32_t tw = t0 <= WARMUP ? 0 : t0 - WARMUP;
    FmCarry pv;
    bool big_a = false, big_b = false;
    __syncwarp();  // the previous piece is done with the buffers
    uint32_t off = 0;  // byte offset of the current tile buffer: 0 or FM_BUF_STRIDE
    if (tw == 0) {
      const uint32_t v = *reinterpret_cast<volatile uint32_t *>(tail + 2);
      const uint32_t cur = (v & 0x7fffffffu) == p.call_id ? (v >> 31) ^ 1u : v >> 31;
      FmTile::load_carry(pv, blob + cur * FmTile::CARRY_WORDS, lane);
      big_a = __shfl_sync(FULL, pv.hist, 16) != 0;
      big_b = __shfl_sync(FULL, pv.hist, 17) != 0;
      // raw history of the block's head, into window 31's physical order (chunk i at i ^ 3)
      if (lane < 16)
        *reinterpret_cast<uint32_t *>(buf0 - 64 + 16 * ((lane >> 2) ^ 3) + 4 * (lane & 3)) =
            FmTile::hist_from_state(pv.hist, fmt, (lane & 1) == 0);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) { pv.th[i] = 0.f; pv.dw[i] = 0; }
      pv.ew = 0;
      pv.hist = 0;
      // the history of the warm-up tile only feeds outputs that are thrown away
      if (lane < 16) *reinterpret_cast<uint32_t *>(buf0 - 64 + 4 * lane) = 0x80808080u;
    }
    ering[lane] = pv.ew;
    const float k = p.scale[ch];
    int16_t *out = p.pcm + (uint64_t)ch * p.pcm_stride;
    const uint32_t partial = (t1 == n_tiles && (p.n_samples & (TILE - 1))) ? 1u : 0u;
    const uint32_t tf = t1 - partial;
    const uint8_t *g = src + (uint64_t)tw * TILE_BYTES + 16 * lane;
    if (tw < tf) io.fill_full(off, g);
    else tile_fill(buf0 + off, g - 16 * lane, lane, (int)(p.n_samples - tw * TILE) >> 3);
    cp_async_commit();
#pragma unroll FM_UNROLL
    for (uint32_t t = tw; t < t1; ++t) {
      const uint32_t nxt = FM_BUF_STRIDE - off;
      g += TILE_BYTES;
      if (t + 1 < tf) io.fill_full(nxt, g);
      else if (t + 1 < t1) tile_fill(buf0 + nxt, g - 16 * lane, lane, (int)(p.n_samples - (t + 1) * TILE) >> 3);
      cp_async_commit();
      cp_async_wait<1>();
      __syncwarp();
      const int r = (int)min((uint32_t)TILE, p.n_samples - t * TILE) >> 5;
      bool ok = r == 32;  // a partial tile (stale bytes behind the data) takes the SIMT path
      if (ok) {
        ok = fmt == FMT_U8_OFFSET_ROTATE ? FmTile::theta_mma<true>(buf0_s + off, mm, p.lut, thbuf, lane)
                                         : FmTile::theta_mma<false>(buf0_s + off, mm, p.lut, thbuf, lane);
      }
      float th[8];
      if (ok) {
        __syncwarp();
        const u32x4 v0 = lds_u4(thbuf + lane * FM_TH_STRIDE), v1 = lds_u4(thbuf + lane * FM_TH_STRIDE + 4);
        th[0] = u2f(v0.x); th[1] = u2f(v0.y); th[2] = u2f(v0.z); th[3] = u2f(v0.w);
        th[4] = u2f(v1.x); th[5] = u2f(v1.y); th[6] = u2f(v1.z); th[7] = u2f(v1.w);
      } else {
        FmTile::theta_simt(buf0 + off, fmt, p.lut, lane, th);
      }
      // the next tile's history: this tile's last valid window, physical order kept
      if (lane < 16) {
        const int last = r - 1;
        const uint32_t wv = *reinterpret_cast<const uint32_t *>(buf0 + off + 64 * last + 16 * ((lane >> 2) ^ ((last >> 1) & 3)) +
                                                                4 * (lane & 3));
        *reinterpret_cast<uint32_t *>(buf0 + nxt - 64 + 16 * ((lane >> 2) ^ 3) + 4 * (lane & 3)) = wv;
        pv.hist = wv;  // raw, logical order: chunk lane >> 2, word lane & 3
      }
      __syncwarp();  // buffer `off` may be refilled (tile t+2), thbuf rewritten
      const int pcm = FmTile::tile(th, k, pv, lane, r, big_a, big_b, ering);
      if (t >= t0 && lane < r) out[(uint64_t)t * 32 + lane] = (int16_t)pcm;
      off = nxt;
    }
    if (t1 == n_tiles) {
      const uint32_t nv = (*reinterpret_cast<volatile uint32_t *>(tail + 2) >> 31) ^ 1u;
      if (lane < 16) pv.hist = FmTile::hist_to_state(pv.hist, fmt, (lane & 1) == 0);
      if (lane == 16) pv.hist = big_a;
      if (lane == 17) pv.hist = big_b;
      FmTile::store_carry(pv, blob + nv * FmTile::CARRY_WORDS, lane);
      __syncwarp();
      if (lane == 0) *reinterpret_cast<volatile uint32_t *>(tail + 2) = (nv << 31) | p.call_id;
    }
  }
}

// ---------------------------------------------------------------------------
// Wide-band FM (WbFmDemodulator.cc). Three stages pipelined over tile rounds:
//   round k, worker warp of a channel : C(k-2) then A(k)
//   round k, recurrence warp          : B(k-1), lane == channel
// A: front end, 16-tap pre-filter at 256 kS/s -> (int8) -> atan2 table -> first
//    difference, wrap, * k -> numerator of the de-emphasis filter: u[n], 1024 floats
//    into ring slot k&1 of the channel.
// B: y[n] = fl(u[n] - fl(a1 * y[n-1])), written back in place. Nothing else: the warp's
//    dependent FMUL->FSUB chain is the critical path of a round.
// C: d[n] = (int16_t)y[n] -> 8-tap 4:1 -> 12-tap 4:1 -> 40-tap 2:1 -> PCM, read from slot
//    (k-2)&1 = k&1 before A(k) overwrites it.
// One CTA barrier per round.
// ---------------------------------------------------------------------------
struct WbCarry {
  uint32_t a[4], b[4];  // the lane's rotation groups 4..7: 16 samples of pre-filter history
  float th31;           // theta of the lane's last sample
  float v31;            // k * dtheta of the lane's last sample
  uint32_t dw[2];       // the lane's last four de-emphasised samples (int16 x 2 per word)
  uint32_t e1w[4];      // the lane's eight decimator-1 outputs
  uint32_t ew;          // the lane's two decimator-2 outputs
};

struct WbTile {
  static constexpr int NREG_A = 10, NREG_C = 7, NREG = NREG_A + NREG_C;
  // blob: NREG words per lane; tail: y[n-1], v[n-1] of the de-emphasis IIR (NOT cleared
  // by a reset, WbFmDemodulator.cc:304-320), clamp flag
  static constexpr int STATE_BYTES = NREG * 128 + 16;
  static constexpr int MAX_WORKERS = 19;
  // Warp w issues from scheduler w & 3. The recurrence warp (warp 3) carries the round's
  // critical path, a dependent FMUL->FSUB chain; how many workers may share its scheduler is
  // a launch parameter (s3). Measured on B200: once the warp does nothing but the chain,
  // sharing with up to four workers costs nothing (profiles/r01v2_wbfm_sweep.txt).
  // s3 = how many workers may share scheduler 3 with the recurrence warp
  __host__ __device__ static constexpr bool is_worker(int warp, int s3) {
    return (warp & 3) != 3 || (warp != 3 && (warp >> 2) <= s3);
  }
  __host__ __device__ static constexpr int worker_index(int warp, int s3) {
    int n = 0;
    for (int w = 0; w < warp; ++w) n += is_worker(w, s3) ? 1 : 0;
    return n;
  }
  __host__ __device__ static constexpr int warps_for(int workers, int s3) {
    int n = 4;
    while (worker_index(n, s3) < workers) ++n;
    return n;
  }
  static constexpr int RING_BYTES = 2 * 4096 + 16;  // two slots + pad: row stride == 16 (mod 128)
  __host__ __device__ static constexpr int smem_bytes(int nw) { return nw * (TILE_BYTES + RING_BYTES) + 64; }

  // u[n] of row (= lane) `row`, 16-byte chunk j (four samples): rows are XOR-swizzled so
  // that a quarter-warp writing chunk j of eight consecutive rows hits distinct banks
  __device__ __forceinline__ static int u_off(int row, int j) { return 128 * row + 16 * (j ^ (row & 7)); }

  // ---- A ----
  // The pre-filter runs with every tap doubled (|2 h| <= 31866 still fits int16) and the
  // rounding constant doubled: acc' = 2 acc exactly, so (acc >> 15) & 255 -- the int8
  // truncation of WbFmDemodulator.cc:393-397 -- is simply byte 2 of acc'.
  struct Pre2 {
    static constexpr int N = taps::WB_PRE::N;
    SDR_HD static constexpr int tap(int k) { return 2 * taps::WB_PRE::tap(k); }
  };
  // table index of sample N: byte 0 = (uint8)(i + 128), byte 1 = (uint8)(q + 128)
  template <int N>
  __device__ __forceinline__ static uint32_t lut_index(const uint32_t (&ea)[12], const uint32_t (&eb)[12]) {
    const uint32_t ai = (uint32_t)fir_s8<Pre2, 16 + N, 12>(ea, 1 << 15);
    const uint32_t aq = (uint32_t)fir_s8<Pre2, 16 + N, 12>(eb, 1 << 15);
    return (__byte_perm(ai, aq, 0x7762) & 0xffffu) ^ 0x8080u;
  }
  template <int N0>
  __device__ __forceinline__ static void theta4(const uint32_t (&ea)[12], const uint32_t (&eb)[12], const float *lut,
                                                float (&th)[4]) {
    // theta = table[(uint8)(q+128)][(uint8)(i+128)] (WbFmDemodulator.cc:458-462)
    const uint32_t x0 = lut_index<N0>(ea, eb), x1 = lut_index<N0 + 1>(ea, eb);
    const uint32_t x2 = lut_index<N0 + 2>(ea, eb), x3 = lut_index<N0 + 3>(ea, eb);
    th[0] = ld_lut(lut + x0);
    th[1] = ld_lut(lut + x1);
    th[2] = ld_lut(lut + x2);
    th[3] = ld_lut(lut + x3);
  }
  // four samples from their thetas: returns the chunk of u, advances (th_prev, v_prev)
  __device__ __forceinline__ static u32x4 u4(const float (&th)[4], float k, float &th_prev, float &v_prev) {
    const float b0 = (float)(0.0253863), b1 = (float)(0.0253863);
    float u[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float v = fmul(k, wrap_pi(fsub(th[i], th_prev)));
      u[i] = fadd(fmul(b0, v), fmul(b1, v_prev));
      th_prev = th[i];
      v_prev = v;
    }
    return u32x4{f2u(u[0]), f2u(u[1]), f2u(u[2]), f2u(u[3])};
  }
  template <int J>
  __device__ __forceinline__ static void u_chunks(const uint32_t (&ea)[12], const uint32_t (&eb)[12], const float *lut,
                                                  float k, float &th_prev, float &v_prev, char *slot, int lane) {
    if constexpr (J < 7) {
      float th[4];
      theta4<4 * J>(ea, eb, lut, th);
      sts_u4(slot + u_off(lane, J), u4(th, k, th_prev, v_prev));
      u_chunks<J + 1>(ea, eb, lut, k, th_prev, v_prev, slot, lane);
    }
  }

  // A(k): w = the lane's 64 input bytes; writes the lane's 32 u values into `slot`.
  // v_boundary: v[n-1] at the head of the tile (carried; scaled with the gain it was made with).
  __device__ __forceinline__ static void part_a(const uint32_t (&w)[16], int fmt, float k, const float *lut, WbCarry &pv,
                                                float &v_boundary, char *slot, int lane, int r) {
    uint32_t a[8], b[8];
#pragma unroll
    for (int g = 0; g < 8; ++g) front_end_group(fmt, w[2 * g], w[2 * g + 1], a[g], b[g]);
    uint32_t ea[12], eb[12];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      ea[i] = shfl_prev(a[4 + i], pv.a[i], 1, lane);
      eb[i] = shfl_prev(b[4 + i], pv.b[i], 1, lane);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) { ea[4 + i] = a[i]; eb[4 + i] = b[i]; }

    // The lane's LAST four samples first: theta[31] and v[31] = k * wrap(theta[31] - theta[30])
    // depend on this lane's data only, and the lane above needs them before it can start.
    float th_last[4];
    theta4<28>(ea, eb, lut, th_last);
    const float my_th31 = th_last[3];
    const float my_v31 = fmul(k, wrap_pi(fsub(th_last[3], th_last[2])));
    float th_prev = shfl_prev(my_th31, pv.th31, 1, lane);
    float v_prev = __shfl_up_sync(FULL, my_v31, 1);
    if (lane == 0) v_prev = v_boundary;
    u_chunks<0>(ea, eb, lut, k, th_prev, v_prev, slot, lane);
    sts_u4(slot + u_off(lane, 7), u4(th_last, k, th_prev, v_prev));

    // carry: last valid lane's values feed the next tile
    v_boundary = __shfl_sync(FULL, my_v31, r - 1);
    if (r == 32) {
#pragma unroll
      for (int i = 0; i < 4; ++i) { pv.a[i] = a[4 + i]; pv.b[i] = b[4 + i]; }
      pv.th31 = my_th31;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        pv.a[i] = roll_prev(a[4 + i], pv.a[i], r, lane);
        pv.b[i] = roll_prev(b[4 + i], pv.b[i], r, lane);
      }
      pv.th31 = roll_prev(my_th31, pv.th31, r, lane);
    }
  }

  // ---- C ----
  template <int M>
  __device__ __forceinline__ static int dec1_one(const uint32_t (&ext)[18]) {
    const uint32_t w[4] = {ext[2 * M], ext[2 * M + 1], ext[2 * M + 2], ext[2 * M + 3]};
    static_assert(taps::WB_DEC1::SAFE >= 32768, "decimator 1 must be clamp-free");
    return (int)(int16_t)(fir_s16_fast<taps::WB_DEC1, 7, 4>(w) >> 15);
  }
  // C(j): dW = the lane's 32 de-emphasised samples; returns the lane's PCM sample
  __device__ __forceinline__ static int part_c(const uint32_t (&dW)[16], WbCarry &pv, int lane, int r, bool &big_b) {
    // decimator 1: 8 taps, 4:1; output m uses d[4m-4 .. 4m+3]
    uint32_t ext[18];
    ext[0] = shfl_prev(dW[14], pv.dw[0], 1, lane);
    ext[1] = shfl_prev(dW[15], pv.dw[1], 1, lane);
#pragma unroll
    for (int i = 0; i < 16; ++i) ext[2 + i] = dW[i];
    uint32_t e1w[4];
    e1w[0] = pack_i16x2(dec1_one<0>(ext), dec1_one<1>(ext));
    e1w[1] = pack_i16x2(dec1_one<2>(ext), dec1_one<3>(ext));
    e1w[2] = pack_i16x2(dec1_one<4>(ext), dec1_one<5>(ext));
    e1w[3] = pack_i16x2(dec1_one<6>(ext), dec1_one<7>(ext));
    // decimator 2: 12 taps, 4:1, clamp-free (decimator 1 output <= 29126 <= FM_POST::SAFE)
    uint32_t de[8];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      de[i] = shfl_prev(e1w[i], pv.e1w[i], 1, lane);
      de[4 + i] = e1w[i];
    }
    const uint32_t w0[6] = {de[0], de[1], de[2], de[3], de[4], de[5]};
    const uint32_t w1[6] = {de[2], de[3], de[4], de[5], de[6], de[7]};
    const int e0 = (int)(int16_t)(fir_s16_fast<taps::FM_POST, 11, 6>(w0) >> 15);
    const int e1 = (int)(int16_t)(fir_s16_fast<taps::FM_POST, 11, 6>(w1) >> 15);
    const uint32_t ew = pack_i16x2(e0, e1);
    const bool cur_b =
        __any_sync(FULL, (iabs(e0) > taps::AUDIO40::SAFE || iabs(e1) > taps::AUDIO40::SAFE) && lane < r);
    const bool exact_b = cur_b || big_b;
    // audio decimator: 40 taps, 2:1
    uint32_t ee[20];
    ee[19] = ew;
    FmTile::gather_e<1>(ee, ew, pv.ew, lane);
    const int pcm = (int)(int16_t)(fir_s16<taps::AUDIO40, 39, 20>(ee, exact_b) >> 15);
    big_b = cur_b || (r < 32 && big_b);
    if (r == 32) {
      pv.dw[0] = dW[14]; pv.dw[1] = dW[15];
#pragma unroll
      for (int i = 0; i < 4; ++i) pv.e1w[i] = e1w[i];
      pv.ew = ew;
    } else {
      pv.dw[0] = roll_prev(dW[14], pv.dw[0], r, lane);
      pv.dw[1] = roll_prev(dW[15], pv.dw[1], r, lane);
#pragma unroll
      for (int i = 0; i < 4; ++i) pv.e1w[i] = roll_prev(e1w[i], pv.e1w[i], r, lane);
      pv.ew = roll_prev(ew, pv.ew, r, lane);
    }
    return pcm;
  }

  __device__ __forceinline__ static void load_carry(WbCarry &c, const uint32_t *blob, int lane) {
#pragma unroll
    for (int i = 0; i < 4; ++i) { c.a[i] = blob[i * 32 + lane]; c.b[i] = blob[(4 + i) * 32 + lane]; }
    c.th31 = u2f(blob[8 * 32 + lane]);
    c.v31 = 0.f;
    c.dw[0] = blob[10 * 32 + lane]; c.dw[1] = blob[11 * 32 + lane];
#pragma unroll
    for (int i = 0; i < 4; ++i) c.e1w[i] = blob[(12 + i) * 32 + lane];
    c.ew = blob[16 * 32 + lane];
  }
  __device__ __forceinline__ static void store_carry(const WbCarry &c, uint32_t *blob, int lane) {
#pragma unroll
    for (int i = 0; i < 4; ++i) { blob[i * 32 + lane] = c.a[i]; blob[(4 + i) * 32 + lane] = c.b[i]; }
    blob[8 * 32 + lane] = f2u(c.th31);
    blob[9 * 32 + lane] = 0;
    blob[10 * 32 + lane] = c.dw[0]; blob[11 * 32 + lane] = c.dw[1];
#pragma unroll
    for (int i = 0; i < 4; ++i) blob[(12 + i) * 32 + lane] = c.e1w[i];
    blob[16 * 32 + lane] = c.ew;
  }
};

// blockDim = 32 * WbTile::warps_for(p.G, s3): warp 3 runs the recurrences, the warps
// WbTile::is_worker() names are workers, the rest only keep the barrier count. All roles
// share one round loop, so every thread of the CTA meets the same barrier instruction.
__global__ void __launch_bounds__(768, 1) wbfm_tile_kernel(const __grid_constant__ LaunchParams p) {
  using T = WbTile;
  extern __shared__ uint4 smem_raw[];
  char *smem = reinterpret_cast<char *>(smem_raw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nw = (int)p.G;
  const int s3 = (int)p.aux;
  const bool is_iir = warp == 3;
  const bool is_worker = !is_iir && T::is_worker(warp, s3);
  const uint32_t list0 = blockIdx.x * (uint32_t)nw;
  const int n_here = (int)min((uint32_t)nw, p.n_list - list0);
  const uint32_t n_tiles = (p.n_samples + TILE - 1) / TILE;
  char *ring_base = smem + nw * TILE_BYTES;   // after nw input slots: nw rings of RING_BYTES

  const int slot_id = is_iir ? lane : T::worker_index(warp, s3);  // channel slot in this CTA
  const bool owned = (is_iir || is_worker) && slot_id < n_here;
  const uint32_t ch = owned ? p.chan_ids[list0 + slot_id] : 0;
  const bool active = owned && !(p.allowed && !p.allowed[ch]);  // a squelched channel is skipped
  uint32_t *blob = reinterpret_cast<uint32_t *>(p.state + (uint64_t)ch * p.state_stride);
  char *ring = ring_base + (active ? slot_id : 0) * T::RING_BYTES;

  // ---- worker state ----
  WbCarry pv;
  const uint8_t *src = p.iq + (uint64_t)ch * p.ch_stride;
  int16_t *out = p.pcm + (uint64_t)ch * p.pcm_stride;
  char *in_slot = smem + (active && is_worker ? slot_id : 0) * TILE_BYTES;
  float k = 0.f, v_boundary = 0.f;
  bool big_b = false, no_patch = false;
  // ---- recurrence state ----
  float y1 = 0.f;
  const float a1 = (float)(-0.9492274);

  if (is_worker) {
    if (active) {
      T::load_carry(pv, blob, lane);
      v_boundary = u2f(blob[T::NREG * 32 + 1]);
      big_b = blob[T::NREG * 32 + 2] != 0;
      k = p.scale[ch];
      // |y| <= max(|y[-1]|, |u|max / (1 - |a1|)) < 3.2 |k|: with |k| < 1e8 and |y[-1]| < 1e9 no
      // value can reach 2^31, where cvt.rzi (saturating) and x86 cvttss2si (wrapping) differ
      no_patch = fabsf(k) < 1e8f && fabsf(u2f(blob[T::NREG * 32])) < 1e9f;
      tile_fill(in_slot, src, lane, (int)min((uint32_t)TILE, p.n_samples) >> 3);
    }
    cp_async_commit();
  } else if (is_iir && active) {
    y1 = u2f(blob[T::NREG * 32]);
  }

  for (uint32_t kk = 0; kk < n_tiles + 2; ++kk) {
    if (is_worker && active) {
      char *slot = ring + (kk & 1) * 4096;
      if (kk >= 2) {
        // C(kk-2): the recurrence warp left y[0..1023] where u was; (int16_t)y of the lane's row
        const uint32_t t = kk - 2;
        const int r = (int)min((uint32_t)TILE, p.n_samples - t * TILE) >> 5;
        uint32_t dW[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const u32x4 v = lds_u4(slot + T::u_off(lane, j));
          if (no_patch) {
            dW[2 * j] = __byte_perm((uint32_t)f2i_rz(u2f(v.x)), (uint32_t)f2i_rz(u2f(v.y)), 0x5410);
            dW[2 * j + 1] = __byte_perm((uint32_t)f2i_rz(u2f(v.z)), (uint32_t)f2i_rz(u2f(v.w)), 0x5410);
          } else {
            dW[2 * j] = f2i16x2_wrap(u2f(v.x), u2f(v.y));
            dW[2 * j + 1] = f2i16x2_wrap(u2f(v.z), u2f(v.w));
          }
        }
        const int pcm = T::part_c(dW, pv, lane, r, big_b);
        if (lane < r) out[(uint64_t)t * 32 + lane] = (int16_t)pcm;
        __syncwarp();  // every lane has read y before A overwrites the slot
      }
      if (kk < n_tiles) {
        cp_async_wait<0>();
        __syncwarp();
        uint32_t w[16];
        tile_read(in_slot, lane, w);
        __syncwarp();
        if (kk + 1 < n_tiles) {  // the single input slot is free again: fetch the next tile now
          const uint32_t s1 = (kk + 1) * TILE;
          tile_fill(in_slot, src + (uint64_t)s1 * 2, lane, (int)min((uint32_t)TILE, p.n_samples - s1) >> 3);
        }
        cp_async_commit();
        const int r = (int)min((uint32_t)TILE, p.n_samples - kk * TILE) >> 5;
        T::part_a(w, p.fmt, k, p.lut, pv, v_boundary, slot, lane, r);
      }
    } else if (is_iir && active && kk >= 1 && kk <= n_tiles) {
      // B(kk-1): y[n] = fl(u[n] - fl(a1 * y[n-1])) in place, lane == channel (IirFilter.cc:161-176)
      const uint32_t t = kk - 1;
      const int r = (int)min((uint32_t)TILE, p.n_samples - t * TILE) >> 5;
      char *slot = ring + (t & 1) * 4096;
      for (int row = 0; row < r; ++row) {
        u32x4 v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = lds_u4(slot + T::u_off(row, j));
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float y0 = fsub(u2f(v[j].x), fmul(a1, y1));
          const float y2 = fsub(u2f(v[j].y), fmul(a1, y0));
          const float y3 = fsub(u2f(v[j].z), fmul(a1, y2));
          y1 = fsub(u2f(v[j].w), fmul(a1, y3));
          sts_u4(slot + T::u_off(row, j), u32x4{f2u(y0), f2u(y2), f2u(y3), f2u(y1)});
        }
      }
    }
    __syncthreads();
  }

  if (active) {
    if (is_worker) {
      T::store_carry(pv, blob, lane);
      if (lane == 0) {
        blob[T::NREG * 32 + 1] = f2u(v_boundary);
        blob[T::NREG * 32 + 2] = big_b;
      }
    } else {
      blob[T::NREG * 32] = f2u(y1);
    }
  }
}

// ---------------------------------------------------------------------------
// IQ dump (IqDataProcessor.cc:756-760 -> UdpClient::sendData): the block as the demodulators
// and the dump's link partner see it -- signed, Fs/4-rotated, interleaved I,Q -- for the
// channels on `list`. One thread converts one 16-byte piece (two rotation periods); the
// reference sends it on in datagrams of at most 2048 bytes, which are consecutive slices.
// ---------------------------------------------------------------------------
struct DumpParams {
  const uint8_t *iq;
  uint64_t ch_stride;
  uint64_t bytes;        // per channel, a multiple of 64
  int fmt;
  const uint32_t *list;  // dumped channel ids
  uint32_t n_list;
  int8_t *out;           // [n_list][out_stride]
  uint64_t out_stride;
};

__global__ void __launch_bounds__(256) iq_dump_kernel(const __grid_constant__ DumpParams p) {
  const uint64_t pieces = p.bytes / 16;
  const uint32_t li = blockIdx.y;
  const uint8_t *src = p.iq + (uint64_t)p.list[li] * p.ch_stride;
  int8_t *dst = p.out + (uint64_t)li * p.out_stride;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < pieces;
       i += (uint64_t)gridDim.x * blockDim.x) {
    uint4 v = __ldg(reinterpret_cast<const uint4 *>(src) + i);
    if (p.fmt == FMT_U8_OFFSET_ROTATE) {
      // z0 kept, z1 -> (-Q1, I1); z2 -> (-I2, -Q2), z3 -> (Q3, -I3)   (IqDataProcessor.cc:567-611)
      v.x = offset_and_negate(byte_perm(v.x, 0u, 0x2310), 0x00ff0000u, 0x00010000u);
      v.y = offset_and_negate(byte_perm(v.y, 0u, 0x2310), 0xff00ffffu, 0x01000101u);
      v.z = offset_and_negate(byte_perm(v.z, 0u, 0x2310), 0x00ff0000u, 0x00010000u);
      v.w = offset_and_negate(byte_perm(v.w, 0u, 0x2310), 0xff00ffffu, 0x01000101u);
    }
    reinterpret_cast<uint4 *>(dst)[i] = v;
  }
}


// ---------------------------------------------------------------------------
// Squelch (IqDataProcessor.cc:764-765 -> Squelch.cc:227-273): mean of the max + min/2
// magnitude estimate over the block (SignalDetector.cc:205-273), dBFS through the 7-bit
// table (DbfsCalculator.cc:111-147), threshold, two-state tracker with a one-block tail
// (SignalTracker.cc:104-145). One CTA per channel; runs before the demodulation kernels
// when a threshold that can close is set or signal reports are wanted. The call's bytes are
// judged as blocks of block_bytes (the last one may be shorter), each as its own acceptIqData
// call would be; the tracker steps from one block to the next.
// ---------------------------------------------------------------------------
struct SquelchParams {
  const uint8_t *iq;
  uint64_t ch_stride;
  uint64_t n_bytes;
  uint64_t block_bytes;       // bytes per judged block (n_bytes: one decision for the call)
  uint32_t n_channels;        // row length of allowed / magnitude
  int fmt;
  const int32_t *threshold;   // [n_channels] dBFS
  const uint32_t *gain_db;    // [n_channels] tuner gain (radio_adjustableReceiveGainInDb)
  uint8_t *tracking;          // [n_channels] SignalTracker state, carried across blocks and calls
  uint8_t *allowed;           // [n_blocks][n_channels] out: gate of each block
  uint32_t *magnitude;        // [n_blocks][n_channels] out: mean magnitude of each block
  const int32_t *db_table;    // [128] (int32_t)(20 log10f(i)), built by the host libm
};

__global__ void __launch_bounds__(128) squelch_kernel(const SquelchParams q) {
  const uint32_t ch = blockIdx.x;
  const uint8_t *src = q.iq + (uint64_t)ch * q.ch_stride;
  const uint32_t flip = q.fmt == FMT_U8_OFFSET_ROTATE ? 0x80808080u : 0u;  // the rotation does not change |.|
  __shared__ unsigned long long s_part[4];
  uint32_t k = 0;
  for (uint64_t off = 0; off < q.n_bytes; off += q.block_bytes, ++k) {
    const uint64_t len = q.n_bytes - off < q.block_bytes ? q.n_bytes - off : q.block_bytes;
    unsigned long long sum = 0;
    for (uint64_t c = threadIdx.x; c < len / 16; c += blockDim.x) {
      const u32x4 v = ld_stream_u4(src + off + 16 * c);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
      uint32_t part = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t a = __vabs4(w[i] ^ flip);          // |i|, |q| as uint8; |-128| = 128
        const uint32_t b = __byte_perm(a, 0, 0x2301);     // partner of each byte
        const uint32_t mx = __vmaxu4(a, b), mn = __vminu4(a, b);
        const uint32_t m = (mx & 0x00ff00ffu) + ((mn >> 1) & 0x007f007fu);  // two magnitudes <= 192
        part += (m & 0xffffu) + (m >> 16);
      }
      sum += part;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(FULL, sum, o);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned long long total = s_part[0] + s_part[1] + s_part[2] + s_part[3];
      const uint32_t n = (uint32_t)(len / 2);
      const uint32_t mag = (uint32_t)(total / n);
      const uint32_t idx = mag > 127u ? 127u : mag;
      int32_t db = q.db_table[idx] - 42;
      db -= (int32_t)q.gain_db[ch];
      const bool present = db >= q.threshold[ch];
      const bool tracking = q.tracking[ch] != 0;
      const size_t at = (size_t)k * q.n_channels + ch;
      q.allowed[at] = (present || tracking) ? 1 : 0;  // START / PRESENT / END-of-signal tail
      q.tracking[ch] = present ? 1 : 0;
      q.magnitude[at] = mag;
    }
    __syncthreads();  // s_part is written again by the next block
  }
}

// ---------------------------------------------------------------------------
// PCM compaction after a call demodulated in block passes: block k's samples were written at
// column k * block_samples; the open blocks' samples move to the front of the row, in block
// order. One CTA per channel. A block moves only when an earlier block was closed, so its
// destination ends at or before its source starts; the blocks move one after the other, so a
// later block's destination (which may lie in an earlier block's source) is written only once
// that source has been read.
// ---------------------------------------------------------------------------
struct CompactParams {
  int16_t *pcm;               // [n_channels][pcm_stride]
  uint64_t pcm_stride;        // int16 elements between channels (a multiple of 8)
  const uint8_t *allowed;     // [n_blocks][n_channels] gates of the call
  uint32_t n_channels;
  uint32_t n_blocks;
  uint32_t block_samples;     // PCM samples of a full block (a multiple of 32)
  uint32_t last_samples;      // PCM samples of the last block (any count)
};

__global__ void __launch_bounds__(256) pcm_compact_kernel(const CompactParams p) {
  const uint32_t ch = blockIdx.x;
  int16_t *row = p.pcm + (uint64_t)ch * p.pcm_stride;
  uint4 *row8 = reinterpret_cast<uint4 *>(row);  // 8 samples per uint4
  uint32_t dst = 0;  // a multiple of 32: every block before the last is block_samples long
  for (uint32_t k = 0; k < p.n_blocks; ++k) {
    if (!p.allowed[(size_t)k * p.n_channels + ch]) continue;
    const uint32_t len = k + 1 == p.n_blocks ? p.last_samples : p.block_samples;
    const uint32_t src = k * p.block_samples;
    if (dst != src) {  // uniform over the CTA
      for (uint32_t i = threadIdx.x; i < len / 8; i += blockDim.x) row8[dst / 8 + i] = row8[src / 8 + i];
      for (uint32_t i = len / 8 * 8 + threadIdx.x; i < len; i += blockDim.x) row[dst + i] = row[src + i];
      __syncthreads();
    }
    dst += len;
  }
}

}  // namespace sdr
#endif  // SDR_DEVICE_BUILD
