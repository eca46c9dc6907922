// Shared device/host helpers for libduckdb_mb_gpu (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "duckdb_mb_gpu.h"

namespace dmb {

constexpr int kThreads = 256;          // CTA size of every streaming kernel
constexpr int kVec = DMB_VECTOR_SIZE;  // 2048 rows per DuckDB vector / output tile
constexpr int kNumSMs = 148;           // B200

void set_error(const char *fmt, ...);
int32_t check_cuda(cudaError_t e, const char *what);

// ---- 16-byte payload types -------------------------------------------------------------
struct alignas(16) i128 {
  uint64_t lo;
  int64_t hi;
};
struct alignas(16) u128 {
  uint64_t lo;
  uint64_t hi;
};
struct alignas(16) interval_t {  // duckdb_interval
  int32_t months;
  int32_t days;
  int64_t micros;
};
struct alignas(16) month_day_nano_t {  // Arrow month_day_nano_interval
  int32_t months;
  int32_t days;
  int64_t nanos;
};

// R consecutive values moved as one naturally aligned vector (1..16 bytes)
template <typename T, int R>
struct alignas(sizeof(T) * R) Pack {
  T v[R];
};

// ---- streaming (evict-first) vector loads / stores: every byte is touched exactly once ----
template <int N>
struct RawVec;
template <>
struct RawVec<1> { using type = unsigned char; };
template <>
struct RawVec<2> { using type = unsigned short; };
template <>
struct RawVec<4> { using type = unsigned int; };
template <>
struct RawVec<8> { using type = uint2; };
template <>
struct RawVec<16> { using type = uint4; };

template <typename P>
__device__ __forceinline__ P ld_stream(const P *p) {
  using R = typename RawVec<sizeof(P)>::type;
  R r = __ldcs(reinterpret_cast<const R *>(p));
  P out;
  memcpy(&out, &r, sizeof(P));
  return out;
}
template <typename P>
__device__ __forceinline__ void st_stream(P *p, const P &v) {
  using R = typename RawVec<sizeof(P)>::type;
  R r;
  memcpy(&r, &v, sizeof(P));
  __stcs(reinterpret_cast<R *>(p), r);
}

// ---- chunk geometry ------------------------------------------------------------------------
struct BatchView {
  const uint32_t *counts;  // [nchunks]
  const int64_t *row_off;  // [nchunks+1]
  int64_t nchunks;
  int64_t nrows;
};

// largest c in [0, nchunks) with row_off[c] <= row; for row < nrows that chunk is non-empty
__device__ __forceinline__ int64_t find_chunk(const BatchView &b, int64_t row) {
  int64_t lo = 0, hi = b.nchunks;
  while (hi - lo > 1) {
    int64_t mid = (lo + hi) >> 1;
    if (__ldg(b.row_off + mid) <= row) lo = mid; else hi = mid;
  }
  return lo;
}

// `take` (1..64) validity bits of chunk rows [local, local+take); bit i = row local+i valid
__device__ __forceinline__ uint64_t chunk_valid_bits(const uint64_t *vslab, const dmb_vec_desc *vecs,
                                                     int64_t c, int local, int take) {
  uint64_t keep = take >= 64 ? ~0ull : ((1ull << take) - 1ull);
  int64_t vo = vecs[c].val_off;
  if (vo < 0) return keep;  // NULL validity pointer = all valid (reference: duckdb_native.c:531-533)
  const uint64_t *m = vslab + vo;
  int w = local >> 6, s = local & 63;
  uint64_t bits = __ldg(m + w) >> s;
  if (s && s + take > 64) bits |= __ldg(m + w + 1) << (64 - s);
  return bits & keep;
}

// 64 validity bits of output rows [r0, r0+64) gathered across chunk boundaries (rows >= nrows: 0)
__device__ __forceinline__ uint64_t gather_valid64(const BatchView &b, const uint64_t *vslab,
                                                   const dmb_vec_desc *vecs, int64_t r0) {
  if (r0 >= b.nrows) return 0ull;
  int64_t c = find_chunk(b, r0);
  uint64_t word = 0;
  int filled = 0;
  while (filled < 64 && r0 + filled < b.nrows) {
    int64_t local = r0 + filled - __ldg(b.row_off + c);
    int64_t avail = (int64_t)__ldg(b.counts + c) - local;
    if (avail <= 0) { ++c; continue; }
    int take = (int)(avail < (int64_t)(64 - filled) ? avail : (int64_t)(64 - filled));
    word |= chunk_valid_bits(vslab, vecs, c, (int)local, take) << filled;
    filled += take;
  }
  return word;
}

// tile t (output rows [t*2048, t*2048+2048)) is exactly chunk t, rows [0, count)
__device__ __forceinline__ bool tile_is_regular(const BatchView &b, int64_t t) {
  if (t >= b.nchunks) return false;
  int64_t ro = __ldg(b.row_off + t);
  if (ro != t * (int64_t)kVec) return false;
  uint32_t cnt = __ldg(b.counts + t);
  return cnt == (uint32_t)kVec || ro + cnt == b.nrows;
}

// 8 bytes that are each 0/1 -> 8 bits (byte k -> bit k)
__device__ __forceinline__ uint32_t pack8(uint64_t bytes01) {
  return (uint32_t)((bytes01 * 0x0102040810204080ull) >> 56);
}
// 8 bits -> 8 bytes that are each 0/1
__device__ __forceinline__ uint64_t spread8(uint32_t bits) {
  uint64_t x = (uint64_t)(bits & 0xff) * 0x0101010101010101ull;  // byte m = bits
  x &= 0x8040201008040201ull;                                      // byte m keeps bit m
  x += 0x7f7f7f7f7f7f7f7full;                                      // bit 7 of byte m = (bit m != 0)
  return (x >> 7) & 0x0101010101010101ull;
}

// ---- bitmaps as aligned 32-bit words, misaligned 16-byte vectors (reverse kernels, LIST child copy) -----------------
// An LSB bitmap read as aligned 32-bit words: `w` is the bitmap address rounded down to 4 bytes and
// `base` the bit position of row 0 counted from there (Arrow array offset + the rounded-off bytes).
struct BitSrc {
  const uint32_t *w;
  int64_t base;
};
__device__ __forceinline__ BitSrc bit_src(const uint8_t *bm, int64_t bit_offset) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(bm);
  return BitSrc{reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3), bit_offset + (int64_t)(a & 3u) * 8};
}

// `take` (1..32) bits from bit position p; only the words that hold a requested bit are touched
__device__ __forceinline__ uint32_t load_bits32(const uint32_t *w, int64_t p, int take) {
  const int64_t wi = p >> 5;
  const int s = (int)(p & 31);
  const uint32_t lo = __ldg(w + wi);
  const uint32_t hi = (s + take > 32) ? __ldg(w + wi + 1) : 0u;
  const uint32_t r = __funnelshift_r(lo, hi, (uint32_t)s);
  return take >= 32 ? r : (r & ((1u << take) - 1u));
}

// words [ws, ws+4] of the 8 words (a, b), shifted right by sh bits: the 16 bytes that start m = 4*ws + sh/8
// bytes into a
__device__ __forceinline__ uint4 shift_words(const uint4 &a, const uint4 &b, int ws, uint32_t sh) {
  uint32_t w0, w1, w2, w3, w4;
  switch (ws) {
    case 0: w0 = a.x; w1 = a.y; w2 = a.z; w3 = a.w; w4 = b.x; break;
    case 1: w0 = a.y; w1 = a.z; w2 = a.w; w3 = b.x; w4 = b.y; break;
    case 2: w0 = a.z; w1 = a.w; w2 = b.x; w3 = b.y; w4 = b.z; break;
    default: w0 = a.w; w1 = b.x; w2 = b.y; w3 = b.z; w4 = b.w; break;
  }
  return make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
}

// keep-mask of 32-bit word i of a 16-byte vector of 16/W elements, bit r of `bits` = element r valid
template <int W>
__device__ __forceinline__ uint32_t word_keep(uint32_t bits, int i) {
  if (W >= 4) return ((bits >> (i * 4 / W)) & 1u) ? 0xffffffffu : 0u;
  if (W == 2) {
    const uint32_t b = bits >> (2 * i);
    return ((b & 1u) ? 0x0000ffffu : 0u) | ((b & 2u) ? 0xffff0000u : 0u);
  }
  const uint32_t b = bits >> (4 * i);
  return ((b & 1u) | ((b & 2u) << 7) | ((b & 4u) << 14) | ((b & 8u) << 21)) * 0xffu;
}

// the string_t of dictionary entry idx (<= 12 bytes inlined, else prefix + pointer relative to dict_host_base)
__device__ __forceinline__ uint4 enum_entry(const dmb_enum_job &job, uint32_t idx) {
  const uint32_t o0 = __ldg(job.dict_offsets + idx), o1 = __ldg(job.dict_offsets + idx + 1);
  const uint32_t len = o1 - o0;
  const uint8_t *q = job.dict_data + o0;
  uint4 e = make_uint4(len, 0, 0, 0);
  if (len <= 12u) {
    uint32_t w[3] = {0u, 0u, 0u};
#pragma unroll
    for (uint32_t k = 0; k < 12u; ++k)  // (unrolled: the byte loads are in flight together, one round trip instead of `len`)
      if (k < len) w[k >> 2] |= (uint32_t)__ldg(q + k) << (8u * (k & 3u));
    e.y = w[0]; e.z = w[1]; e.w = w[2];
  } else {
    e.y = (uint32_t)__ldg(q) | ((uint32_t)__ldg(q + 1) << 8) | ((uint32_t)__ldg(q + 2) << 16) | ((uint32_t)__ldg(q + 3) << 24);
    const uint64_t p = job.dict_host_base + o0;
    e.z = (uint32_t)p;
    e.w = (uint32_t)(p >> 32);
  }
  return e;
}


// ---- decoupled look-back: status words (flag in bits 63..62, value below: one word, so no fences are needed) ----
constexpr uint64_t kFlagAggregate = 1ull << 62;
constexpr uint64_t kFlagPrefix = 2ull << 62;
constexpr uint64_t kValueMask = (1ull << 62) - 1ull;
__device__ __forceinline__ uint64_t ld_status(const unsigned long long *p) {
  return *reinterpret_cast<const volatile unsigned long long *>(p);
}
__device__ __forceinline__ unsigned long long global_ns() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }

// Two-level decoupled look-back (string_pack_kernel, enum_pack_kernel, list_emit_kernel).  With ~450 persistent CTAs that claim tiles two iterations ahead, the nearest
// predecessor whose PREFIX is out is typically 150-300 tiles back; a tile-by-tile look-back of 256 words per round then sits
// on the edge between one L2 round trip and two, and the launch is bistable (late prefixes make every look-back longer,
// which makes the prefixes later: 0.82 vs 1.15-1.47 ms per 60 M rows on all-pointer columns).  So tiles also add their
// aggregate to a word per GROUP of 32 tiles (count in bits 56..61, sum below), and the last tile of a group publishes the
// group's inclusive prefix: a look-back reads the <= 63 nearest tiles one by one and everything before them as groups,
// 32 groups (1024 tiles) per round, all loads in flight together.
constexpr unsigned long long kGroupOne = 1ull << 56;
constexpr unsigned long long kGroupSumMask = kGroupOne - 1ull;
__device__ __forceinline__ uint64_t lookback_groups(const unsigned long long *status, const unsigned long long *gsum, const unsigned long long *gpre,
                                                    int64_t tile, int lane, unsigned long long *err_flags, unsigned long long err_bit,
                                                    unsigned long long limit_ns) {
  if (tile <= 0) return 0;
  const int64_t g = tile >> 5;
  const int64_t lo = g >= 1 ? 32 * (g - 1) : 0;  // tiles [lo, tile) are read one by one
  const int64_t idx0 = tile - 1 - lane, idx1 = tile - 33 - lane;
  const bool in0 = idx0 >= lo, in1 = idx1 >= lo;
  int64_t hbase = g - 2;                         // groups hbase, hbase - 1, ... : one per lane
  uint64_t st0 = 0, st1 = 0, ga = 0, gb = 0;
  uint64_t prefix = 0;
  unsigned long long t0 = 0;
  // a needed word is not out yet: poll again at once (an eager look-back -- enum_pack_kernel, list_emit_kernel -- starts
  // when its neighbours are about to publish), back off after a few tries, look at the clock every 64th.  Warp-uniform:
  // true when the wait limit has passed (flagged; the host discards the outputs).
  unsigned spins = 0;
  auto give_up = [&]() -> bool {
    ++spins;
    if (spins > 8u) __nanosleep(100);
    if ((spins & 63u) != 0u && limit_ns != 0ull) return false;  // (a zero limit -- the tests' way to see the error path -- gives up at the first wait)
    const unsigned long long now = global_ns();
    if (t0 == 0) t0 = now;
    if (__any_sync(0xffffffffu, now - t0 > limit_ns)) {
      if (lane == 0) atomicOr(err_flags, err_bit);
      return true;
    }
    return false;
  };
  {
    const int64_t h = hbase - lane;
    if (h >= 0) { ga = ld_status(gpre + h); gb = ld_status(gsum + h); }
  }
  // ---- the nearest tiles
  {
    uint64_t v;
    int state;  // 0: no prefix among them  1: a prefix closed the sum  2: a needed word is not published yet
    while (true) {
      if (in0 && (st0 >> 62) == 0) st0 = ld_status(status + idx0);
      if (in1 && (st1 >> 62) == 0) st1 = ld_status(status + idx1);
      v = 0;
      state = 0;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const uint64_t st = j ? st1 : st0;
        const bool in = j ? in1 : in0;
        if (state == 0) {
          const uint32_t ready = __ballot_sync(0xffffffffu, !in || (st >> 62) != 0);
          const uint32_t is_p = __ballot_sync(0xffffffffu, in && (st >> 62) == 2);
          const int first_p = is_p ? (__ffs(is_p) - 1) : 31;
          const uint32_t need = first_p >= 31 ? 0xffffffffu : ((2u << first_p) - 1u);
          if ((ready & need) != need) state = 2;
          else {
            if (in && lane <= first_p) v += st & kValueMask;
            if (is_p) state = 1;
          }
        }
      }
      if (state != 2) break;
      if (give_up()) { state = 1; break; }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    prefix = v;
    if (state == 1) return prefix;
  }
  // ---- the groups before them
  while (true) {
    const int64_t h = hbase - lane;
    uint32_t is_p;
    int first_p;
    while (true) {
      const bool pa = h < 0 || (ga >> 62) == 2;                    // the inclusive prefix through group h is out (before group 0: 0)
      const bool cb = h >= 0 && ((gb >> 56) & 63ull) == 32ull;     // all 32 aggregates of group h are in its sum
      is_p = __ballot_sync(0xffffffffu, pa);
      first_p = is_p ? (__ffs(is_p) - 1) : 32;
      const uint32_t need = first_p >= 32 ? 0xffffffffu : ((1u << first_p) - 1u);
      const uint32_t compl_ = __ballot_sync(0xffffffffu, cb);
      if ((compl_ & need) == need) break;
      if (give_up()) return prefix;
      if (h >= 0 && !pa && !cb) { ga = ld_status(gpre + h); gb = ld_status(gsum + h); }
    }
    uint64_t v = lane < first_p ? (gb & kGroupSumMask) : ((lane == first_p && h >= 0) ? (ga & kValueMask) : 0ull);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    prefix += v;
    if (is_p) return prefix;
    hbase -= 32;
    ga = gb = 0;
    const int64_t h2 = hbase - lane;
    if (h2 >= 0) { ga = ld_status(gpre + h2); gb = ld_status(gsum + h2); }
  }
}


}  // namespace dmb
