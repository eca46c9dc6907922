// K6 arrow_to_chunk: Arrow buffers -> DuckDB DataChunk vectors (the bulk door behind the
// appender).  Chunk k of the output is rows [2048k, 2048k+2048): payload slab at k*2048*W bytes,
// validity slab at k*32 uint64 words, so both slabs are dense in row order.
//   * fixed width: copy / narrow with NULL payloads zeroed, 128-bit accesses when the Arrow slice
//     start is 16-byte aligned (an Arrow `offset` only guarantees element alignment)
//   * Arrow validity bitmap at an arbitrary bit offset -> uint64 masks (funnel shift)
//   * Arrow bool bits -> DuckDB bool bytes
//   * decimal128 -> DECIMAL int64/int32/int16 (low bytes)
//   * utf8 -> duckdb_string_t: <= 12 bytes inlined (zero padded), else 4-byte prefix + pointer to
//     the bytes in place in the *host* Arrow data buffer (SURVEY.md §8d); validity via warp ballot
//
// Replaces the reference's row-at-a-time appends src/duckdb_native.c:1116-1235 (one FFI call and
// one duckdb_append_* per cell); the vectors are what duckdb_append_data_chunk (:2109-2132) takes.

#include <type_traits>

#include "dmb_common.cuh"

namespace dmb {

// rows of the warp whose first row is row0 that lie below nrows (0..32)
__device__ __forceinline__ int rev_warp_live(int64_t nrows, int64_t row0) {
  const int64_t left = nrows - row0;
  return left <= 0 ? 0 : (left < 32 ? (int)left : 32);
}

// the validity word of that warp: bit k for row row0 + k, 0 past the live rows; an absent bitmap is all valid
__device__ __forceinline__ uint32_t rev_warp_bits(const BitSrc &bs, bool has_bm, int live, int64_t row0) {
  return live == 0 ? 0u : (has_bm ? load_bits32(bs.w, bs.base + row0, live) : (live == 32 ? 0xffffffffu : ((1u << live) - 1u)));
}

// an Arrow dictionary index, sign- or zero-extended; an unsigned 64-bit index past 2^63 comes out negative, i.e. out of
// range as well
template <typename I>
__device__ __forceinline__ int64_t rev_dict_index(I raw, bool is_signed) {
  constexpr int kShift = 64 - 8 * (int)sizeof(I);
  return is_signed ? (int64_t)((uint64_t)raw << kShift) >> kShift : (int64_t)(uint64_t)raw;
}

// 64 validity bits for output word w (rows 64w..64w+63), rows >= nrows are 0
__device__ __forceinline__ uint64_t rev_valid_word(const BitSrc &bs, bool has_bm, int64_t nrows, int64_t w) {
  const int64_t r0 = w << 6;
  if (r0 >= nrows) return 0ull;
  const int64_t left = nrows - r0;
  const int live = left < 64 ? (int)left : 64;
  if (!has_bm) return live == 64 ? ~0ull : ((1ull << live) - 1ull);
  const int64_t p = bs.base + r0;
  const uint64_t lo = load_bits32(bs.w, p, live < 32 ? live : 32);
  const uint64_t hi = live > 32 ? load_bits32(bs.w, p + 32, live - 32) : 0u;
  return lo | (hi << 32);
}

template <typename S, typename D>
__device__ __forceinline__ D narrow(const S &v) {
  D d;
  memcpy(&d, &v, sizeof(D));  // little endian: low bytes
  return d;
}

// Same-width copy with NULL payloads zeroed.  The Arrow slice start is only element-aligned, so the input is
// read as the aligned 16-byte vectors around it (4 per thread in flight); a lane takes the vector that follows
// its own from its neighbour by shuffle and the byte shift is a funnel shift.
template <int W>
__device__ __forceinline__ void rev_copy(const dmb_rev_fixed_job &job, int64_t nrows) {
  constexpr int R = 16 / W;
  constexpr int U = 4;
  const uint8_t *in = reinterpret_cast<const uint8_t *>(job.in_values);
  uint8_t *out = reinterpret_cast<uint8_t *>(job.out_data);
  const int m = (int)(reinterpret_cast<uintptr_t>(in) & 15u);
  const uint4 *al = reinterpret_cast<const uint4 *>(in - m);
  const int ws = m >> 2;
  const uint32_t sh = (uint32_t)(m & 3) * 8u;
  const bool has_bm = job.in_validity != nullptr;
  const BitSrc bs = bit_src(job.in_validity, job.in_bit_offset);
  const int64_t nvec = nrows / R;
  const int lane = threadIdx.x & 31;
  for (int64_t base = (int64_t)blockIdx.x * (U * kThreads); base < nvec; base += (int64_t)gridDim.x * (U * kThreads)) {
    uint4 a[U], b[U];
    uint32_t bits[U];
    // every load of the iteration is issued before anything waits: the vectors, lane 31's extra vector, the bitmap words
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t v = base + u * kThreads + threadIdx.x;
      a[u] = v < nvec ? ld_stream(al + v) : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t v = base + u * kThreads + threadIdx.x;
      b[u] = make_uint4(0, 0, 0, 0);
      if (m && v < nvec && (lane == 31 || v + 1 >= nvec)) b[u] = ld_stream(al + v + 1);
      bits[u] = (has_bm && v < nvec) ? load_bits32(bs.w, bs.base + v * R, R) : 0xffffffffu;
    }
    if (m) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t v = base + u * kThreads + threadIdx.x;
        const uint32_t nx = __shfl_down_sync(0xffffffffu, a[u].x, 1), ny = __shfl_down_sync(0xffffffffu, a[u].y, 1);
        const uint32_t nz = __shfl_down_sync(0xffffffffu, a[u].z, 1), nw = __shfl_down_sync(0xffffffffu, a[u].w, 1);
        if (!(lane == 31 || v + 1 >= nvec)) b[u] = make_uint4(nx, ny, nz, nw);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t v = base + u * kThreads + threadIdx.x;
      if (v >= nvec) continue;
      uint4 o = m ? shift_words(a[u], b[u], ws, sh) : a[u];
      o.x &= word_keep<W>(bits[u], 0);
      o.y &= word_keep<W>(bits[u], 1);
      o.z &= word_keep<W>(bits[u], 2);
      o.w &= word_keep<W>(bits[u], 3);
      st_stream(reinterpret_cast<uint4 *>(out) + v, o);
    }
  }
  // the last nrows % R rows
  if (blockIdx.x == 0) {
    for (int64_t row = nvec * R + threadIdx.x; row < nrows; row += kThreads) {
      const bool valid = has_bm ? (load_bits32(bs.w, bs.base + row, 1) != 0u) : true;
      for (int k = 0; k < W; ++k) out[row * W + k] = valid ? in[row * W + k] : (uint8_t)0;
    }
  }
}

// decimal128 -> narrower DECIMAL: low bytes, NULL payloads zeroed
template <typename D>
__device__ __forceinline__ void rev_narrow(const dmb_rev_fixed_job &job, int64_t nrows) {
  const uint64_t *in = reinterpret_cast<const uint64_t *>(job.in_values);  // Arrow buffers are 8-byte aligned
  D *out = reinterpret_cast<D *>(job.out_data);
  const bool has_bm = job.in_validity != nullptr;
  const BitSrc bs = bit_src(job.in_validity, job.in_bit_offset);
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  for (int64_t row = (int64_t)blockIdx.x * kThreads + threadIdx.x; row < nrows; row += stride) {
    const uint64_t lo = __ldcs(in + 2 * row);
    const bool valid = has_bm ? (load_bits32(bs.w, bs.base + row, 1) != 0u) : true;
    out[row] = valid ? narrow<uint64_t, D>(lo) : D{};
  }
}

// Arrow bool bits -> bool bytes: a thread handles 16 rows -> one 16-byte store
__device__ __forceinline__ void rev_bits_to_bool(const dmb_rev_fixed_job &job, int64_t nrows) {
  uint8_t *out = reinterpret_cast<uint8_t *>(job.out_data);
  const bool has_bm = job.in_validity != nullptr;
  const BitSrc vs = bit_src(reinterpret_cast<const uint8_t *>(job.in_values), job.in_bit_offset);
  const BitSrc bs = bit_src(job.in_validity, job.in_bit_offset);
  const int64_t ngroups = (nrows + 15) >> 4;
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  for (int64_t g = (int64_t)blockIdx.x * kThreads + threadIdx.x; g < ngroups; g += stride) {
    const int64_t r0 = g << 4;
    const int live = nrows - r0 < 16 ? (int)(nrows - r0) : 16;
    uint32_t bits = load_bits32(vs.w, vs.base + r0, live);
    if (has_bm) bits &= load_bits32(bs.w, bs.base + r0, live);
    const uint64_t lo = spread8(bits), hi = spread8(bits >> 8);
    if (live == 16) {
      st_stream(reinterpret_cast<uint4 *>(out + r0), make_uint4((uint32_t)lo, (uint32_t)(lo >> 32), (uint32_t)hi, (uint32_t)(hi >> 32)));
    } else {
      for (int k = 0; k < live; ++k) out[r0 + k] = (uint8_t)((k < 8 ? lo >> (8 * k) : hi >> (8 * (k - 8))) & 0xff);
    }
  }
}

__global__ void __launch_bounds__(kThreads, 4)
rev_fixed_kernel(const dmb_rev_fixed_job *__restrict__ jobs, int64_t nrows) {
  __shared__ dmb_rev_fixed_job s_job;
  if (threadIdx.x < sizeof(dmb_rev_fixed_job) / 8)
    reinterpret_cast<uint64_t *>(&s_job)[threadIdx.x] = reinterpret_cast<const uint64_t *>(jobs + blockIdx.y)[threadIdx.x];
  __syncthreads();
  const dmb_rev_fixed_job &job = s_job;
  if (job.out_data) {
    switch (job.op) {
      case DMB_REV_COPY1: rev_copy<1>(job, nrows); break;
      case DMB_REV_COPY2: rev_copy<2>(job, nrows); break;
      case DMB_REV_COPY4: rev_copy<4>(job, nrows); break;
      case DMB_REV_COPY8: rev_copy<8>(job, nrows); break;
      case DMB_REV_COPY16: rev_copy<16>(job, nrows); break;
      case DMB_REV_BITS_TO_BOOL: rev_bits_to_bool(job, nrows); break;
      case DMB_REV_I128_TO_I64: rev_narrow<uint64_t>(job, nrows); break;
      case DMB_REV_I128_TO_I32: rev_narrow<uint32_t>(job, nrows); break;
      case DMB_REV_I128_TO_I16: rev_narrow<uint16_t>(job, nrows); break;
      default: break;
    }
  }
  // validity masks for every vector slot (capacity rows: bits past nrows are 0)
  if (job.out_validity) {
    const int64_t nwords = ((nrows + kVec - 1) / kVec) * DMB_VALIDITY_WORDS;
    const int64_t stride = (int64_t)gridDim.x * kThreads;
    const bool has_bm = job.in_validity != nullptr;
    const BitSrc bs = bit_src(job.in_validity, job.in_bit_offset);
    int nulls = 0;
    for (int64_t w = (int64_t)blockIdx.x * kThreads + threadIdx.x; w < nwords; w += stride) {
      uint64_t word = rev_valid_word(bs, has_bm, nrows, w);
      __stcs(reinterpret_cast<unsigned long long *>(job.out_validity + w), word);
      int64_t left = nrows - (w << 6);
      int live = left <= 0 ? 0 : (left < 64 ? (int)left : 64);
      nulls += live - __popcll(word);
    }
    if (job.null_count) {
      nulls = __reduce_add_sync(0xffffffffu, nulls);
      if ((threadIdx.x & 31) == 0 && nulls) atomicAdd(job.null_count, (unsigned long long)nulls);
    }
  }
}

// utf8 -> duckdb_string_t, two rows per thread in flight.  A warp's 32 rows share one validity word (which is also
// the word the mask slab takes) and read 33 offsets: one per lane plus one for lane 31.
template <bool LARGE>
__global__ void __launch_bounds__(kThreads)
rev_string_kernel(dmb_rev_string_job job, int64_t nrows) {
  constexpr int U = 2;
  using off_t = typename std::conditional<LARGE, long long, int>::type;
  const off_t *off = reinterpret_cast<const off_t *>(job.in_offsets);
  const int lane = threadIdx.x & 31;
  const int64_t capacity = ((nrows + kVec - 1) / kVec) * (int64_t)kVec;  // a multiple of U * kThreads
  const bool has_bm = job.in_validity != nullptr;
  const bool has_data = job.in_data != nullptr;
  const BitSrc bs = bit_src(job.in_validity, job.in_bit_offset);
  uint4 *out = reinterpret_cast<uint4 *>(job.out);
  uint32_t *out_val32 = reinterpret_cast<uint32_t *>(job.out_validity);
  int nulls = 0;
  for (int64_t base = (int64_t)blockIdx.x * (U * kThreads); base < capacity; base += (int64_t)gridDim.x * (U * kThreads)) {
    off_t o0[U], o1[U];
    uint32_t vb[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row = base + u * kThreads + threadIdx.x;
      o0[u] = __ldg(off + (row < nrows ? row : nrows));
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row = base + u * kThreads + threadIdx.x;
      const int64_t row0 = row - lane;
      const int64_t left = nrows - row0;
      const int live = left <= 0 ? 0 : (left < 32 ? (int)left : 32);
      vb[u] = live == 0 ? 0u : (has_bm ? load_bits32(bs.w, bs.base + row0, live) : (live == 32 ? 0xffffffffu : ((1u << live) - 1u)));
      if (lane == 0) {
        if (out_val32) out_val32[row >> 5] = vb[u];
        nulls += live - __popc(vb[u]);
      }
      o1[u] = __shfl_down_sync(0xffffffffu, o0[u], 1);
      if (lane == 31) o1[u] = __ldg(off + (row + 1 < nrows ? row + 1 : nrows));
    }
    uint32_t w[U][4], sh[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      // first 12 bytes of the string with 4 aligned 32-bit loads + funnel shifts
      const uint8_t *q = job.in_data + o0[u];
      const uint32_t *b32 = reinterpret_cast<const uint32_t *>(reinterpret_cast<uintptr_t>(q) & ~(uintptr_t)3);
      sh[u] = (uint32_t)(reinterpret_cast<uintptr_t>(q) & 3u) * 8u;
      // all four words, unpredicated: the bytes past the string are the next rows' (or the buffer's 16 bytes of
      // padding, see the header) and are masked off below
      if (has_data) {
        w[u][0] = __ldg(b32);
        w[u][1] = __ldg(b32 + 1);
        w[u][2] = __ldg(b32 + 2);
        w[u][3] = __ldg(b32 + 3);
      } else {
        w[u][0] = w[u][1] = w[u][2] = w[u][3] = 0u;
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row = base + u * kThreads + threadIdx.x;
      const bool valid = (vb[u] >> lane) & 1u;
      uint4 e = make_uint4(0, 0, 0, 0);
      if (valid) {
        const uint32_t len = (uint32_t)(o1[u] - o0[u]);
        const uint32_t r0 = __funnelshift_r(w[u][0], w[u][1], sh[u]), r1 = __funnelshift_r(w[u][1], w[u][2], sh[u]),
                       r2 = __funnelshift_r(w[u][2], w[u][3], sh[u]);
        e.x = len;
        if (len <= 12u) {
          auto keep = [](uint32_t word, int nb) { return nb >= 4 ? word : (nb <= 0 ? 0u : (word & ((1u << (8 * nb)) - 1u))); };
          e.y = keep(r0, (int)len);
          e.z = keep(r1, (int)len - 4);
          e.w = keep(r2, (int)len - 8);
        } else {
          e.y = r0;  // prefix
          const uint64_t p = job.data_host_base + (uint64_t)o0[u];
          e.z = (uint32_t)p;
          e.w = (uint32_t)(p >> 32);
        }
      }
      st_stream(out + row, e);
    }
  }
  if (job.null_count && lane == 0 && nulls) atomicAdd(job.null_count, (unsigned long long)nulls);
}

// Arrow list offsets -> duckdb_list_entry + list masks (rows, two per thread in flight, offsets read like
// rev_string_kernel), then every chunk's child mask (one 64-bit word per thread, funnel shifted from the dense child
// bitmap so that chunk k's mask starts at its first element).
template <bool LARGE>
__global__ void __launch_bounds__(kThreads)
rev_list_kernel(dmb_rev_list_job job, int64_t nrows) {
  constexpr int U = 2;
  using off_t = typename std::conditional<LARGE, long long, int>::type;
  const off_t *off = reinterpret_cast<const off_t *>(job.in_offsets);
  const int lane = threadIdx.x & 31;
  const int64_t nchunks = (nrows + kVec - 1) / kVec;
  const int64_t capacity = nchunks * (int64_t)kVec;  // a multiple of U * kThreads
  const bool has_bm = job.in_validity != nullptr;
  const BitSrc bs = bit_src(job.in_validity, job.in_bit_offset);
  uint4 *out = reinterpret_cast<uint4 *>(job.out_entries);
  uint32_t *out_val32 = reinterpret_cast<uint32_t *>(job.out_validity);
  const int64_t off0 = (int64_t)__ldg(off);
  int nulls = 0;
  bool bad = false;
  for (int64_t base = (int64_t)blockIdx.x * (U * kThreads); base < capacity; base += (int64_t)gridDim.x * (U * kThreads)) {
    off_t o0[U], o1[U];
    int64_t cbase[U];
    uint32_t vb[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row = base + u * kThreads + threadIdx.x;
      o0[u] = __ldg(off + (row < nrows ? row : nrows));
      cbase[u] = (int64_t)__ldg(off + (row & ~(int64_t)(kVec - 1)));  // same address for the whole warp
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row = base + u * kThreads + threadIdx.x;
      const int64_t row0 = row - lane;
      const int64_t left = nrows - row0;
      const int live = left <= 0 ? 0 : (left < 32 ? (int)left : 32);
      vb[u] = live == 0 ? 0u : (has_bm ? load_bits32(bs.w, bs.base + row0, live) : (live == 32 ? 0xffffffffu : ((1u << live) - 1u)));
      if (lane == 0) {
        out_val32[row >> 5] = vb[u];
        nulls += live - __popc(vb[u]);
      }
      o1[u] = __shfl_down_sync(0xffffffffu, o0[u], 1);
      if (lane == 31) o1[u] = __ldg(off + (row + 1 < nrows ? row + 1 : nrows));
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row = base + u * kThreads + threadIdx.x;
      uint4 e = make_uint4(0, 0, 0, 0);
      if (row < nrows) {
        const int64_t len = (int64_t)o1[u] - (int64_t)o0[u];
        bad |= len < 0;
        const uint64_t eo = (uint64_t)((int64_t)o0[u] - cbase[u]);
        const uint64_t el = ((vb[u] >> lane) & 1u) && len > 0 ? (uint64_t)len : 0ull;
        e = make_uint4((uint32_t)eo, (uint32_t)(eo >> 32), (uint32_t)el, (uint32_t)(el >> 32));
      }
      st_stream(out + row, e);
    }
  }
  if (job.null_count && lane == 0 && nulls) atomicAdd(job.null_count, (unsigned long long)nulls);
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(job.error, 1u);
  // child masks: word w belongs to the chunk k with child_word[k] <= w < child_word[k+1]
  const int64_t nwords = __ldg(job.child_word + nchunks);
  const bool has_cbm = job.in_child_validity != nullptr;
  const BitSrc cs = bit_src(job.in_child_validity, job.child_bit_offset);
  for (int64_t w = (int64_t)blockIdx.x * kThreads + threadIdx.x; w < nwords; w += (int64_t)gridDim.x * kThreads) {
    int64_t lo = 0, hi = nchunks;
    while (hi - lo > 1) {
      const int64_t mid = (lo + hi) >> 1;
      if (__ldg(job.child_word + mid) <= w) lo = mid; else hi = mid;
    }
    const int64_t r0 = lo * kVec, r1 = r0 + kVec < nrows ? r0 + kVec : nrows;
    const int64_t e0 = (int64_t)__ldg(off + r0) - off0, size = (int64_t)__ldg(off + r1) - off0 - e0;
    const BitSrc chunk_bits{cs.w, cs.base + e0};
    __stcs(reinterpret_cast<unsigned long long *>(job.out_child_validity + w), rev_valid_word(chunk_bits, has_cbm, size, w - __ldg(job.child_word + lo)));
  }
}

// bits [r0, r0 + 64) of a row bitmap (bit k: row r0 + k), 0 outside rows [0, nrows); r0 > -64.  An absent bitmap is all
// valid.
__device__ __forceinline__ uint64_t rev_mask_bits64(const BitSrc &bs, bool has_bm, int64_t nrows, int64_t r0) {
  const int lead = r0 < 0 ? (int)(-r0) : 0;  // the first word of an output at a bit phase starts before row 0
  const int64_t first = r0 + lead, left = nrows - first;
  if (left <= 0) return 0ull;
  const int live = left < 64 - lead ? (int)left : 64 - lead;
  uint64_t v;
  if (!has_bm) {
    v = live == 64 ? ~0ull : ((1ull << live) - 1ull);
  } else {
    const uint64_t lo = load_bits32(bs.w, bs.base + first, live < 32 ? live : 32);
    const uint64_t hi = live > 32 ? load_bits32(bs.w, bs.base + first + 32, live - 32) : 0u;
    v = lo | (hi << 32);
  }
  return v << lead;
}

// STRUCT validity: out = a AND b over nrows rows, written as whole 64-bit words from bit out_bit_offset on, every bit
// outside [out_bit_offset, out_bit_offset + nrows) zero.  One thread per output word; grid.y = job.
__global__ void __launch_bounds__(kThreads)
rev_mask_kernel(const dmb_rev_mask_job *__restrict__ jobs, int64_t nrows) {
  const dmb_rev_mask_job job = jobs[blockIdx.y];
  const int64_t nwords = ((job.out_bit_offset + nrows + kVec - 1) / kVec) * DMB_VALIDITY_WORDS;
  const BitSrc a = bit_src(job.in_a, job.a_bit_offset), b = bit_src(job.in_b, job.b_bit_offset);
  const bool has_a = job.in_a != nullptr, has_b = job.in_b != nullptr;
  for (int64_t w = (int64_t)blockIdx.x * kThreads + threadIdx.x; w < nwords; w += (int64_t)gridDim.x * kThreads) {
    const int64_t r0 = (w << 6) - job.out_bit_offset;
    __stcs(reinterpret_cast<unsigned long long *>(job.out + w), rev_mask_bits64(a, has_a, nrows, r0) & rev_mask_bits64(b, has_b, nrows, r0));
  }
}

// ---- ENUM: labels -> positions (dmb_rev_enum_job).  One row per thread; a warp's 32 rows share one validity word, which
// is also the mask word the ballot of the rows that got a position writes.
extern __shared__ uint4 rev_enum_smem[];  // the lookup table, the remap or a dictionary's string_t table, when it fits
constexpr int kEnumSmemBytes = 48 << 10;

// row `row` of a final-vector or remap launch: `code` is a position, DMB_ENUM_CODE_NULL or DMB_ENUM_CODE_MISSING (unused
// when the row is NULL).  Called by every lane of the warp.
__device__ __forceinline__ void enum_emit(const dmb_rev_enum_job &job, int64_t row, int64_t nrows, uint32_t vb, uint32_t code, int &nulls,
                                          unsigned long long &first_bad) {
  const int lane = threadIdx.x & 31;
  const bool in = row < nrows, valid = (vb >> lane) & 1u;
  if (job.out_width == 0) {
    if (in) __stcs(reinterpret_cast<unsigned int *>(job.out) + row, valid ? code : DMB_ENUM_CODE_NULL);
    return;
  }
  const bool ok = valid && code < DMB_ENUM_CODE_NULL;
  if (valid && code == DMB_ENUM_CODE_MISSING && (unsigned long long)row < first_bad) first_bad = (unsigned long long)row;
  const uint32_t word = __ballot_sync(0xffffffffu, ok);
  const uint32_t v = ok ? code : 0u;
  switch (job.out_width) {
    case 1: reinterpret_cast<uint8_t *>(job.out)[row] = (uint8_t)v; break;
    case 2: __stcs(reinterpret_cast<unsigned short *>(job.out) + row, (unsigned short)v); break;
    default: __stcs(reinterpret_cast<unsigned int *>(job.out) + row, v); break;
  }
  if (lane == 0) {
    reinterpret_cast<uint32_t *>(job.out_validity)[row >> 5] = word;
    const int64_t left = nrows - row;
    nulls += (left <= 0 ? 0 : (left < 32 ? (int)left : 32)) - __popc(word);
  }
}

__device__ __forceinline__ void enum_finish(const dmb_rev_enum_job &job, int nulls, unsigned long long first_bad) {
  if (first_bad != ~0ull) atomicMin(job.error, first_bad);
  if (job.null_count && (threadIdx.x & 31) == 0 && nulls) atomicAdd(job.null_count, (unsigned long long)nulls);
}

// utf8 rows -> positions through the lookup table.  Offsets are read one per lane (lane 31 loads one more), the first 12
// bytes of a row by 4 aligned words + funnel shifts, as in rev_string_kernel.
template <bool LARGE>
__global__ void __launch_bounds__(kThreads)
rev_enum_string_kernel(dmb_rev_enum_job job, int64_t nrows, int64_t capacity, int smem) {
  using off_t = typename std::conditional<LARGE, long long, int>::type;
  const uint4 *tab = reinterpret_cast<const uint4 *>(job.table);
  if (smem) {
    for (uint32_t i = threadIdx.x; i < 2 * job.table_size; i += kThreads) rev_enum_smem[i] = __ldg(tab + i);
    __syncthreads();
    tab = rev_enum_smem;
  }
  const uint32_t mask = job.table_size - 1;
  const off_t *off = reinterpret_cast<const off_t *>(job.in_offsets);
  const int lane = threadIdx.x & 31;
  const bool has_bm = job.in_validity != nullptr;
  const BitSrc bs = bit_src(job.in_validity, job.in_bit_offset);
  int nulls = 0;
  unsigned long long first_bad = ~0ull;
  for (int64_t base = (int64_t)blockIdx.x * kThreads; base < capacity; base += (int64_t)gridDim.x * kThreads) {
    const int64_t row = base + threadIdx.x, row0 = row - lane;
    const off_t o0 = __ldg(off + (row < nrows ? row : nrows));
    const int64_t left = nrows - row0;
    const int live = left <= 0 ? 0 : (left < 32 ? (int)left : 32);
    const uint32_t vb = live == 0 ? 0u : (has_bm ? load_bits32(bs.w, bs.base + row0, live) : (live == 32 ? 0xffffffffu : ((1u << live) - 1u)));
    off_t o1 = __shfl_down_sync(0xffffffffu, o0, 1);
    if (lane == 31) o1 = __ldg(off + (row + 1 < nrows ? row + 1 : nrows));
    uint32_t code = DMB_ENUM_CODE_MISSING;
    if ((vb >> lane) & 1u) {
      const uint32_t len = (uint32_t)(o1 - o0);
      const uint8_t *q = job.in_data + o0;
      const uint32_t *b32 = reinterpret_cast<const uint32_t *>(reinterpret_cast<uintptr_t>(q) & ~(uintptr_t)3);
      const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(q) & 3u) * 8u;
      const uint32_t a0 = __ldg(b32), a1 = __ldg(b32 + 1), a2 = __ldg(b32 + 2), a3 = __ldg(b32 + 3);
      auto keep = [](uint32_t word, int nb) { return nb >= 4 ? word : (nb <= 0 ? 0u : (word & ((1u << (8 * nb)) - 1u))); };
      const uint32_t w0 = keep(__funnelshift_r(a0, a1, sh), (int)len), w1 = keep(__funnelshift_r(a1, a2, sh), (int)len - 4),
                     w2 = keep(__funnelshift_r(a2, a3, sh), (int)len - 8);
      uint32_t tail = 0;
      if (len > 12u) {
        const uint8_t *t = q + len - 4;
        const uint32_t *t32 = reinterpret_cast<const uint32_t *>(reinterpret_cast<uintptr_t>(t) & ~(uintptr_t)3);
        tail = __funnelshift_r(__ldg(t32), __ldg(t32 + 1), (uint32_t)(reinterpret_cast<uintptr_t>(t) & 3u) * 8u);
      }
      code = enum_probe(tab, mask, len, w0, w1, w2, tail, q, job.label_offsets, job.label_data);
    }
    enum_emit(job, row, nrows, vb, code, nulls, first_bad);
  }
  enum_finish(job, nulls, first_bad);
}

// Arrow dictionary indices -> positions through the remap (the codes of the dictionary's labels); four rows per thread
// in flight, each warp's loads and stores contiguous.
template <typename I>
__global__ void __launch_bounds__(kThreads)
rev_enum_index_kernel(dmb_rev_enum_job job, int64_t nrows, int64_t capacity, int smem) {
  constexpr int U = 4;
  const uint32_t *remap = job.remap;
  if (smem) {
    uint32_t *s = reinterpret_cast<uint32_t *>(rev_enum_smem);
    for (int64_t i = threadIdx.x; i < job.dict_len; i += kThreads) s[i] = __ldg(remap + i);
    __syncthreads();
    remap = s;
  }
  const I *in = reinterpret_cast<const I *>(job.in_indices);
  const int lane = threadIdx.x & 31;
  const bool has_bm = job.in_validity != nullptr;
  const BitSrc bs = bit_src(job.in_validity, job.in_bit_offset);
  int nulls = 0;
  unsigned long long first_bad = ~0ull;
  for (int64_t base = (int64_t)blockIdx.x * (U * kThreads); base < capacity; base += (int64_t)gridDim.x * (U * kThreads)) {
    I raw[U];
    uint32_t vb[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row = base + u * kThreads + threadIdx.x;
      raw[u] = row < nrows ? __ldcs(in + row) : I(0);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row0 = base + u * kThreads + threadIdx.x - lane;
      vb[u] = rev_warp_bits(bs, has_bm, rev_warp_live(nrows, row0), row0);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row = base + u * kThreads + threadIdx.x;
      const int64_t idx = rev_dict_index(raw[u], job.index_signed != 0);
      uint32_t code = DMB_ENUM_CODE_MISSING;
      if (((vb[u] >> lane) & 1u) && idx >= 0 && idx < job.dict_len) code = remap[idx];
      enum_emit(job, row, nrows, vb[u], code, nulls, first_bad);
    }
  }
  enum_finish(job, nulls, first_bad);
}

// ---- VARCHAR / BLOB from Arrow string views (dmb_rev_view_job): a 16 B -> 16 B streaming transform, four rows per thread
// in flight; a warp's 32 rows share one validity word, which is also the mask word.
__device__ __forceinline__ uint32_t keep_bytes(uint32_t word, int nb) { return nb >= 4 ? word : (nb <= 0 ? 0u : (word & ((1u << (8 * nb)) - 1u))); }

__global__ void __launch_bounds__(kThreads)
rev_view_kernel(dmb_rev_view_job job, int64_t nrows, int64_t capacity) {
  constexpr int U = 4;
  const uint4 *in = reinterpret_cast<const uint4 *>(job.in_views);
  const longlong2 *bufs = reinterpret_cast<const longlong2 *>(job.buffers);
  const int lane = threadIdx.x & 31;
  const bool has_bm = job.in_validity != nullptr;
  const BitSrc bs = bit_src(job.in_validity, job.in_bit_offset);
  uint4 *out = reinterpret_cast<uint4 *>(job.out);
  uint32_t *out_val32 = reinterpret_cast<uint32_t *>(job.out_validity);
  int nulls = 0;
  unsigned long long first_bad = ~0ull;
  for (int64_t base = (int64_t)blockIdx.x * (U * kThreads); base < capacity; base += (int64_t)gridDim.x * (U * kThreads)) {
    uint4 v[U];
    uint32_t vb[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row = base + u * kThreads + threadIdx.x;
      v[u] = row < nrows ? ld_stream(in + row) : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row0 = base + u * kThreads + threadIdx.x - lane;
      const int live = rev_warp_live(nrows, row0);
      vb[u] = rev_warp_bits(bs, has_bm, live, row0);
      if (lane == 0) {
        if (out_val32) out_val32[row0 >> 5] = vb[u];
        nulls += live - __popc(vb[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row = base + u * kThreads + threadIdx.x;
      uint4 e = make_uint4(0, 0, 0, 0);
      if ((vb[u] >> lane) & 1u) {
        const int len = (int)v[u].x;
        bool bad = len < 0;
        if (len >= 0 && len <= 12) {
          e = make_uint4(v[u].x, keep_bytes(v[u].y, len), keep_bytes(v[u].z, len - 4), keep_bytes(v[u].w, len - 8));
        } else if (len > 12) {
          const uint32_t idx = v[u].z;
          const int off = (int)v[u].w;
          bad = (int64_t)idx >= job.nbuffers || off < 0;
          if (!bad) {
            const longlong2 b = __ldg(bufs + idx);
            bad = (int64_t)off + len > b.y;
            const uint64_t p = (uint64_t)b.x + (uint64_t)off;
            if (!bad) e = make_uint4(v[u].x, v[u].y, (uint32_t)p, (uint32_t)(p >> 32));
          }
        }
        if (bad && (unsigned long long)row < first_bad) first_bad = (unsigned long long)row;
      }
      st_stream(out + row, e);
    }
  }
  if (first_bad != ~0ull) atomicMin(job.error, first_bad);
  if (job.null_count && lane == 0 && nulls) atomicAdd(job.null_count, (unsigned long long)nulls);
}

// ---- VARCHAR / BLOB from Arrow dictionary indices (dmb_rev_dict_job): row r takes table[index] (one 16-byte entry, from
// shared memory when the table fits); four rows per thread in flight, the mask word is the ballot of the rows that got a
// valid entry.
template <typename I>
__global__ void __launch_bounds__(kThreads)
rev_dict_kernel(dmb_rev_dict_job job, int64_t nrows, int64_t capacity, int smem) {
  constexpr int U = 4;
  const uint4 *tab = reinterpret_cast<const uint4 *>(job.table);
  if (smem) {
    for (int64_t i = threadIdx.x; i < job.dict_len; i += kThreads) rev_enum_smem[i] = __ldg(tab + i);
    __syncthreads();
    tab = rev_enum_smem;
  }
  const I *in = reinterpret_cast<const I *>(job.in_indices);
  const int lane = threadIdx.x & 31;
  const bool has_bm = job.in_validity != nullptr;
  const BitSrc bs = bit_src(job.in_validity, job.in_bit_offset);
  uint4 *out = reinterpret_cast<uint4 *>(job.out);
  uint32_t *out_val32 = reinterpret_cast<uint32_t *>(job.out_validity);
  int nulls = 0;
  unsigned long long first_bad = ~0ull;
  for (int64_t base = (int64_t)blockIdx.x * (U * kThreads); base < capacity; base += (int64_t)gridDim.x * (U * kThreads)) {
    I raw[U];
    uint32_t vb[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row = base + u * kThreads + threadIdx.x;
      raw[u] = row < nrows ? __ldcs(in + row) : I(0);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row0 = base + u * kThreads + threadIdx.x - lane;
      vb[u] = rev_warp_bits(bs, has_bm, rev_warp_live(nrows, row0), row0);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row = base + u * kThreads + threadIdx.x;
      const int64_t idx = rev_dict_index(raw[u], job.index_signed != 0);
      uint4 e = make_uint4(0, 0, 0, 0);
      bool ok = false;
      if ((vb[u] >> lane) & 1u) {
        if (idx < 0 || idx >= job.dict_len) {
          if ((unsigned long long)row < first_bad) first_bad = (unsigned long long)row;
        } else {
          const uint4 t = tab[idx];
          ok = t.x != DMB_DICT_ENTRY_NULL;
          if (ok) e = t;
        }
      }
      const uint32_t word = __ballot_sync(0xffffffffu, ok);
      st_stream(out + row, e);
      if (lane == 0) {
        out_val32[row >> 5] = word;
        nulls += rev_warp_live(nrows, row) - __popc(word);
      }
    }
  }
  if (first_bad != ~0ull) atomicMin(job.error, first_bad);
  if (job.null_count && lane == 0 && nulls) atomicAdd(job.null_count, (unsigned long long)nulls);
}

__global__ void rev_dict_mark_kernel(dmb_string_t *table, const uint64_t *masks, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads)
    if (!((__ldg(masks + (i >> 6)) >> (i & 63)) & 1ull)) reinterpret_cast<uint32_t *>(table + i)[0] = DMB_DICT_ENTRY_NULL;
}

// the key of a label on the host: what rev_enum_string_kernel computes from the row's bytes
void enum_host_key(const uint8_t *p, uint32_t len, uint32_t *w, uint32_t *tail) {
  uint8_t b[12] = {0};
  if (len) memcpy(b, p, len < 12 ? len : 12);
  memcpy(w, b, 12);
  *tail = 0;
  if (len > 12) memcpy(tail, p + len - 4, 4);
}

}  // namespace dmb

using namespace dmb;

extern "C" int32_t dmb_rev_enum_table(const dmb_enum_dict *d, uint32_t table_size, void *slots) {
  if (!d || !slots || (d->size && !d->offsets)) { set_error("dmb_rev_enum_table: null dictionary or table"); return 0; }
  if (table_size == 0 || (table_size & (table_size - 1)) || table_size <= d->size) {
    set_error("dmb_rev_enum_table: a table of %u slots cannot hold %u labels (a power of two above the label count)", table_size, d->size);
    return 0;
  }
  if (d->size && (d->offsets[0] != 0 || (d->offsets[d->size] && !d->data))) { set_error("ENUM dictionary offsets must start at 0 and come with data"); return 0; }
  for (uint32_t i = 0; i < d->size; ++i)
    if (d->offsets[i + 1] < d->offsets[i]) { set_error("ENUM dictionary offsets are not monotonic at label %u", i); return 0; }
  uint4 *s = static_cast<uint4 *>(slots);
  for (uint32_t i = 0; i < table_size; ++i) {
    s[2 * i] = make_uint4(DMB_ENUM_CODE_MISSING, 0, 0, 0);
    s[2 * i + 1] = make_uint4(0, 0, 0, 0);
  }
  const uint8_t *data = reinterpret_cast<const uint8_t *>(d->data);
  for (uint32_t p = 0; p < d->size; ++p) {
    const uint8_t *q = data + d->offsets[p];
    const uint32_t len = d->offsets[p + 1] - d->offsets[p];
    uint32_t w[3], tail;
    enum_host_key(q, len, w, &tail);
    const uint32_t dup = enum_probe(s, table_size - 1, len, w[0], w[1], w[2], tail, q, d->offsets, data);
    if (dup != DMB_ENUM_CODE_MISSING) {
      set_error("ENUM labels %u and %u are both '%.*s'", dup, p, (int)(len < 64 ? len : 64), (const char *)q);
      return 0;
    }
    uint32_t i = dmb_enum_hash(len, w[0], w[1], w[2], tail) & (table_size - 1);
    while (s[2 * i].x != DMB_ENUM_CODE_MISSING) i = (i + 1) & (table_size - 1);
    s[2 * i] = make_uint4(p, len, dmb_enum_hash(len, w[0], w[1], w[2], tail), 0);
    s[2 * i + 1] = make_uint4(w[0], w[1], w[2], tail);
  }
  return 1;
}

extern "C" int64_t dmb_rev_enum_lookup(const void *slots, uint32_t table_size, const dmb_enum_dict *d, const uint8_t *bytes, uint32_t len) {
  if (!slots || !d || table_size == 0 || (len && !bytes)) return -1;
  uint32_t w[3], tail;
  enum_host_key(bytes, len, w, &tail);
  const uint32_t p = enum_probe(static_cast<const uint4 *>(slots), table_size - 1, len, w[0], w[1], w[2], tail, bytes, d->offsets,
                                reinterpret_cast<const uint8_t *>(d->data));
  return p == DMB_ENUM_CODE_MISSING ? -1 : (int64_t)p;
}

extern "C" int32_t dmb_dev_rev_enum_batch(const dmb_rev_enum_job *job, int64_t nrows, void *stream) {
  if (!job) { set_error("dmb_dev_rev_enum_batch: job is null"); return -1; }
  if (nrows <= 0) return 0;
  const int ow = job->out_width, iw = job->index_width;
  if ((ow != 0 && ow != 1 && ow != 2 && ow != 4) || (iw != 0 && iw != 1 && iw != 2 && iw != 4 && iw != 8) || (ow == 0 && iw != 0)) {
    set_error("dmb_dev_rev_enum_batch: out_width %d / index_width %d", ow, iw);
    return -1;
  }
  if (!job->out || (ow && (!job->out_validity || !job->error)) ||
      (iw == 0 && (!job->in_offsets || !job->in_data || !job->table || !job->label_offsets || !job->table_size ||
                   (job->table_size & (job->table_size - 1)))) ||
      (iw && (!job->in_indices || job->dict_len < 0 || (job->dict_len && !job->remap)))) {
    set_error("dmb_dev_rev_enum_batch: a required pointer is null or the table size is not a power of two");
    return -1;
  }
  const int64_t chunks = ((nrows + kVec - 1) / kVec) * (int64_t)kVec;
  const int64_t max_grid = (int64_t)kNumSMs * 8;
  cudaStream_t st = (cudaStream_t)stream;
  if (iw == 0) {
    const int64_t capacity = ow ? chunks : ((nrows + 31) / 32) * 32;  // remap mode: codes only, no masks to fill
    const size_t tb = (size_t)job->table_size * DMB_ENUM_SLOT_BYTES;
    const int smem = tb <= (size_t)kEnumSmemBytes ? (int)tb : 0;
    const int64_t blocks = (capacity + kThreads - 1) / kThreads;
    const int gx = (int)(blocks < max_grid ? blocks : max_grid);
    if (job->large_offsets) rev_enum_string_kernel<true><<<gx, kThreads, smem, st>>>(*job, nrows, capacity, smem);
    else rev_enum_string_kernel<false><<<gx, kThreads, smem, st>>>(*job, nrows, capacity, smem);
    return check_cuda(cudaGetLastError(), "rev_enum_string_kernel launch");
  }
  const size_t rb = (size_t)job->dict_len * 4;
  const int smem = rb <= (size_t)kEnumSmemBytes ? (int)((rb + 15) & ~(size_t)15) : 0;
  const int64_t blocks = chunks / (4 * kThreads);
  const int gx = (int)(blocks < max_grid ? blocks : max_grid);
  switch (iw) {
    case 1: rev_enum_index_kernel<uint8_t><<<gx, kThreads, smem, st>>>(*job, nrows, chunks, smem); break;
    case 2: rev_enum_index_kernel<unsigned short><<<gx, kThreads, smem, st>>>(*job, nrows, chunks, smem); break;
    case 4: rev_enum_index_kernel<unsigned int><<<gx, kThreads, smem, st>>>(*job, nrows, chunks, smem); break;
    default: rev_enum_index_kernel<unsigned long long><<<gx, kThreads, smem, st>>>(*job, nrows, chunks, smem); break;
  }
  return check_cuda(cudaGetLastError(), "rev_enum_index_kernel launch");
}

extern "C" int32_t dmb_dev_rev_view_batch(const dmb_rev_view_job *job, int64_t nrows, void *stream) {
  if (!job) { set_error("dmb_dev_rev_view_batch: job is null"); return -1; }
  if (nrows <= 0) return 0;
  if (!job->in_views || !job->out || !job->error || job->nbuffers < 0 || (job->nbuffers && !job->buffers) ||
      (reinterpret_cast<uintptr_t>(job->in_views) & 15u)) {
    set_error("dmb_dev_rev_view_batch: a required pointer is null or the views are not 16-byte aligned");
    return -1;
  }
  const int64_t capacity = ((nrows + kVec - 1) / kVec) * (int64_t)kVec;  // a multiple of 4 * kThreads
  const int64_t blocks = capacity / (4 * kThreads), max_grid = (int64_t)kNumSMs * 8;
  const int gx = (int)(blocks < max_grid ? blocks : max_grid);
  rev_view_kernel<<<gx, kThreads, 0, (cudaStream_t)stream>>>(*job, nrows, capacity);
  return check_cuda(cudaGetLastError(), "rev_view_kernel launch");
}

extern "C" int32_t dmb_dev_rev_dict_batch(const dmb_rev_dict_job *job, int64_t nrows, void *stream) {
  if (!job) { set_error("dmb_dev_rev_dict_batch: job is null"); return -1; }
  if (nrows <= 0) return 0;
  const int iw = job->index_width;
  if (iw != 1 && iw != 2 && iw != 4 && iw != 8) { set_error("dmb_dev_rev_dict_batch: index_width %d", iw); return -1; }
  if (!job->in_indices || !job->out || !job->out_validity || !job->error || job->dict_len < 0 || (job->dict_len && !job->table)) {
    set_error("dmb_dev_rev_dict_batch: a required pointer is null");
    return -1;
  }
  const int64_t capacity = ((nrows + kVec - 1) / kVec) * (int64_t)kVec;
  const size_t tb = (size_t)job->dict_len * sizeof(dmb_string_t);
  const int smem = tb <= (size_t)kEnumSmemBytes ? (int)tb : 0;
  const int64_t blocks = capacity / (4 * kThreads), max_grid = (int64_t)kNumSMs * 8;
  const int gx = (int)(blocks < max_grid ? blocks : max_grid);
  cudaStream_t st = (cudaStream_t)stream;
  switch (iw) {
    case 1: rev_dict_kernel<uint8_t><<<gx, kThreads, smem, st>>>(*job, nrows, capacity, smem); break;
    case 2: rev_dict_kernel<unsigned short><<<gx, kThreads, smem, st>>>(*job, nrows, capacity, smem); break;
    case 4: rev_dict_kernel<unsigned int><<<gx, kThreads, smem, st>>>(*job, nrows, capacity, smem); break;
    default: rev_dict_kernel<unsigned long long><<<gx, kThreads, smem, st>>>(*job, nrows, capacity, smem); break;
  }
  return check_cuda(cudaGetLastError(), "rev_dict_kernel launch");
}

extern "C" int32_t dmb_dev_rev_dict_mark(dmb_string_t *table, const uint64_t *masks, int64_t n, void *stream) {
  if (n <= 0) return 0;
  if (!table || !masks) { set_error("dmb_dev_rev_dict_mark: table or masks is null"); return -1; }
  const int64_t blocks = (n + kThreads - 1) / kThreads, max_grid = (int64_t)kNumSMs * 8;
  rev_dict_mark_kernel<<<(int)(blocks < max_grid ? blocks : max_grid), kThreads, 0, (cudaStream_t)stream>>>(table, masks, n);
  return check_cuda(cudaGetLastError(), "rev_dict_mark_kernel launch");
}

extern "C" int32_t dmb_dev_rev_fixed_batch(const dmb_rev_fixed_job *jobs_dev, const dmb_rev_fixed_job *jobs_host,
                                           int32_t njobs, int64_t nrows, void *stream) {
  if (njobs <= 0 || nrows <= 0) return 0;
  if (!jobs_dev || !jobs_host) { set_error("dmb_dev_rev_fixed_batch: jobs is null"); return -1; }
  for (int32_t j = 0; j < njobs; ++j)
    if (jobs_host[j].op < 0 || jobs_host[j].op >= DMB_REV_COUNT) { set_error("dmb_dev_rev_fixed_batch: bad op %d", jobs_host[j].op); return -1; }
  int64_t blocks = (nrows / 2 + 4 * kThreads - 1) / (4 * kThreads);  // a CTA iteration moves 4 * 256 vectors of >= 2 rows
  int64_t max_grid = (int64_t)kNumSMs * 4;
  int gx = (int)(blocks < 1 ? 1 : (blocks < max_grid ? blocks : max_grid));
  rev_fixed_kernel<<<dim3(gx, njobs), kThreads, 0, (cudaStream_t)stream>>>(jobs_dev, nrows);
  return check_cuda(cudaGetLastError(), "rev_fixed_kernel launch");
}

extern "C" int32_t dmb_dev_rev_mask_batch(const dmb_rev_mask_job *jobs_dev, const dmb_rev_mask_job *jobs_host, int32_t njobs,
                                          int64_t nrows, void *stream) {
  if (njobs <= 0 || nrows <= 0) return 0;
  if (!jobs_dev || !jobs_host) { set_error("dmb_dev_rev_mask_batch: jobs is null"); return -1; }
  if (njobs > 65535) { set_error("dmb_dev_rev_mask_batch: %d jobs (at most 65535)", njobs); return -1; }
  for (int32_t j = 0; j < njobs; ++j)
    if (!jobs_host[j].out || jobs_host[j].out_bit_offset < 0 || jobs_host[j].out_bit_offset > 63 || jobs_host[j].a_bit_offset < 0 ||
        jobs_host[j].b_bit_offset < 0) {
      set_error("dmb_dev_rev_mask_batch: job %d has no output or a bit offset out of range", j);
      return -1;
    }
  const int64_t words = ((nrows + 63 + kVec - 1) / kVec) * DMB_VALIDITY_WORDS;  // the most any job writes
  const int64_t blocks = (words + kThreads - 1) / kThreads, max_grid = (int64_t)kNumSMs * 8;
  const int gx = (int)(blocks < max_grid ? blocks : max_grid);
  rev_mask_kernel<<<dim3(gx, njobs), kThreads, 0, (cudaStream_t)stream>>>(jobs_dev, nrows);
  return check_cuda(cudaGetLastError(), "rev_mask_kernel launch");
}

extern "C" int32_t dmb_dev_rev_string_batch(const dmb_rev_string_job *job, int64_t nrows, void *stream) {
  if (!job) { set_error("dmb_dev_rev_string_batch: job is null"); return -1; }
  if (nrows <= 0) return 0;
  int64_t capacity = ((nrows + kVec - 1) / kVec) * (int64_t)kVec;
  int64_t blocks = capacity / (2 * kThreads);
  int64_t max_grid = (int64_t)kNumSMs * 8;
  int gx = (int)(blocks < max_grid ? blocks : max_grid);
  if (job->large_offsets) rev_string_kernel<true><<<gx, kThreads, 0, (cudaStream_t)stream>>>(*job, nrows);
  else rev_string_kernel<false><<<gx, kThreads, 0, (cudaStream_t)stream>>>(*job, nrows);
  return check_cuda(cudaGetLastError(), "rev_string_kernel launch");
}

extern "C" int32_t dmb_dev_rev_list_batch(const dmb_rev_list_job *job, int64_t nrows, void *stream) {
  if (!job) { set_error("dmb_dev_rev_list_batch: job is null"); return -1; }
  if (nrows <= 0) return 0;
  if (!job->in_offsets || !job->child_word || !job->out_entries || !job->out_validity || !job->out_child_validity || !job->error) {
    set_error("dmb_dev_rev_list_batch: a required pointer is null");
    return -1;
  }
  int64_t capacity = ((nrows + kVec - 1) / kVec) * (int64_t)kVec;
  int64_t blocks = capacity / (2 * kThreads);
  int64_t max_grid = (int64_t)kNumSMs * 8;
  int gx = (int)(blocks < max_grid ? blocks : max_grid);
  if (job->large_offsets) rev_list_kernel<true><<<gx, kThreads, 0, (cudaStream_t)stream>>>(*job, nrows);
  else rev_list_kernel<false><<<gx, kThreads, 0, (cudaStream_t)stream>>>(*job, nrows);
  return check_cuda(cudaGetLastError(), "rev_list_kernel launch");
}
