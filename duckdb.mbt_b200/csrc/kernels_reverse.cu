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

}  // namespace dmb

using namespace dmb;

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
