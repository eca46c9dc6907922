// K5 string_unpack: duckdb_string_t[16 B] -> Arrow utf8 (offsets + data) in ONE pass.
//
// Tile = 512 consecutive rows of one chunk (four tiles per 2048-row vector).  A CTA
//   1. claims the next tile from a global ticket (so every predecessor belongs to a running CTA: the look-back always makes progress),
//   2. loads the tile's string_t into shared memory with coalesced 128-bit loads (read once),
//   3. block-scans the (validity-masked) lengths into tile-local offsets and, in the same scan, a
//      running maximum that gives every row the first row of its RUN: a maximal sequence of rows
//      whose source bytes follow one another in the heap (DuckDB fills its string heap in row
//      order, so runs are long; an inlined string or a scattered pointer starts a new run),
//   4. publishes its aggregate and resolves its exclusive base by decoupled look-back over the
//      predecessors' 64-bit status words (flag | value in one word, so no fences are needed),
//   5. writes offsets (coalesced), and
//   6. gathers the bytes OUTPUT-centrically: a thread owns one 16-byte aligned vector of the
//      output stream.  Rows first publish, per vector, which row holds the vector's first byte
//      (a 2-byte map entry: O(1) lookup, no search).  A vector that lies inside one run (the
//      common case) is three aligned 64-bit loads, two funnel shifts and one 128-bit streaming
//      store, with no branches on the data.  Vectors that straddle a run boundary are queued in
//      a shared-memory list and finished afterwards by a dense loop that walks their rows and
//      merges the pieces with byte masks, so the divergent work is paid per such vector and not
//      per warp.  Consecutive threads read consecutive heap bytes and write consecutive
//      vectors; the data bytes never touch shared memory.
//
// Replaces the reference's per-cell string_t read src/duckdb_native.c:597-603 and the two-pass
// malloc/strlen/memcpy getters :2474-2510 and :2699-2755.  DMB_STR_REF_BLOB reproduces the
// getter's NUL-terminated stream (strlen semantics) instead of Arrow offsets.

#include "dmb_common.cuh"

namespace dmb {

constexpr int kStrTileRows = 512;
constexpr int kStrMinCtas = 7;                          // CTAs per SM of string_batch_kernel (launch bound)
constexpr int kStrTilesPerChunk = kVec / kStrTileRows;
constexpr int kStrPerThread = kStrTileRows / kThreads;  // 2 consecutive rows per thread in the scan
constexpr int kMapVecs = 2048;                          // output vectors per window (32 KiB of utf8 data)
constexpr uint32_t kMaxRowBytes = 1u << 21;             // tile-local sums stay below 2^32 (<= 2048 rows * 2 MiB)


// scratch layout (uint64 words): [0] tile ticket  [1] error flags  [2..] tile status
enum { kErrTileTooBig = 1, kErrOffsetOverflow = 2, kErrHeapRange = 4, kErrDataCap = 8, kErrTimeout = 16 };

// Tiles are claimed from a global ticket (scratch[0], zeroed by the launch wrapper), never from blockIdx: CUDA does
// not promise to dispatch CTAs in blockIdx order, and a look-back may only wait for tiles that RUNNING CTAs own.
__device__ __forceinline__ int64_t claim_tile(unsigned long long *scratch, long long *slot) {
  if (threadIdx.x == 0) *slot = (long long)atomicAdd(scratch, 1ull);
  __syncthreads();
  return (int64_t)*slot;
}

struct StrSmem {
  uint4 str[kStrTileRows];            // string_t copies
  uint64_t src[kStrTileRows];         // device (generic) address of every row's first byte, minus its tile-local offset
  uint32_t off[kStrTileRows + 4];     // tile-local exclusive offsets; off[kStrTileRows] = tile total
  uint16_t run[kStrTileRows];         // first row of the run a row belongs to
  union {
    struct {
      uint16_t first_row[kMapVecs + 2];  // per output vector of the window: the row that holds its first byte
      uint16_t slow[kMapVecs];           // window-local ids of the vectors that straddle a run boundary
    };
    alignas(16) uint8_t stage[kStrTileRows * 13 + 32];  // all-inline tiles: the tile's whole output (<= 13 B per row)
  };
  uint4 low_mask[17];                 // low_mask[d]: bytes < d of a 16-byte vector are 0xff
  uint32_t warp_sum[kThreads / 32];
  uint32_t warp_run[kThreads / 32];
  uint64_t base;
  long long ticket;
};


// (y:x) >> s bits, s in {0, 8, ..., 56}
__device__ __forceinline__ uint64_t funnel64(uint64_t x, uint64_t y, uint32_t s) {
  const uint32_t x0 = (uint32_t)x, x1 = (uint32_t)(x >> 32), y0 = (uint32_t)y, y1 = (uint32_t)(y >> 32);
  const bool up = s >= 32u;
  const uint32_t a = up ? x1 : x0, b = up ? y0 : x1, c = up ? y1 : y0;
  const uint32_t lo = __funnelshift_r(a, b, s), hi = __funnelshift_r(b, c, s);  // shift taken mod 32
  return ((uint64_t)hi << 32) | lo;
}

// 16 source bytes starting at sp (any alignment) as two 64-bit words.  Aligned loads only; the
// word past the 16 bytes is read only when it holds needed bytes.
__device__ __forceinline__ void load16(const uint8_t *sp, uint64_t &w0, uint64_t &w1) {
  const uintptr_t vs = reinterpret_cast<uintptr_t>(sp);
  const uint32_t t = (uint32_t)vs & 7u;
  const uint64_t *ab = reinterpret_cast<const uint64_t *>(vs - t);
  const uint64_t x0 = ab[0], x1 = ab[1], x2 = t ? ab[2] : 0ull;
  w0 = funnel64(x0, x1, 8u * t);
  w1 = funnel64(x1, x2, 8u * t);
}

// Merge source bytes [sp, sp + (d1 - d0)) into bytes [d0, d1) of the 16-byte vector (w0, w1).
// Whole aligned 64-bit words are read, but only words that hold needed bytes, so nothing outside
// the heap copy (+ its >= 16 bytes of padding) or the shared-memory string_t tile is touched.
// low_mask is the shared-memory byte-mask table.
__device__ __forceinline__ void emit(uint64_t &w0, uint64_t &w1, const uint8_t *sp, uint32_t d0, uint32_t d1,
                                     const uint4 *low_mask) {
  const uintptr_t vs = reinterpret_cast<uintptr_t>(sp) - d0;  // source address of vector byte 0
  const uint32_t t = (uint32_t)vs & 7u;
  const uint64_t *ab = reinterpret_cast<const uint64_t *>(vs - t);
  const uint32_t f = d0 + t, l = d1 + t;  // needed source bytes, relative to ab: [f, l)
  const uint64_t x0 = f < 8u ? ab[0] : 0ull;
  const uint64_t x1 = (f < 16u && l > 8u) ? ab[1] : 0ull;
  const uint64_t x2 = l > 16u ? ab[2] : 0ull;  // l > 16 implies t != 0
  const uint64_t v0 = funnel64(x0, x1, 8u * t), v1 = funnel64(x1, x2, 8u * t);
  const uint4 hi = low_mask[d1], lo = low_mask[d0];
  const uint64_t m0 = (((uint64_t)hi.y << 32) | hi.x) & ~(((uint64_t)lo.y << 32) | lo.x);
  const uint64_t m1 = (((uint64_t)hi.w << 32) | hi.z) & ~(((uint64_t)lo.w << 32) | lo.z);
  w0 |= v0 & m0;
  w1 |= v1 & m1;
}

// bytes [nb0, nb1) of a 32-bit word, 0 <= nb0 < nb1 <= 4
__device__ __forceinline__ uint32_t byte_mask32(uint32_t nb0, uint32_t nb1) {
  const uint32_t hi = nb1 >= 4u ? 0xffffffffu : ((1u << (8u * nb1)) - 1u);
  return hi & ~((1u << (8u * nb0)) - 1u);
}

// place `val` (already positioned) into a 32-bit word of the zeroed inline stage: whole word ->
// store, part -> OR (neighbouring rows own the other bytes)
__device__ __forceinline__ void put32(uint32_t *w, uint32_t val, int nb0, int nb1) {
  nb0 = nb0 < 0 ? 0 : nb0;
  nb1 = nb1 > 4 ? 4 : nb1;
  if (nb1 <= nb0) return;
  if (nb1 - nb0 == 4) *w = val;
  else atomicOr(w, val & byte_mask32((uint32_t)nb0, (uint32_t)nb1));
}

// Step 6 of string_batch_kernel (see the header comment): output-centric gather of a tile whose
// sm.str / sm.src / sm.off / sm.run / sm.low_mask are filled.  `len` / `my_off` are the calling
// thread's own consecutive rows (tid * kStrPerThread + k) and its tile-local exclusive offset.
template <int MODE>
__device__ __forceinline__ void gather_runs(StrSmem &sm, int tid, int lane, int warp, const uint32_t (&len)[kStrPerThread],
                                            uint32_t my_off, uint32_t total, uint32_t mis, uint8_t *gbase, uint32_t nvec) {
  for (uint32_t q0 = 0; q0 < nvec; q0 += kMapVecs) {
    const uint32_t q1 = q0 + kMapVecs < nvec ? q0 + kMapVecs : nvec;
    const uint32_t qmap = q1 < nvec ? q1 + 1u : q1;  // one entry past the window: the fast-path test looks at v + 1
    // (a) every non-empty row publishes the vectors v with L(v) inside the row
    {
      uint32_t o = my_off;
#pragma unroll
      for (int k = 0; k < kStrPerThread; ++k) {
        const uint32_t start = o, stop = o + len[k];
        o = stop;
        if (stop == start) continue;
        uint32_t qa = start == 0u ? 0u : (start + mis + 15u) >> 4;  // first v with L(v) >= start
        uint32_t qb = (stop + mis + 15u) >> 4;                      // first v with L(v) >= stop
        qa = qa > q0 ? qa : q0;
        qb = qb < qmap ? qb : qmap;
        for (uint32_t q = qa; q < qb; ++q) sm.first_row[q - q0] = (uint16_t)(tid * kStrPerThread + k);
      }
    }
    __syncthreads();
    // (b) fast pass: every warp owns an equal, contiguous share of the window's vectors; vectors
    //     inside one run are finished here, the others go to the warp's own queue
    uint16_t *my_slow = sm.slow + warp * (kMapVecs / (kThreads / 32));
    uint32_t nslow = 0;
    const uint32_t per_warp = ((q1 - q0 + (kThreads / 32) * 32u - 1u) / ((kThreads / 32) * 32u)) * 32u;  // <= 256, multiple of 32
    const uint32_t wq0 = q0 + (uint32_t)warp * per_warp < q1 ? q0 + (uint32_t)warp * per_warp : q1;
    const uint32_t wq1 = wq0 + per_warp < q1 ? wq0 + per_warp : q1;
    for (uint32_t vb = wq0; vb < wq1; vb += 32) {
      const uint32_t v = vb + lane;
      bool slow = false;
      if (v < wq1) {
        const uint32_t vbeg = v << 4;
        const bool whole = (v > 0 || mis == 0) && (vbeg + 16u - mis <= total) && (v + 1u < nvec);
        const int r = sm.first_row[v - q0];
        slow = !whole || sm.run[r] != sm.run[sm.first_row[v + 1u - q0]];
        if (!slow) {
          uint64_t w0, w1;
          load16(reinterpret_cast<const uint8_t *>(sm.src[r] + (vbeg - mis)), w0, w1);
          st_stream(reinterpret_cast<uint4 *>(gbase + vbeg),
                    make_uint4((uint32_t)w0, (uint32_t)(w0 >> 32), (uint32_t)w1, (uint32_t)(w1 >> 32)));
        }
      }
      const uint32_t ballot = __ballot_sync(0xffffffffu, slow);
      if (slow) my_slow[nslow + __popc(ballot & ((1u << lane) - 1u))] = (uint16_t)(v - q0);
      nslow += __popc(ballot);
    }
    __syncwarp();
    // (c) dense pass over the warp's queued vectors: walk the rows, merge the pieces
#pragma unroll 1
    for (uint32_t idx = lane; idx < nslow; idx += 32) {
      const uint32_t v = q0 + my_slow[idx];
      const uint32_t vbeg = v << 4;                    // position + mis of the vector's first byte
      const uint32_t lo = v ? vbeg - mis : 0u;         // tile-local bytes [lo, hi) owned by this vector
      const uint32_t hi = (vbeg + 16u - mis) < total ? (vbeg + 16u - mis) : total;
      int r = sm.first_row[v - q0];
      uint64_t w0 = 0, w1 = 0;
      uint32_t seg_pos = lo;                           // current source stream covers [seg_pos, seg_end)
      const uint8_t *sp = reinterpret_cast<const uint8_t *>(sm.src[r] + lo);
      uint32_t row_end = sm.off[r + 1];
      uint32_t seg_end = MODE == DMB_STR_REF_BLOB ? row_end - 1u : row_end;  // payload end; the terminator stays 0
#pragma unroll 1
      while (row_end < hi) {
        int r2 = r + 1;                                // next non-empty row (off[] is packed: it starts at row_end)
        uint32_t o2 = sm.off[r2 + 1];
        while (o2 == row_end) { ++r2; o2 = sm.off[r2 + 1]; }
        const bool same_run = sm.run[r2] == sm.run[r];
        r = r2;
        if (same_run) {                                // heap bytes continue: same stream
          row_end = o2;
          seg_end = o2;
          continue;
        }
        if (seg_end > seg_pos) emit(w0, w1, sp, seg_pos + mis - vbeg, seg_end + mis - vbeg, sm.low_mask);
        seg_pos = row_end;
        sp = reinterpret_cast<const uint8_t *>(sm.src[r2] + row_end);
        row_end = o2;
        seg_end = MODE == DMB_STR_REF_BLOB ? o2 - 1u : o2;
      }
      {
        const uint32_t e = seg_end < hi ? seg_end : hi;
        if (e > seg_pos) emit(w0, w1, sp, seg_pos + mis - vbeg, e + mis - vbeg, sm.low_mask);
      }
      const bool full = (v > 0 || mis == 0) && (vbeg + 16u - mis <= total);
      if (full) {
        st_stream(reinterpret_cast<uint4 *>(gbase + vbeg),
                  make_uint4((uint32_t)w0, (uint32_t)(w0 >> 32), (uint32_t)w1, (uint32_t)(w1 >> 32)));
      } else {  // the neighbouring tiles own the other bytes of this vector
        const uint32_t b0 = lo + mis - vbeg, b1 = hi + mis - vbeg;
        for (uint32_t q = b0; q < b1; ++q) gbase[vbeg + q] = (uint8_t)((q < 8 ? w0 : w1) >> (8u * (q & 7u)));
      }
    }
    if (q1 < nvec) __syncthreads();
  }
}

template <int MODE>
__global__ void __launch_bounds__(kThreads, kStrMinCtas)
string_batch_kernel(dmb_string_job job, BatchView b, unsigned long long *scratch, int64_t ntiles) {
  __shared__ StrSmem sm;
  unsigned long long *status = scratch + 2;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  const int64_t tile = claim_tile(scratch, &sm.ticket);
  if (tile >= ntiles) return;
  if (tid < 17) {
    const uint32_t d = (uint32_t)tid;
    auto m = [&](uint32_t w) { return d >= 4u * w + 4u ? 0xffffffffu : (d <= 4u * w ? 0u : ((1u << (8u * (d - 4u * w))) - 1u)); };
    sm.low_mask[tid] = make_uint4(m(0), m(1), m(2), m(3));
  }
  const int64_t c = tile / kStrTilesPerChunk;
  const int r_begin = (int)(tile % kStrTilesPerChunk) * kStrTileRows;
  const int count = (int)__ldg(b.counts + c);
  int nrows_tile = count - r_begin;
  nrows_tile = nrows_tile < 0 ? 0 : (nrows_tile > kStrTileRows ? kStrTileRows : nrows_tile);
  const dmb_vec_desc vd = job.vecs[c];
  const uint4 *in = reinterpret_cast<const uint4 *>(reinterpret_cast<const uint8_t *>(job.in) + vd.data_off) + r_begin;
  const uint64_t *mask = vd.val_off < 0 ? nullptr : job.in_validity + vd.val_off;

  // 2. + 3. every thread loads its own consecutive rows (and lane 0 the row before them) straight
  //    into registers, together with the validity words, then derives length and source address;
  //    a row that contributes no bytes (NULL, empty, bad pointer) gets length 0 and is never
  //    touched again.  The shared-memory copy serves the inlined strings and the gather.
  int flags = 0;  // 1: a pointer (non-inlined) row is present  2: bad heap pointer  4: oversized row
  uint4 ent[kStrPerThread];
  bool ok[kStrPerThread];
#pragma unroll
  for (int k = 0; k < kStrPerThread; ++k) {
    const int i = tid * kStrPerThread + k;
    ent[k] = make_uint4(0, 0, 0, 0);
    ok[k] = false;
    if (i < nrows_tile) {
      ent[k] = ld_stream(in + i);
      const int row = r_begin + i;
      ok[k] = mask ? ((__ldg(mask + (row >> 6)) >> (row & 63)) & 1ull) : true;
    }
  }
#pragma unroll
  for (int k = 0; k < kStrPerThread; ++k) {
    const int i = tid * kStrPerThread + k;
    if (i < nrows_tile) sm.str[i] = ent[k];
  }
  if (MODE == DMB_STR_REF_BLOB) __syncthreads();  // strlen below reads inlined bytes of other threads' rows
  auto row_info = [&](int i, const uint4 &e, bool valid, uint32_t &l_out, uint64_t &src_out) {
    l_out = 0;
    src_out = 0;
    if (i < 0 || i >= nrows_tile) return;
    if (valid) {
      uint32_t l = e.x;
      const uint8_t *src = reinterpret_cast<const uint8_t *>(&sm.str[i]) + 4;
      if (l > 12u) {
        const uint64_t p = ((uint64_t)e.w << 32) | (uint64_t)e.z;
        const uint64_t rel = p - job.heap_host_base;
        if (l >= kMaxRowBytes) { flags |= 4; l = 0; }
        else if (p < job.heap_host_base || rel + l > job.heap_len) { flags |= 2; l = 0; }
        src = job.heap_dev + rel;
        if (l) {  // pull the heap bytes towards L2 while the scan and the look-back run
          flags |= 1;
          asm volatile("prefetch.global.L2 [%0];" ::"l"(src + l - 1u));
        }
      }
      if (MODE == DMB_STR_REF_BLOB) {  // strlen() of the malloc'ed copy: stop at an embedded NUL
        uint32_t n = 0;
        while (n < l && src[n] != 0) ++n;
        l = n;
      }
      l_out = l;
      src_out = reinterpret_cast<uint64_t>(src);
    }
    if (MODE == DMB_STR_REF_BLOB) l_out += 1;  // terminator; a NULL row is a lone '\0'
  };
  uint32_t len[kStrPerThread];
  uint64_t srcp[kStrPerThread];
  uint32_t tsum = 0;
#pragma unroll
  for (int k = 0; k < kStrPerThread; ++k) {
    row_info(tid * kStrPerThread + k, ent[k], ok[k], len[k], srcp[k]);
    tsum += len[k];
  }
  // run starts: row i starts a run unless its bytes directly follow those of row i-1
  uint32_t start_row[kStrPerThread];  // i + 1 when row i starts a run, else 0 (max-scanned below)
  {
    // the row before this thread's rows belongs to the previous lane; the first row of a warp
    // always starts a run (one extra boundary per 64 rows instead of a cross-warp dependency)
    uint32_t pl = __shfl_up_sync(0xffffffffu, len[kStrPerThread - 1], 1);
    uint64_t ps = __shfl_up_sync(0xffffffffu, srcp[kStrPerThread - 1], 1);
    if (lane == 0) pl = 0u;
#pragma unroll
    for (int k = 0; k < kStrPerThread; ++k) {
      const bool follows = MODE != DMB_STR_REF_BLOB && pl != 0u && srcp[k] == ps + pl;
      start_row[k] = (len[k] != 0u && !follows) ? (uint32_t)(tid * kStrPerThread + k) + 1u : 0u;
      if (len[k] != 0u) { pl = len[k]; ps = srcp[k]; } else { pl = 0u; }
    }
  }
  uint32_t incl = tsum;
  uint32_t rmax = 0;
#pragma unroll
  for (int k = 0; k < kStrPerThread; ++k) rmax = rmax > start_row[k] ? rmax : start_row[k];
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t n = __shfl_up_sync(0xffffffffu, incl, d);
    const uint32_t m = __shfl_up_sync(0xffffffffu, rmax, d);
    if (lane >= d) { incl += n; rmax = rmax > m ? rmax : m; }
  }
  if (lane == 31) { sm.warp_sum[warp] = incl; sm.warp_run[warp] = rmax; }
  const uint32_t rmax_excl_lane = __shfl_up_sync(0xffffffffu, rmax, 1);
  // __syncthreads_or yields a predicate, not the OR of the values: it carries the "pointer row
  // present" bit; the (rare) error bits are reported by the thread that saw them
  if (flags & 6) atomicOr(scratch + 1, (unsigned long long)(((flags & 2) ? kErrHeapRange : 0) | ((flags & 4) ? kErrTileTooBig : 0)));
  const int tile_flags = __syncthreads_or(flags & 1);
  uint32_t warp_excl = 0, tile_total = 0, run_excl = 0;
#pragma unroll
  for (int w = 0; w < kThreads / 32; ++w) {
    const uint32_t s = sm.warp_sum[w];
    const uint32_t m = sm.warp_run[w];
    if (w < warp) { warp_excl += s; run_excl = run_excl > m ? run_excl : m; }
    tile_total += s;
  }
  if (lane > 0) run_excl = run_excl > rmax_excl_lane ? run_excl : rmax_excl_lane;
  const uint32_t my_off = warp_excl + incl - tsum;
  {
    uint32_t o = my_off, run = run_excl;
#pragma unroll
    for (int k = 0; k < kStrPerThread; ++k) {
      sm.off[tid * kStrPerThread + k] = o;
      sm.src[tid * kStrPerThread + k] = srcp[k] - o;  // address of tile-local byte 0 if this row's stream started there
      o += len[k];
      run = run > start_row[k] ? run : start_row[k];
      sm.run[tid * kStrPerThread + k] = (uint16_t)run;  // (first row of the run) + 1; only read for non-empty rows
    }
    if (tid == kThreads - 1) sm.off[kStrTileRows] = o;
  }

  // 4. decoupled look-back (warp 0)
  if (warp == 0) {
    const uint64_t agg = (uint64_t)tile_total;
    if (lane == 0) atomicExch(status + tile, (tile == 0 ? kFlagPrefix : kFlagAggregate) | agg);
    uint64_t prefix = 0;
    if (tile > 0) {
      int64_t look = tile - 1;
      while (true) {
        const int64_t idx = look - lane;
        uint64_t st = kFlagPrefix;  // before tile 0: prefix 0
        if (idx >= 0) {
          do { st = ld_status(status + idx); } while ((st >> 62) == 0);
        }
        const uint32_t is_p = __ballot_sync(0xffffffffu, (st >> 62) == 2);
        const int first_p = is_p ? (__ffs(is_p) - 1) : 32;
        uint64_t v = lane <= first_p ? (st & kValueMask) : 0ull;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
        prefix += v;
        if (is_p) break;
        look -= 32;
      }
      if (lane == 0) atomicExch(status + tile, kFlagPrefix | ((prefix + agg) & kValueMask));
    }
    if (lane == 0) sm.base = prefix;
  }
  __syncthreads();
  const uint64_t base = sm.base;

  // 5. offsets
  {
    const int64_t out_row0 = __ldg(b.row_off + c) + r_begin;
    const bool overflow = MODE != DMB_STR_ARROW_LARGE && base + tile_total > 0x7fffffffull;
    if (overflow && tid == 0) atomicOr(scratch + 1, (unsigned long long)kErrOffsetOverflow);
    if (MODE == DMB_STR_ARROW_LARGE) {
      int64_t *oo = reinterpret_cast<int64_t *>(job.out_offsets);
      for (int i = tid; i < nrows_tile; i += kThreads) __stcs(reinterpret_cast<long long *>(oo + out_row0 + i), (long long)(base + sm.off[i]));
      if (tile == ntiles - 1 && tid == 0) oo[b.nrows] = (int64_t)(base + tile_total);
    } else {
      int32_t *oo = reinterpret_cast<int32_t *>(job.out_offsets);
      for (int i = tid; i < nrows_tile; i += kThreads) __stcs(oo + out_row0 + i, (int32_t)(base + sm.off[i]));
      if (tile == ntiles - 1 && tid == 0) oo[b.nrows] = (int32_t)(base + tile_total);
    }
    if (tile == ntiles - 1 && tid == 0 && job.total_bytes) *job.total_bytes = base + tile_total;
  }
  if (tile_total == 0) return;
  if (job.out_data_cap && base + tile_total > job.out_data_cap) {  // aliased pointers: more bytes than the caller sized for
    if (tid == 0) atomicOr(scratch + 1, (unsigned long long)kErrDataCap);
    return;
  }

  // 6. output-centric gather.  Vector v covers tile-local bytes [16v - mis, 16v - mis + 16), i.e. a
  //    16-byte aligned vector of out_data; L(v) = max(16v - mis, 0) is its first owned byte.
  const uint32_t total = tile_total;
  const uint32_t mis = (uint32_t)(base & 15ull);
  uint8_t *gbase = job.out_data + (base - mis);
  const uint32_t nvec = (mis + total + 15u) >> 4;
  if ((tile_flags & 1) == 0) {
    // All rows are inlined (<= 12 payload bytes each, in registers): one lane per row shifts its
    // bytes to the stage's word phase and ORs them into a zeroed shared-memory image of the tile's
    // output, which then leaves with coalesced 128-bit stores.
    const uint32_t end = mis + total;
    const uint32_t nstage = (end + 15u) >> 4;
    uint4 *sv = reinterpret_cast<uint4 *>(sm.stage);
    for (uint32_t i = tid; i < nstage; i += kThreads) sv[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    uint32_t *sw = reinterpret_cast<uint32_t *>(sm.stage);
#pragma unroll 1
    for (int i = tid; i < nrows_tile; i += kThreads) {
      const uint32_t s0 = mis + sm.off[i], s1 = mis + sm.off[i + 1];
      const uint32_t pay_end = MODE == DMB_STR_REF_BLOB ? s1 - 1u : s1;  // the terminator stays 0
      if (pay_end <= s0) continue;
      const uint4 e = sm.str[i];
      const uint32_t a = s0 & 3u, sh = 8u * a;
      const int l = (int)(pay_end - s0);
      uint32_t *w = sw + (s0 >> 2);
      put32(w, e.y << sh, (int)a, (int)a + l);
      put32(w + 1, __funnelshift_l(e.y, e.z, sh), (int)a - 4, (int)a + l - 4);
      put32(w + 2, __funnelshift_l(e.z, e.w, sh), (int)a - 8, (int)a + l - 8);
      put32(w + 3, __funnelshift_l(e.w, 0u, sh), (int)a - 12, (int)a + l - 12);
    }
    __syncthreads();
    for (uint32_t v = tid; v < nstage; v += kThreads) {
      const uint32_t p = 16u * v;
      if (p >= mis && p + 16u <= end) {
        st_stream(reinterpret_cast<uint4 *>(gbase + p), sv[v]);
      } else {  // the neighbouring tiles own the other bytes of this vector
        const uint32_t b0 = p > mis ? p : mis, b1 = (p + 16u) < end ? (p + 16u) : end;
        for (uint32_t q = b0; q < b1; ++q) gbase[q] = sm.stage[q];
      }
    }
    return;
  }
  gather_runs<MODE>(sm, tid, lane, warp, len, my_off, total, mis, gbase, nvec);
}

// ------------------------------------------------------------------ TMA-staged pack kernel
// string_pack_kernel<LARGE, R>: the Arrow utf8 path for columns of short strings (the common case:
// names, flags, comments).  The run-gather above pays ~20 warp-instructions per row when runs are
// short and every tile stalls on its own dependent chain (metadata -> string_t -> scan ->
// look-back -> gather).  This kernel is a persistent, warp-specialised pipeline: the byte movement
// in and out of the SM is done by the copy engine (cp.async.bulk), every long-latency step of tile
// t+1 is issued while tile t is being packed, and the SIMT part is row-centric and small.
//
//   CTA = NW worker warps + two single-purpose warps; tiles (NW*32*R consecutive rows of a chunk) are
//   claimed in order from a global ticket, so every predecessor of a claimed tile is owned by a
//   running CTA (the look-back cannot starve).  NW = 8 (3 CTAs per SM) for columns with a heap and
//   16 (2 CTAs per SM) for the lean heap-less form (pack_warps()).
//
//   P  claims tile j+2 (ticket, chunk metadata) and bulk-loads its string_t (and validity words)
//      into the S buffer the workers have just left; when the workers have packed a tile it
//      sends the stage O to out_data with bulk stores: one for the 16-byte aligned interior and
//      sm_100's byte-masked form (cp.async.bulk ... .cp_mask) for the ragged first / last vector,
//      whose other bytes belong to the neighbouring tiles.
//   W  front(j): own R consecutive rows from S -> lengths, block scan, span min/max (redux.sync);
//      one thread publishes the tile's aggregate and fetches the tile's heap span [hmin, hmax) into H[j&1] with ONE bulk copy.
//      back(j-1): offsets straight from registers (vector stores), then every thread streams its
//      rows' bytes (registers for inlined strings, the staged span for pointer strings) into the
//      output stage O with 32-bit funnel shifts: interior words are plain stores, the <= 2 words
//      a thread shares with its neighbours are written byte by byte.
//   L  decoupled look-back of tile j, started lazily (when the workers have scanned it: by then
//      its predecessors' aggregates, often their prefixes, are out) and due only when tile j-1
//      has been packed.
//
// A tile whose span or output does not fit the stages (scattered pointers, a long string) is copied
// row by row, one warp per row and one byte per lane, straight from the heap to out_data.
//
// profiles/r02_string_pack_kernel_iterations.txt has what each of these measures bought: pointer rows copied four words at
// a time, loads first; string_t read from S in a lane-rotated order (no bank conflicts); the inlined rows' last-word select
// as two bit tests; the two-level look-back (lookback_groups); UNIFY (inlined rows through a per-thread scratch slot and
// the pointer rows' copy loop).
constexpr uint32_t kPackTail = 1792;  // bytes of bookkeeping in front of the stages
constexpr int kMetaRing = 8;  // tiles j-1 (being sent) .. j+3 (ticket and metadata claimed) are alive at once
constexpr uint32_t kPackScratchPerThread = 12u;  // UNIFY kernels: one 12-byte slot per worker thread behind H
// worker warps per CTA: 8 with a heap (16 were no faster on the C2 columns), 16 for the heap-less lean form (faster than 8:
// see dmb_dev_string_batch)
__host__ __device__ constexpr int pack_warps(bool heap) { return heap ? 8 : 16; }

struct TileMeta {
  long long tile;            // -1: no more tiles
  long long out_row0;        // first output row of the tile
  int32_t nrows;             // rows of the tile that exist (chunk count - r_begin, clamped)
  int32_t has_mask;
  // written by P once the tile's string_t have landed and been summed
  uint32_t total;            // bytes of the tile
  uint32_t hmin;             // heap span start, 16-byte units from the heap base
  uint32_t hbytes;           // heap span bytes (multiple of 16)
  int32_t staged;            // the tile fits the stages
  // written by P with the ticket: where the tile's string_t / validity words are (the bulk loads are issued later, when S frees)
  const uint8_t *src;
  const uint64_t *val;       // nullptr: no mask
};

constexpr int kPackMaxWarps = 16;
struct PackPartials {
  uint32_t warp_sum[kPackMaxWarps];
  uint32_t warp_hmin[kPackMaxWarps];
  uint32_t warp_hmax[kPackMaxWarps];
  uint32_t warp_cmin[kPackMaxWarps];  // min / max over the warp's pointer rows of (pointer - tile-local offset):
  uint32_t warp_cmax[kPackMaxWarps];  // all equal <=> the tile's bytes are one contiguous piece of the heap
  uint32_t not_one_run;               // set by any warp that holds an inlined row or two runs
};

struct PackTail {
  unsigned long long mbar_s[2];
  unsigned long long mbar_h[2];
  unsigned long long base[kMetaRing];
  TileMeta meta[kMetaRing];
  PackPartials part[2];
  alignas(16) unsigned long long vmask[2][kVec / 64];  // validity words of the tile in S[slot] (bulk-copy destination)
};
static_assert(sizeof(PackTail) <= kPackTail, "PackTail");

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
// A wait that cannot end must not hang the GPU.  Look-backs (the only waits on OTHER CTAs) give up after 4 s with an
// error flag and let the launch finish; the mbarrier waits inside a CTA depend only on that CTA's own warps and copy
// engine transactions, so one that is still pending after 3x that long is a protocol bug: it traps.
constexpr unsigned long long kWaitLimitNs = 4000000000ull;
// the look-back's limit, adjustable from the host (dmb_dev_set_lookback_limit_ns): tests set it to 0 to see the error path
// end in a reported flag and a usable context
__device__ unsigned long long g_lookback_limit_ns = kWaitLimitNs;
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
  // try_wait suspends the thread in hardware until the phase completes or the time hint (ns) runs out:
  // with the default (short) limit the retry loop alone took a third of the kernel's issue slots
  uint32_t done;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(done) : "r"(mbar), "r"(parity), "r"(20000u) : "memory");
  if (done) return;
  unsigned long long t0 = 0;
  for (uint32_t spins = 1;; ++spins) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(mbar), "r"(parity), "r"(20000u) : "memory");
    if (done) return;
    if ((spins & 63u) == 0u) {
      const unsigned long long now = global_ns();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 3ull * kWaitLimitNs) __trap();
    }
  }
}
__device__ __forceinline__ void mbar_arrive(uint32_t mbar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(mbar) : "memory"); }
__device__ __forceinline__ void bulk_load(uint32_t dst_smem, const void *src, uint32_t bytes, uint32_t mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst_smem), "l"(__cvta_generic_to_global(src)), "r"(bytes), "r"(mbar) : "memory");
}
__device__ __forceinline__ void bulk_store(void *dst, uint32_t src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               ::"l"(__cvta_generic_to_global(dst)), "r"(src_smem), "r"(bytes) : "memory");
}
// byte i of every 16-byte chunk is copied iff bit i of `mask` is set (PTX ISA 8.6, sm_100)
__device__ __forceinline__ void bulk_store_masked(void *dst, uint32_t src_smem, uint32_t bytes, uint32_t mask) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.cp_mask [%0], [%1], %2, %3;"
               ::"l"(__cvta_generic_to_global(dst)), "r"(src_smem), "r"(bytes), "h"((unsigned short)mask) : "memory");
}
__device__ __forceinline__ void bulk_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_store_drain() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// named barriers: `sync` waits, `arrive` only signals; n = arriving + waiting threads
__device__ __forceinline__ void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }
// role <-> role hand-offs inside a CTA are NAMED BARRIERS (bar.arrive / bar.sync): a warp that waits on one is parked by
// the hardware and issues nothing.  (As mbarrier.try_wait loops they took a quarter of the kernel's issue slots away
// from the warps that were packing.)  F: worker warp 0 -> L, "tile k is scanned and its aggregate is out" (64 threads);
// B: L -> workers, "tile k's base is resolved" (workers + 32).  Each comes as an alternating pair: the producer of
// phase k + 2 cannot reach its arrive before the consumer has left phase k (see the order of front / back below).
enum { kBarWorkers = 1, kBarBase = 3, kBarPacked = 4, kBarF0 = 5, kBarF1 = 6, kBarB0 = 7, kBarB1 = 8 };

// bytes [b0, b1) of `v` into the word at `w` (the other bytes belong to neighbouring threads)
__device__ __forceinline__ void store_bytes(uint32_t *w, uint32_t v, uint32_t b0, uint32_t b1) {
  uint8_t *p = reinterpret_cast<uint8_t *>(w);
#pragma unroll
  for (uint32_t k = 0; k < 4; ++k)
    if (k >= b0 && k < b1) p[k] = (uint8_t)(v >> (8u * k));
}

// low `n` bytes set, n in 0..3
__device__ __forceinline__ uint32_t low_bytes3(uint32_t n) { return (1u << (8u * n)) - 1u; }

// bytes a row contributes: 0 for NULL / past the chunk / an unusable pointer (flagged); P and the
// workers must agree on this, it defines the tile totals
template <bool HEAP>
__device__ __forceinline__ uint32_t row_bytes(const dmb_string_job &job, uint32_t x, uint32_t z, uint32_t w, bool live, int &flags,
                                              uint32_t &lo16, uint32_t &hi16) {
  uint32_t l = live ? x : 0u;
  lo16 = 0xffffffffu;
  hi16 = 0u;
  if (l > 12u) {
    const uint64_t p = ((uint64_t)w << 32) | (uint64_t)z;
    const uint64_t rel = p - job.heap_host_base;
    if (l >= kMaxRowBytes) { flags |= 4; l = 0; }
    else if (!HEAP || p < job.heap_host_base || rel + l > job.heap_len) { flags |= 2; l = 0; }  // !HEAP: the column registered no heap
    else { lo16 = (uint32_t)(rel >> 4); hi16 = (uint32_t)((rel + l + 15u) >> 4); }
  }
  return l;
}

// per-tile state a worker thread carries from front() to back()
template <int R>
struct RowState {
  uint32_t len[R];            // row_bytes()
  uint32_t y[R], z[R], w[R];  // string_t words 1..3: inlined payload, or prefix + pointer
  uint32_t my_off;            // tile-local offset of the thread's first row
};

template <bool LARGE, int R, bool HEAP, bool UNIFY = true>
__global__ void __launch_bounds__(pack_warps(HEAP) * 32 + 64, HEAP ? 3 : 2)
string_pack_kernel(dmb_string_job job, BatchView b, unsigned long long *scratch, int64_t ntiles,
                   uint32_t ostage_bytes, uint32_t hstage_bytes) {
  static_assert(R == 2 || R == 4, "rows per worker thread");
  constexpr int NW = pack_warps(HEAP);
  constexpr int kWT = NW * 32;             // worker threads
  constexpr int kRows = kWT * R;
  constexpr int kTilesPerChunk = kVec / kRows;
  constexpr uint32_t kSBytes = (uint32_t)kRows * 16u;
  constexpr int kWL = kWT + 32;            // workers + T
  extern __shared__ __align__(128) uint8_t dsm[];
  PackTail &pt = *reinterpret_cast<PackTail *>(dsm);
  uint8_t *sbuf = dsm + kPackTail;                   // S[2]: string_t tiles
  uint8_t *ostage = sbuf + 2u * kSBytes;             // O: output stage
  uint8_t *hbuf = ostage + ostage_bytes;             // H[2]: heap spans (each hstage_bytes + 16)
  const uint32_t hstride = hstage_bytes + 16u;
  unsigned long long *status = scratch + 2;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  if (tid == 0) {
    mbar_init(smem_u32(&pt.mbar_s[0]), 1);
    mbar_init(smem_u32(&pt.mbar_s[1]), 1);
    mbar_init(smem_u32(&pt.mbar_h[0]), 1);
    mbar_init(smem_u32(&pt.mbar_h[1]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp == NW) {
    // ------------------------------------------------------------ P: tickets, string_t bulk loads ...
    // claim tile k: ticket + chunk metadata, bulk load of its string_t (+ validity words) into S[k&1]
    // claim tile k: ticket + chunk metadata.  Done one tile EARLIER than the bulk load of its string_t (which has to wait for
    // the S buffer): the ticket atomic and the dependent metadata loads (two L2 round trips) are then off the path between
    // "S is free" and "the load is in flight" -- with two CTAs of 18 warps per SM (the heap-less form) the workers had
    // spent 11 % of their stall samples waiting for S
    auto claim = [&](int k) {
      TileMeta &m = pt.meta[k & (kMetaRing - 1)];
      long long tile = (long long)atomicAdd(scratch, 1ull);
      if (tile >= ntiles) tile = -1;
      m.tile = tile;
      if (tile < 0) return;
      const int64_t c = tile / kTilesPerChunk;
      const int r_begin = (int)(tile % kTilesPerChunk) * kRows;
      const int count = (int)__ldg(b.counts + c);
      const dmb_vec_desc vd = job.vecs[c];
      int nrows_tile = count - r_begin;
      nrows_tile = nrows_tile < 0 ? 0 : (nrows_tile > kRows ? kRows : nrows_tile);
      m.out_row0 = __ldg(b.row_off + c) + r_begin;
      m.nrows = nrows_tile;
      m.has_mask = vd.val_off >= 0;
      m.src = reinterpret_cast<const uint8_t *>(job.in) + vd.data_off + (uint64_t)r_begin * 16u;
      m.val = vd.val_off >= 0 ? job.in_validity + vd.val_off + (r_begin >> 6) : nullptr;
    };
    // bulk load of tile k's string_t (+ validity words) into S[k&1]
    auto load = [&](int k) {
      const TileMeta &m = pt.meta[k & (kMetaRing - 1)];
      const int slot = k & 1;
      const uint32_t mb = smem_u32(&pt.mbar_s[slot]);
      if (m.tile < 0) {  // no tile: complete the phase all the same, the others learn it from meta
        mbar_arrive(mb);
        return;
      }
      // a DuckDB vector always has STANDARD_VECTOR_SIZE entries of storage: the whole tile is readable
      mbar_expect_tx(mb, kSBytes + (m.val ? (uint32_t)kRows / 8u : 0u));
      bulk_load(smem_u32(sbuf + (uint32_t)slot * kSBytes), m.src, kSBytes, mb);
      if (m.val) bulk_load(smem_u32(&pt.vmask[slot][0]), m.val, (uint32_t)kRows / 8u, mb);
    };
    // ... and T: when the workers have packed a tile, send the stage to out_data with bulk stores and
    // hand the stage back.  Both jobs are triggered by the end of a worker iteration.
    // Tickets run three tiles ahead, loads two (A/B in one run, 60 M rows: heap-less columns 0.270 -> 0.254 ms, all-pointer columns
    // 0.772 -> 0.741 ms, l_comment / l_shipinstruct shapes unchanged within the box-to-box noise of +-1 %)
    if (lane == 0) {
      claim(0);
      claim(1);  // (also past the end: the workers must meet a tile that says so)
      claim(2);
      load(0);
      load(1);
    }
    bar_arrive(kBarBase, kWL);  // the stage is free
    for (int j = 0;; ++j) {
      bar_sync(kBarPacked, kWL);  // the workers have finished iteration j: tile j-1 packed, tile j scanned
      bool more = false;
      if (lane == 0) {
        if (j > 0) {
          const TileMeta &mp = pt.meta[(j - 1) & (kMetaRing - 1)];
          const uint64_t base = pt.base[(j - 1) & (kMetaRing - 1)];
          const uint32_t total = mp.total;
          if (!LARGE && base + total > 0x7fffffffull) atomicOr(scratch + 1, (unsigned long long)kErrOffsetOverflow);
          if (mp.tile == ntiles - 1) {
            if (LARGE) reinterpret_cast<long long *>(job.out_offsets)[b.nrows] = (long long)(base + total);
            else reinterpret_cast<int32_t *>(job.out_offsets)[b.nrows] = (int32_t)(base + total);
            if (job.total_bytes) *job.total_bytes = base + total;
          }
          const bool over_cap = job.out_data_cap && base + total > job.out_data_cap;
          if (over_cap) atomicOr(scratch + 1, (unsigned long long)kErrDataCap);
          if (total && mp.staged && !over_cap) {
            // stage byte q is global byte gbase + q
            const uint32_t mis = (uint32_t)(base & 15ull);
            uint8_t *gbase = job.out_data + (base - mis);
            const uint32_t end = mis + total;
            const uint32_t q0 = mis ? 16u : 0u, q1 = end & ~15u;
            const uint32_t so = smem_u32(ostage);
            if (mis) bulk_store_masked(gbase, so, 16u, (0xffffu << mis) & (end < 16u ? (1u << end) - 1u : 0xffffu));
            if (q1 > q0) bulk_store(gbase + q0, so + q0, q1 - q0);
            if ((end & 15u) && q1 >= q0) bulk_store_masked(gbase + q1, so + q1, 16u, (1u << (end & 15u)) - 1u);
            bulk_store_commit();
            bulk_store_drain();  // the stage is free again once the copy engine has read it
          }
        }
        more = pt.meta[j & (kMetaRing - 1)].tile >= 0;
      }
      more = __shfl_sync(0xffffffffu, more, 0);
      if (!more) break;
      bar_arrive(kBarBase, kWL);  // the stage is free
      if (lane == 0) {
        // S[j&1] held tile j: the workers have scanned it (barrier above)
        load(j + 2);
        claim(j + 3);
      }
      __syncwarp();
    }
    return;
  }

  if (warp == NW + 1) {
    // ------------------------------------------------------------ L: look-back
    for (int k = 0;; ++k) {
      const TileMeta &m = pt.meta[k & (kMetaRing - 1)];
      // a lazy look-back is a short one: by the time the workers have scanned tile k its predecessors' aggregates (often
      // their prefixes) are out, and the result is not needed before tile k-1 is packed
      bar_sync(kBarF0 + (k & 1), 64);  // tile k is scanned, its aggregate is published (or there is no tile k)
      const long long tile = m.tile;
      if (tile < 0) break;
      const uint64_t base = lookback_groups(status, status + ntiles, status + ntiles + ((ntiles + 31) >> 5), tile, lane, status - 1, (unsigned long long)kErrTimeout, g_lookback_limit_ns);
      if (lane == 0) {
        if (tile > 0) atomicExch(status + tile, kFlagPrefix | ((base + m.total) & kValueMask));
        // the last tile of a group of 32 also publishes the group's inclusive prefix, in an array of its own (32 groups = 256 bytes)
        if ((tile & 31) == 31) atomicExch(status + ntiles + ((ntiles + 31) >> 5) + (tile >> 5), kFlagPrefix | ((base + m.total) & kValueMask));
        pt.base[k & (kMetaRing - 1)] = base;
      }
      __syncwarp();
      bar_arrive(kBarB0 + (k & 1), kWT + 32);  // the workers may place tile k
    }
    return;
  }

  // -------------------------------------------------------------- W, columns without a heap: the lean form
  // Every string is inlined (<= 12 bytes, a pointer entry is an error), so the workers need none of the span / run / funnel
  // machinery below.  Rows are owned STRIPED (stripe k of warp w = tile rows w*32*R + 32*k + lane): the string_t leave S
  // with conflict-free 16-byte loads, two stripes' lengths share one 32-bit scan (a stripe sums to <= 384 < 2^16), offsets
  // leave as coalesced 4-byte stores, and the bytes are placed one by one straight at their FINAL alignment in the stage (the
  // base is known by then), which P sends out with bulk stores: no copy-out pass.  Same roles, barriers and look-back as
  // the general form.  (A one-CTA-per-tile kernel does the same work in ~2 warp-instructions per row but sits on its
  // dependent chain: ticket -> metadata -> string_t -> scan -> look-back -> stores; here P and L hide that chain.)
  if constexpr (!HEAP) {
    uint32_t c_len[R], c_y[R], c_z[R], c_w[R], c_off[R], c_lmax = 0u;
    bool cur_valid = false;
    const int row0 = warp * (32 * R) + lane;
    for (int j = 0;; ++j) {
      if (j > 0 && !cur_valid) break;
      const int slot = j & 1;
      mbar_wait(smem_u32(&pt.mbar_s[slot]), (uint32_t)(j >> 1) & 1u);
      TileMeta &mj = pt.meta[j & (kMetaRing - 1)];
      const bool nxt_valid = mj.tile >= 0;
      uint32_t n_len[R], n_y[R], n_z[R], n_w[R], n_off[R], n_lmax = 0u;
      if (nxt_valid) {
        const int nrows = mj.nrows;
        const bool has_mask = mj.has_mask != 0;
        const uint4 *s = reinterpret_cast<const uint4 *>(sbuf + (uint32_t)slot * kSBytes);
        int bad = 0;
#pragma unroll
        for (int k = 0; k < R; ++k) {
          const int row = row0 + 32 * k;
          const uint4 e = s[row];
          bool live = row < nrows;
          if (has_mask) live = live && ((pt.vmask[slot][row >> 6] >> (row & 63)) & 1ull);
          uint32_t l = live ? e.x : 0u;
          if (l > 12u) { bad = 1; l = 0u; }  // a pointer string, but the column registered no heap
          n_len[k] = l; n_y[k] = e.y; n_z[k] = e.z; n_w[k] = e.w;
          n_lmax = n_lmax > l ? n_lmax : l;
        }
        uint32_t carry = 0u;
#pragma unroll
        for (int k = 0; k < R; k += 2) {
          const uint32_t both = n_len[k] | (n_len[k + 1] << 16);
          uint32_t incl = both;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const uint32_t n = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += n;
          }
          const uint32_t tot = __shfl_sync(0xffffffffu, incl, 31);
          const uint32_t excl = incl - both;
          n_off[k] = carry + (excl & 0xffffu);
          carry += tot & 0xffffu;
          n_off[k + 1] = carry + (excl >> 16);
          carry += tot >> 16;
        }
        PackPartials &pp = pt.part[slot];
        if (lane == 0) pp.warp_sum[warp] = carry;
        if (bad) atomicOr(scratch + 1, (unsigned long long)kErrHeapRange);
        n_lmax = __reduce_max_sync(0xffffffffu, n_lmax);
        bar_sync(kBarWorkers, kWT);
        // the NW warp sums: one load per lane + a shuffle scan (as NW loads + selects per thread this was 11 % of the kernel)
        uint32_t wincl = lane < NW ? pp.warp_sum[lane] : 0u;
        const uint32_t wown = wincl;
#pragma unroll
        for (int d = 1; d < NW; d <<= 1) {
          const uint32_t n = __shfl_up_sync(0xffffffffu, wincl, d);
          if (lane >= d) wincl += n;
        }
        const uint32_t warp_excl = __shfl_sync(0xffffffffu, wincl - wown, warp);
        const uint32_t total = __shfl_sync(0xffffffffu, wincl, NW - 1);
#pragma unroll
        for (int k = 0; k < R; ++k) n_off[k] += warp_excl;
        if (tid == 0) {
          mj.total = total;
          mj.hmin = 0u;
          mj.hbytes = 0u;
          mj.staged = 1;
          atomicExch(status + mj.tile, (mj.tile == 0 ? kFlagPrefix : kFlagAggregate) | (uint64_t)total);
          atomicAdd(status + ntiles + (mj.tile >> 5), kGroupOne | (unsigned long long)total);
        }
      }
      if (warp == 0) {  // L: tile j's look-back is due (or: there is no tile j)
        __syncwarp();
        bar_arrive(kBarF0 + (j & 1), 64);
      }
      // ---- back(tile j-1)
      uint64_t base = 0;
      if (cur_valid) {
        bar_sync(kBarB0 + ((j - 1) & 1), kWT + 32);  // L has resolved tile j-1
        base = pt.base[(j - 1) & (kMetaRing - 1)];
        const TileMeta &mc = pt.meta[(j - 1) & (kMetaRing - 1)];
        const int nrows = mc.nrows;
        long long *oo64 = reinterpret_cast<long long *>(job.out_offsets) + (mc.out_row0 + row0);
        int32_t *oo32 = reinterpret_cast<int32_t *>(job.out_offsets) + (mc.out_row0 + row0);
#pragma unroll
        for (int k = 0; k < R; ++k) {
          if (row0 + 32 * k < nrows) {
            if (LARGE) __stcs(oo64 + 32 * k, (long long)(base + c_off[k]));
            else __stcs(oo32 + 32 * k, (int32_t)((uint32_t)base + c_off[k]));
          }
        }
      }
      bar_sync(kBarBase, kWL);  // the stage is free (P has sent tile j-2)
      if (cur_valid) {
        const uint32_t mis = (uint32_t)(base & 15ull);
#pragma unroll
        for (int k = 0; k < R; ++k) c_off[k] += mis;  // (the offsets have left: from here on, the stage byte of the row's first byte)
#pragma unroll
        for (int i = 0; i < 12; ++i) {
          if ((uint32_t)i >= c_lmax) break;  // warp-uniform: one test per byte position up to the warp's longest string, then out
#pragma unroll
          for (int k = 0; k < R; ++k) {
            const uint32_t wsel = i < 4 ? c_y[k] : (i < 8 ? c_z[k] : c_w[k]);
            if ((uint32_t)i < c_len[k]) ostage[c_off[k] + i] = (uint8_t)(wsel >> (8 * (i & 3)));
          }
        }
        fence_proxy_async_smem();
      }
      bar_arrive(kBarPacked, kWL);
#pragma unroll
      for (int k = 0; k < R; ++k) { c_len[k] = n_len[k]; c_y[k] = n_y[k]; c_z[k] = n_z[k]; c_w[k] = n_w[k]; c_off[k] = n_off[k]; }
      c_lmax = n_lmax;
      cur_valid = nxt_valid;
    }
    return;
  }

  // -------------------------------------------------------------- W: scan (front) and pack (back)
  RowState<R> cur, nxt;
  bool cur_valid = false;
  uint32_t phase_h0 = 0, phase_h1 = 0;
  for (int j = 0;; ++j) {
    if (j > 0 && !cur_valid) break;  // tickets are monotonic: no tile j-1, no tile j
    // ---- front(tile j)
    const int slot = j & 1;
    mbar_wait(smem_u32(&pt.mbar_s[slot]), (uint32_t)(j >> 1) & 1u);  // P has claimed tile j (or found none)
    const bool nxt_valid = pt.meta[j & (kMetaRing - 1)].tile >= 0;
    if (nxt_valid) {
      const int nrows = pt.meta[j & (kMetaRing - 1)].nrows;
      const uint4 *s = reinterpret_cast<const uint4 *>(sbuf + (uint32_t)slot * kSBytes) + tid * R;
      uint64_t vword = ~0ull;
      if (pt.meta[j & (kMetaRing - 1)].has_mask) vword = pt.vmask[slot][(tid * R) >> 6] >> ((tid * R) & 63);
      int flags = 0;  // 2: bad heap pointer  4: oversized row
      uint32_t tsum = 0u, hmin = 0xffffffffu, hmax = 0u;
      uint4 ent[R];
      // a thread's R string_t are 16 R consecutive bytes: read in row order, the eight lanes of a quarter warp would hit
      // only 8 / R of the eight 16-byte bank groups.  Lane i starts at row (i / (8 / R)) mod R instead and the rows are
      // rotated back in registers.
      const int rot = R == 4 ? (lane >> 1) & 3 : (lane >> 2) & 1;
      uint4 t[R];
#pragma unroll
      for (int k = 0; k < R; ++k) t[k] = s[(k + rot) & (R - 1)];
      auto sel = [](bool c, const uint4 &a, const uint4 &b) { return make_uint4(c ? a.x : b.x, c ? a.y : b.y, c ? a.z : b.z, c ? a.w : b.w); };
      if (R == 2) {
        ent[0] = sel(rot != 0, t[1 % R], t[0]);
        ent[1 % R] = sel(rot != 0, t[0], t[1 % R]);
      } else {
        uint4 u[R];
#pragma unroll
        for (int k = 0; k < R; ++k) u[k] = sel((rot & 1) != 0, t[(k + 3) & (R - 1)], t[k]);
#pragma unroll
        for (int k = 0; k < R; ++k) ent[k] = sel((rot & 2) != 0, u[(k + 2) & (R - 1)], u[k]);
      }
#pragma unroll
      for (int k = 0; k < R; ++k) {
        const uint4 e = ent[k];
        uint32_t lo16, hi16;
        const uint32_t l = row_bytes<HEAP>(job, e.x, e.z, e.w, ((vword >> k) & 1ull) && tid * R + k < nrows, flags, lo16, hi16);
        nxt.len[k] = l; nxt.y[k] = e.y; nxt.z[k] = e.z; nxt.w[k] = e.w;
        tsum += l;
        hmin = hmin < lo16 ? hmin : lo16;
        hmax = hmax > hi16 ? hmax : hi16;
      }
      if (flags) atomicOr(scratch + 1, (unsigned long long)(((flags & 2) ? kErrHeapRange : 0) | ((flags & 4) ? kErrTileTooBig : 0)));
      uint32_t incl = tsum;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t n = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += n;
      }
      PackPartials &pp = pt.part[slot];
      if (HEAP) {
        hmin = __reduce_min_sync(0xffffffffu, hmin);
        hmax = __reduce_max_sync(0xffffffffu, hmax);
        if (lane == 0) { pp.warp_hmin[warp] = hmin; pp.warp_hmax[warp] = hmax; }
      }
      if (lane == 31) pp.warp_sum[warp] = incl;
      if (tid == 0) pp.not_one_run = 0u;
      bar_sync(kBarWorkers, kWT);  // (every warp has also finished packing tile j-2: H[slot] is free)
      uint32_t warp_excl = 0;
#pragma unroll
      for (int w = 0; w < NW; ++w) warp_excl += w < warp ? pp.warp_sum[w] : 0u;
      nxt.my_off = warp_excl + incl - tsum;
      if (HEAP) {
        // is the tile one run?  (every non-empty row a pointer row whose bytes follow its predecessor's in the heap)
        uint32_t cmin = 0xffffffffu, cmax = 0u, o = nxt.my_off;
#pragma unroll
        for (int k = 0; k < R; ++k) {
          const uint32_t l = nxt.len[k];
          if (l != 0u) {
            const uint32_t c = nxt.z[k] - o;
            cmin = l > 12u ? (cmin < c ? cmin : c) : 0u;
            cmax = l > 12u ? (cmax > c ? cmax : c) : 0xffffffffu;  // an inlined row: never one run
          }
          o += l;
        }
        // (read after the next barrier, in back(); most tiles of a mixed column are settled by the first test)
        if (__any_sync(0xffffffffu, cmin == 0u && cmax == 0xffffffffu)) {
          if (lane == 0) pp.not_one_run = 1u;
        } else {
          cmin = __reduce_min_sync(0xffffffffu, cmin);
          cmax = __reduce_max_sync(0xffffffffu, cmax);
          if (lane == 0) { pp.warp_cmin[warp] = cmin; pp.warp_cmax[warp] = cmax; }
        }
      }
      if (tid == 0) {
        // the tile's heap span [hmin, hmax) -> H[slot], one bulk copy
        TileMeta &m = pt.meta[j & (kMetaRing - 1)];
        uint32_t total = 0;
        hmin = 0xffffffffu;
        hmax = 0u;
#pragma unroll
        for (int w = 0; w < NW; ++w) {
          total += pp.warp_sum[w];
          if (HEAP) {
            hmin = hmin < pp.warp_hmin[w] ? hmin : pp.warp_hmin[w];
            hmax = hmax > pp.warp_hmax[w] ? hmax : pp.warp_hmax[w];
          }
        }
        const uint32_t hbytes = hmax > hmin ? (hmax - hmin) << 4 : 0u;
        const bool staged = !HEAP || (hbytes <= hstage_bytes && total + 48u <= ostage_bytes &&
                                       (hbytes == 0u || (reinterpret_cast<uintptr_t>(job.heap_dev) & 15u) == 0u));
        m.hmin = hmin;
        m.hbytes = hbytes;
        m.staged = staged;
        // the tile's aggregate goes out here (a separate warp that summed the lengths as soon as the string_t landed, one
        // iteration earlier, made the look-backs behind it a little shorter but cost 3 % of the kernel: every row was read twice)
        m.total = total;
        atomicExch(status + m.tile, (m.tile == 0 ? kFlagPrefix : kFlagAggregate) | (uint64_t)total);
        atomicAdd(status + ntiles + (m.tile >> 5), kGroupOne | (unsigned long long)total);  // (no return value: a reduction at L2)
        if (HEAP && staged && hbytes) {
          const uint32_t mb = smem_u32(&pt.mbar_h[slot]);
          mbar_expect_tx(mb, hbytes);
          bulk_load(smem_u32(hbuf + (uint32_t)slot * hstride), job.heap_dev + ((uint64_t)hmin << 4), hbytes, mb);
        }
      }
    }
    if (warp == 0) {  // L: tile j's look-back is due (or: there is no tile j)
      __syncwarp();
      bar_arrive(kBarF0 + (j & 1), 64);
    }

    // ---- back(tile j-1)
    uint64_t base = 0;
    if (cur_valid) {
      bar_sync(kBarB0 + ((j - 1) & 1), kWT + 32);  // L has resolved tile j-1
      base = pt.base[(j - 1) & (kMetaRing - 1)];
    }
    if (cur_valid) {
      const TileMeta &mc = pt.meta[(j - 1) & (kMetaRing - 1)];
      const int nrows = mc.nrows;
      // offsets: R consecutive values per thread
      {
        const int i0 = tid * R;
        if (LARGE) {
          long long *oo = reinterpret_cast<long long *>(job.out_offsets) + mc.out_row0 + i0;
          uint64_t o = base + cur.my_off;
          if (i0 + R <= nrows && (reinterpret_cast<uintptr_t>(oo) & 15u) == 0u) {
#pragma unroll
            for (int k = 0; k < R; k += 2) {
              const uint64_t o1 = o + cur.len[k];
              __stcs(reinterpret_cast<longlong2 *>(oo + k), make_longlong2((long long)o, (long long)o1));
              o = o1 + cur.len[k + 1];
            }
          } else {
#pragma unroll
            for (int k = 0; k < R; ++k) {
              if (i0 + k < nrows) __stcs(oo + k, (long long)o);
              o += cur.len[k];
            }
          }
        } else {
          int32_t *oo = reinterpret_cast<int32_t *>(job.out_offsets) + mc.out_row0 + i0;
          uint32_t o = (uint32_t)base + cur.my_off;
          constexpr int kV = R == 2 ? 2 : 4;  // values per vector store
          if (i0 + R <= nrows && (reinterpret_cast<uintptr_t>(oo) & (4u * kV - 1u)) == 0u) {
            if (R == 2) {
              __stcs(reinterpret_cast<int2 *>(oo), make_int2((int)o, (int)(o + cur.len[0])));
            } else {
#pragma unroll
              for (int k = 0; k < R; k += 4) {
                const uint32_t o1 = o + cur.len[k], o2 = o1 + cur.len[k + 1], o3 = o2 + cur.len[k + 2];
                __stcs(reinterpret_cast<int4 *>(oo + k), make_int4((int)o, (int)o1, (int)o2, (int)o3));
                o = o3 + cur.len[k + 3];
              }
            }
          } else {
#pragma unroll
            for (int k = 0; k < R; ++k) {
              if (i0 + k < nrows) __stcs(oo + k, (int32_t)o);
              o += cur.len[k];
            }
          }
        }
      }
    }
    bar_sync(kBarBase, kWL);  // the stage is free (T has sent tile j-2)
    if (cur_valid) {
      const TileMeta &mc = pt.meta[(j - 1) & (kMetaRing - 1)];
      const uint32_t mis = (uint32_t)(base & 15ull);
      const uint32_t total = mc.total;
      if (total != 0u && mc.staged) {
        // pack: this thread's rows as one byte stream starting at stage byte mis + my_off
        const int hslot = (j - 1) & 1;
        if (HEAP && mc.hbytes) {
          uint32_t &ph = hslot ? phase_h1 : phase_h0;
          mbar_wait(smem_u32(&pt.mbar_h[hslot]), ph);
          ph ^= 1u;
        }
        uint32_t *ow = reinterpret_cast<uint32_t *>(ostage);
        const uint32_t *hw = reinterpret_cast<const uint32_t *>(hbuf + (uint32_t)hslot * hstride);
        const uint32_t hbase = (mc.hmin << 4) + (uint32_t)job.heap_host_base;  // low 32 bits of the span's host address
        bool one_run = false;
        uint32_t run_c = 0;
        if (HEAP && mc.hbytes && pt.part[hslot].not_one_run == 0u) {
          const PackPartials &pq = pt.part[hslot];
          uint32_t cmin = 0xffffffffu, cmax = 0u;
#pragma unroll
          for (int w = 0; w < NW; ++w) {
            cmin = cmin < pq.warp_cmin[w] ? cmin : pq.warp_cmin[w];
            cmax = cmax > pq.warp_cmax[w] ? cmax : pq.warp_cmax[w];
          }
          one_run = cmin == cmax;
          run_c = cmin;
        }
        if (one_run) {
          // the tile's output is one contiguous piece of the staged span, shifted: out word w = span bytes
          // 4w + d .. 4w + d + 3.  Consecutive lanes, consecutive words: conflict free, no row logic;
          // the bytes outside [mis, mis + total) of the first / last word are masked off by the bulk store
          const uint32_t d = (run_c - hbase) + 64u - mis;  // > 0
          const uint32_t sh = 8u * (d & 3u);
          const uint32_t *s = hw + (d >> 2) - 16;
          const uint32_t wend = (mis + total + 3u) >> 2;
#pragma unroll 2
          for (uint32_t w = (mis >> 2) + (uint32_t)tid; w < wend; w += (uint32_t)kWT) ow[w] = __funnelshift_r(s[w], s[w + 1], sh);
          fence_proxy_async_smem();
        } else {
        const uint32_t pos = mis + cur.my_off;
        uint32_t wp = pos >> 2, fill = pos & 3u, acc = 0u;
        const uint32_t head = fill;                          // bytes of the first word that belong to earlier threads
        const uint32_t shared_wp = fill ? wp : 0xffffffffu;  // a first word that earlier threads also write
        if constexpr (UNIFY) {
        // One code path for every row: an inlined row first drops its 12 payload bytes into the thread's own 12-byte slot of a
        // scratch area behind H (3-word stride: conflict free) and is then copied like a pointer row whose bytes start there.
        // (As two paths, a warp paid for both at every row slot as soon as one lane differed from the others.)
        uint32_t *scr = reinterpret_cast<uint32_t *>(hbuf + 2u * hstride) + tid * 3;
        const uint32_t scr_rel = (uint32_t)(reinterpret_cast<const uint8_t *>(scr) - reinterpret_cast<const uint8_t *>(hw));
#pragma unroll
        for (int k = 0; k < R; ++k) {
          const uint32_t l = cur.len[k];
          if (l == 0u) continue;
          const uint32_t n = fill + l, nw = n >> 2;
          uint32_t srel = cur.z[k] - hbase;  // the row's first byte, relative to hw
          if (l <= 12u) {
            scr[0] = cur.y[k];
            scr[1] = cur.z[k];
            scr[2] = cur.w[k];
            srel = scr_rel;
          }
          // output word m of the row holds source bytes qp-4+4m .. +3
          const uint32_t qp = srel + 4u - fill;
          const uint32_t sq = 8u * (qp & 3u);
          const uint32_t *sp = hw + (qp >> 2);
          uint32_t prev = sp[0];
          const uint32_t x0 = (__funnelshift_r(sp[-1], prev, sq) & ~low_bytes3(fill)) | acc;
          if (nw == 0u) {
            acc = x0 & low_bytes3(n);  // a short inlined row that does not complete the word
          } else {
            if (wp == shared_wp) store_bytes(ow + wp, x0, head, 4u); else ow[wp] = x0;
            // the whole words after the first one: four per iteration, the loads of a group before its stores (the compiler
            // may not move a shared-memory load over a shared-memory store), pointers bumped instead of indices recomputed
            sp += 1;
            uint32_t *op = ow + wp + 1;
            uint32_t left = nw - 1u;
#pragma unroll 1
            for (; left >= 4u; left -= 4u) {
              const uint32_t a0 = sp[0], a1 = sp[1], a2 = sp[2], a3 = sp[3];
              op[0] = __funnelshift_r(prev, a0, sq);
              op[1] = __funnelshift_r(a0, a1, sq);
              op[2] = __funnelshift_r(a1, a2, sq);
              op[3] = __funnelshift_r(a2, a3, sq);
              prev = a3;
              sp += 4;
              op += 4;
            }
            if (left & 2u) {
              const uint32_t a0 = sp[0], a1 = sp[1];
              op[0] = __funnelshift_r(prev, a0, sq);
              op[1] = __funnelshift_r(a0, a1, sq);
              prev = a1;
              sp += 2;
              op += 2;
            }
            if (left & 1u) {
              const uint32_t a0 = sp[0];
              op[0] = __funnelshift_r(prev, a0, sq);
              prev = a0;
              sp += 1;
            }
            acc = (n & 3u) ? (__funnelshift_r(prev, sp[0], sq) & low_bytes3(n & 3u)) : 0u;
          }
          wp += nw;
          fill = n & 3u;
        }
        } else {
#pragma unroll
        for (int k = 0; k < R; ++k) {
          const uint32_t l = cur.len[k];
          if (l == 0u) continue;
          const uint32_t n = fill + l, nw = n >> 2;
          if (l <= 12u) {
            // inlined: payload in registers; bytes past the length are dropped when the last word is kept
            const uint32_t p0 = cur.y[k], p1 = cur.z[k], p2 = cur.w[k];
            const uint32_t s = 8u * fill;
            const uint32_t x0 = acc | (p0 << s);
            const uint32_t x1 = __funnelshift_l(p0, p1, s);
            const uint32_t x2 = __funnelshift_l(p1, p2, s);
            const uint32_t x3 = __funnelshift_l(p2, 0u, s);
            if (nw >= 1u) {
              if (wp == shared_wp) store_bytes(ow + wp, x0, head, 4u); else ow[wp] = x0;
            }
            if (nw >= 2u) ow[wp + 1] = x1;
            if (nw >= 3u) ow[wp + 2] = x2;
            // (nw <= 3; as a chain of equality tests this became a jump table)
            acc = ((nw & 2u) ? ((nw & 1u) ? x3 : x2) : ((nw & 1u) ? x1 : x0)) & low_bytes3(n & 3u);
          } else if (HEAP) {
            // pointer: the staged span.  Output word m of the row holds source bytes qp-4+4m .. +3
            const uint32_t qp = (cur.z[k] - hbase) + 4u - fill;
            const uint32_t sq = 8u * (qp & 3u);
            const uint32_t *s = hw + (qp >> 2);
            uint32_t prev = s[-1], nx = s[0];
            const uint32_t x0 = (__funnelshift_r(prev, nx, sq) & ~low_bytes3(fill)) | acc;
            if (wp == shared_wp) store_bytes(ow + wp, x0, head, 4u); else ow[wp] = x0;  // l > 12: the word always completes
            prev = nx;
            // the whole words after the first one: four per iteration, the loads of a group before its stores (the compiler
            // may not move a shared-memory load over a shared-memory store), pointers bumped instead of indices recomputed:
            // 17 instructions per four words where a plain word-by-word loop took 13 per two
            const uint32_t *sp = s + 1;
            uint32_t *op = ow + wp + 1;
            uint32_t left = nw - 1u;
#pragma unroll 1
            for (; left >= 4u; left -= 4u) {
              const uint32_t a0 = sp[0], a1 = sp[1], a2 = sp[2], a3 = sp[3];
              op[0] = __funnelshift_r(prev, a0, sq);
              op[1] = __funnelshift_r(a0, a1, sq);
              op[2] = __funnelshift_r(a1, a2, sq);
              op[3] = __funnelshift_r(a2, a3, sq);
              prev = a3;
              sp += 4;
              op += 4;
            }
            if (left & 2u) {
              const uint32_t a0 = sp[0], a1 = sp[1];
              op[0] = __funnelshift_r(prev, a0, sq);
              op[1] = __funnelshift_r(a0, a1, sq);
              prev = a1;
              sp += 2;
              op += 2;
            }
            if (left & 1u) {
              const uint32_t a0 = sp[0];
              op[0] = __funnelshift_r(prev, a0, sq);
              prev = a0;
              sp += 1;
            }
            acc = (n & 3u) ? (__funnelshift_r(prev, sp[0], sq) & low_bytes3(n & 3u)) : 0u;
          }
          wp += nw;
          fill = n & 3u;
        }
        }
        if (fill) store_bytes(ow + wp, acc, wp == shared_wp ? head : 0u, fill);  // last word: the next thread owns its other bytes
        fence_proxy_async_smem();
        }
      } else if (HEAP && total != 0u && !(job.out_data_cap && base + total > job.out_data_cap)) {
        // not staged: one warp per row, one byte per lane, heap -> out_data
        uint8_t *out = job.out_data + base;
        uint32_t offk[R];
        offk[0] = cur.my_off;
#pragma unroll
        for (int k = 1; k < R; ++k) offk[k] = offk[k - 1] + cur.len[k - 1];
        auto pick = [&](const uint32_t (&a)[R], int k) {
          uint32_t v = a[0];
#pragma unroll
          for (int i = 1; i < R; ++i) v = k == i ? a[i] : v;
          return v;
        };
#pragma unroll 1
        for (int q = 0; q < 32 * R; ++q) {
          const int owner = q / R, k = q % R;
          const uint32_t l = __shfl_sync(0xffffffffu, pick(cur.len, k), owner);
          if (l == 0u) continue;
          const uint32_t off = __shfl_sync(0xffffffffu, pick(offk, k), owner);
          const uint32_t y = __shfl_sync(0xffffffffu, pick(cur.y, k), owner);
          const uint32_t z = __shfl_sync(0xffffffffu, pick(cur.z, k), owner);
          const uint32_t w = __shfl_sync(0xffffffffu, pick(cur.w, k), owner);
          if (l <= 12u) {
            if ((uint32_t)lane < l) {
              const uint32_t word = lane < 4 ? y : (lane < 8 ? z : w);
              out[off + lane] = (uint8_t)(word >> (8 * (lane & 3)));
            }
          } else {
            const uint8_t *src = job.heap_dev + ((((uint64_t)w << 32) | (uint64_t)z) - job.heap_host_base);
            for (uint32_t i = lane; i < l; i += 32) out[off + i] = src[i];
          }
        }
      }
    }
    bar_arrive(kBarPacked, kWL);
    cur = nxt;
    cur_valid = nxt_valid;
  }
}

// ------------------------------------------------------------------ columns without a heap
// A column whose batch registers no heap (heap_len == 0) can only hold inlined strings (<= 12
// bytes; a pointer entry is reported as kErrHeapRange).  Rows then cost 16 bytes in and ~4 + len
// bytes out, so the per-tile latency chain (load -> scan -> look-back) dominates: this kernel takes
// a whole 2048-row vector per CTA, 8 rows per thread, loads them striped (lane-consecutive rows:
// 512 contiguous bytes per request), scans the lengths with one warp scan per stripe, and builds
// the tile's output in a zeroed shared-memory image straight from registers.  It serves the reference
// blob (DMB_STR_REF_BLOB); the Arrow modes take the pack kernel's lean form.
constexpr int kInlRows = kVec;                       // rows per tile
constexpr int kInlPerThread = kInlRows / kThreads;   // 8
struct InlSmem {
  alignas(16) uint8_t stage[kInlRows * 13 + 32];
  uint32_t warp_sum[kThreads / 32];
  uint64_t base;
  long long ticket;
};

// strlen of the <= l inline bytes (y, z, w), for the reference blob
__device__ __forceinline__ uint32_t inline_strlen(const uint4 &e, uint32_t l) {
  uint32_t n = 0;
  const uint32_t w[3] = {e.y, e.z, e.w};
#pragma unroll
  for (int k = 0; k < 12; ++k) {
    const bool z = ((w[k >> 2] >> (8 * (k & 3))) & 0xffu) == 0u;
    if (n == (uint32_t)k && (uint32_t)k < l && !z) n = k + 1;
  }
  return n;
}

template <int MODE>
__global__ void __launch_bounds__(kThreads, 4)
string_inline_kernel(dmb_string_job job, BatchView b, unsigned long long *scratch, int64_t ntiles) {
  __shared__ InlSmem sm;
  unsigned long long *status = scratch + 2;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t tile = claim_tile(scratch, &sm.ticket);  // = chunk index
  if (tile >= ntiles) return;
  const int count = (int)__ldg(b.counts + tile);
  const dmb_vec_desc vd = job.vecs[tile];
  const uint4 *in = reinterpret_cast<const uint4 *>(reinterpret_cast<const uint8_t *>(job.in) + vd.data_off);
  const uint64_t *mask = vd.val_off < 0 ? nullptr : job.in_validity + vd.val_off;

  // stripe k of warp w holds rows w*256 + k*32 + lane
  uint4 e[kInlPerThread];
  uint32_t len[kInlPerThread];
  int bad = 0;
#pragma unroll
  for (int k = 0; k < kInlPerThread; ++k) {
    const int row = warp * (32 * kInlPerThread) + k * 32 + lane;
    e[k] = make_uint4(0, 0, 0, 0);
    len[k] = 0;
    if (row < count) {
      e[k] = ld_stream(in + row);
      const bool valid = mask ? ((__ldg(mask + (row >> 6)) >> (row & 63)) & 1ull) : true;
      if (valid) {
        uint32_t l = e[k].x;
        if (l > 12u) { bad = 1; l = 0; }  // a pointer string, but the batch registered no heap
        if (MODE == DMB_STR_REF_BLOB) l = inline_strlen(e[k], l);
        len[k] = l;
      }
      if (MODE == DMB_STR_REF_BLOB) len[k] += 1;  // terminator; a NULL row is a lone '\0'
    }
  }
  {  // zero the output image while the loads are in flight
    uint4 *z = reinterpret_cast<uint4 *>(sm.stage);
    for (int i = tid; i < (int)(sizeof(sm.stage) / 16); i += kThreads) z[i] = make_uint4(0, 0, 0, 0);
  }
  // exclusive offsets: one warp scan per stripe, carried across the stripes of the warp
  uint32_t off[kInlPerThread];
  uint32_t carry = 0;
#pragma unroll
  for (int k = 0; k < kInlPerThread; ++k) {
    uint32_t incl = len[k];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t n = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += n;
    }
    off[k] = carry + incl - len[k];
    carry += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (lane == 0) sm.warp_sum[warp] = carry;
  const int any_bad = __syncthreads_or(bad);
  uint32_t warp_excl = 0, tile_total = 0;
#pragma unroll
  for (int w = 0; w < kThreads / 32; ++w) {
    const uint32_t s = sm.warp_sum[w];
    if (w < warp) warp_excl += s;
    tile_total += s;
  }
  if (tid == 0 && any_bad) atomicOr(scratch + 1, (unsigned long long)kErrHeapRange);

  // decoupled look-back (warp 0)
  if (warp == 0) {
    const uint64_t agg = (uint64_t)tile_total;
    if (lane == 0) atomicExch(status + tile, (tile == 0 ? kFlagPrefix : kFlagAggregate) | agg);
    uint64_t prefix = 0;
    if (tile > 0) {
      int64_t look = tile - 1;
      while (true) {
        const int64_t idx = look - lane;
        uint64_t st = kFlagPrefix;
        if (idx >= 0) {
          do { st = ld_status(status + idx); } while ((st >> 62) == 0);
        }
        const uint32_t is_p = __ballot_sync(0xffffffffu, (st >> 62) == 2);
        const int first_p = is_p ? (__ffs(is_p) - 1) : 32;
        uint64_t v = lane <= first_p ? (st & kValueMask) : 0ull;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
        prefix += v;
        if (is_p) break;
        look -= 32;
      }
      if (lane == 0) atomicExch(status + tile, kFlagPrefix | ((prefix + agg) & kValueMask));
    }
    if (lane == 0) sm.base = prefix;
  }
  // the gather into the stage needs only (base & 15); do the part that does not need it first
  __syncthreads();
  const uint64_t base = sm.base;
  const uint32_t mis = (uint32_t)(base & 15ull);
  const int64_t out_row0 = __ldg(b.row_off + tile);
  if (MODE != DMB_STR_ARROW_LARGE && base + tile_total > 0x7fffffffull && tid == 0)
    atomicOr(scratch + 1, (unsigned long long)kErrOffsetOverflow);
  uint32_t *sw = reinterpret_cast<uint32_t *>(sm.stage);
#pragma unroll
  for (int k = 0; k < kInlPerThread; ++k) {
    const int row = warp * (32 * kInlPerThread) + k * 32 + lane;
    if (row < count) {
      const uint32_t o = warp_excl + off[k];
      if (MODE == DMB_STR_ARROW_LARGE) __stcs(reinterpret_cast<long long *>(job.out_offsets) + out_row0 + row, (long long)(base + o));
      else __stcs(reinterpret_cast<int32_t *>(job.out_offsets) + out_row0 + row, (int32_t)(base + o));
      const int l = (int)len[k] - (MODE == DMB_STR_REF_BLOB ? 1 : 0);  // payload bytes; the terminator stays 0
      if (l > 0) {
        const uint32_t s0 = mis + o;
        const uint32_t a = s0 & 3u, sh = 8u * a;
        uint32_t *w = sw + (s0 >> 2);
        put32(w, e[k].y << sh, (int)a, (int)a + l);
        put32(w + 1, __funnelshift_l(e[k].y, e[k].z, sh), (int)a - 4, (int)a + l - 4);
        put32(w + 2, __funnelshift_l(e[k].z, e[k].w, sh), (int)a - 8, (int)a + l - 8);
        put32(w + 3, __funnelshift_l(e[k].w, 0u, sh), (int)a - 12, (int)a + l - 12);
      }
    }
  }
  if (tile == ntiles - 1 && tid == 0) {
    if (MODE == DMB_STR_ARROW_LARGE) reinterpret_cast<int64_t *>(job.out_offsets)[b.nrows] = (int64_t)(base + tile_total);
    else reinterpret_cast<int32_t *>(job.out_offsets)[b.nrows] = (int32_t)(base + tile_total);
    if (job.total_bytes) *job.total_bytes = base + tile_total;
  }
  if (tile_total == 0) return;
  if (job.out_data_cap && base + tile_total > job.out_data_cap) {
    if (tid == 0) atomicOr(scratch + 1, (unsigned long long)kErrDataCap);
    return;
  }
  __syncthreads();
  uint8_t *gbase = job.out_data + (base - mis);
  const uint32_t end = mis + tile_total;
  const uint32_t nstage = (end + 15u) >> 4;
  const uint4 *sv = reinterpret_cast<const uint4 *>(sm.stage);
  for (uint32_t v = tid; v < nstage; v += kThreads) {
    const uint32_t p = 16u * v;
    if (p >= mis && p + 16u <= end) {
      st_stream(reinterpret_cast<uint4 *>(gbase + p), sv[v]);
    } else {  // the neighbouring tiles own the other bytes of this vector
      const uint32_t b0 = p > mis ? p : mis, b1 = (p + 16u) < end ? (p + 16u) : end;
      for (uint32_t q = b0; q < b1; ++q) gbase[q] = sm.stage[q];
    }
  }
}

// ------------------------------------------------------------------ ENUM indices -> utf8, one launch (dmb_dev_enum_utf8)
// Rows are ENUM indices of EW = 1 / 2 / 4 bytes.  A row's string_t is looked up in a table of the dictionary's labels built
// in shared memory (<= DMB_ENUM_FUSED_MAX_LABELS labels of <= 12 bytes), so the 16-byte-per-row string_t intermediate of
// enum_to_string_t_kernel is never written or read.  One CTA per 2048-row vector, claimed from a ticket; the bytes are
// placed at tile-local positions in a shared-memory stage, warp 0 then resolves the prefix by look-back, and the stage
// leaves as destination-aligned 16-byte vectors.  The work is bound by instruction issue (a form of this kernel with
// striped rows, ncu r03b: issue 81 %, DRAM 21 %, 141 thread instructions per row: a byte load per index, up to 12
// predicated byte stores per row, four 2x16-bit warp scans per thread), so the rows are laid out to need few instructions:
//   * a thread owns 8 CONSECUTIVE rows: its indices arrive as one 8 / 16 / 2 x 16-byte load, its validity bits as one byte of the mask
//   * the 8 lengths stay packed in one register (4 bits each); one 32-bit warp scan of the per-thread sums
//   * the thread's bytes are one contiguous stream: labels are appended to a running word with funnel shifts and leave as
//     whole 32-bit words (<= 3 stores per row); only the first / last word of the stream, which the neighbouring threads
//     share, is written byte by byte
//   * the 8 consecutive offsets leave as two 16-byte stores
constexpr int kEnumPackCtas = 6;  // CTAs per SM (launch bound)
template <int EW> struct EnumIndex { typedef uint8_t type; };  // the index type of EW bytes
template <> struct EnumIndex<2> { typedef uint16_t type; };
template <> struct EnumIndex<4> { typedef uint32_t type; };

template <bool LARGE, int EW>
__global__ void __launch_bounds__(kThreads, kEnumPackCtas)
enum_pack_kernel(dmb_string_job job, BatchView b, unsigned long long *scratch, int64_t ntiles, dmb_enum_job ej) {
  constexpr int kR = kVec / kThreads;  // 8 rows per thread
  constexpr int kWarps = kThreads / 32;
  __shared__ __align__(16) uint8_t stage[kVec * 12 + 32];
  __shared__ uint4 s_tab[DMB_ENUM_FUSED_MAX_LABELS + 1];
  __shared__ uint32_t warp_sum[kWarps];
  __shared__ uint64_t base_sh;
  __shared__ long long ticket_sh;
  unsigned long long *status = scratch + 2;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t tile = claim_tile(scratch, &ticket_sh);  // = chunk index; every predecessor is owned by a CTA that is running or done
  if (tile >= ntiles) return;
  const int count = (int)__ldg(b.counts + tile);
  const int64_t out_row0 = __ldg(b.row_off + tile);  // (needed at the very end: as a load down there, 21 % of the stall samples sat on it)
  const dmb_vec_desc vd = ej.vecs[tile];
  const uint64_t *mask = vd.val_off < 0 ? nullptr : ej.in_validity + vd.val_off;
  const uint8_t *in_idx = reinterpret_cast<const uint8_t *>(ej.in_data) + vd.data_off;
  const int i0 = tid * kR;

  // ---- the thread's 8 indices, raw (the index under a NULL row is read and dropped)
  uint32_t raw[EW == 4 ? 8 : (EW == 2 ? 4 : 2)];
  {
    constexpr int kWords = EW == 4 ? 8 : (EW == 2 ? 4 : 2);
    const uint8_t *p = in_idx + (size_t)i0 * EW;
    if (i0 + kR <= count && (reinterpret_cast<uintptr_t>(p) & (EW == 1 ? 7u : 15u)) == 0u) {
      if (EW == 1) {
        const uint2 v = ld_stream(reinterpret_cast<const uint2 *>(p));
        raw[0] = v.x; raw[1] = v.y;
      } else {
#pragma unroll
        for (int q = 0; q < kWords; q += 4) {
          const uint4 v = ld_stream(reinterpret_cast<const uint4 *>(p) + q / 4);
          raw[q] = v.x; raw[q + 1] = v.y; raw[q + 2] = v.z; raw[q + 3] = v.w;
        }
      }
    } else {  // the vector's ragged end, or a vector that is only element-aligned
      typedef typename EnumIndex<EW>::type I;
#pragma unroll
      for (int q = 0; q < kWords; ++q) raw[q] = 0u;
#pragma unroll
      for (int k = 0; k < kR; ++k) {
        const uint32_t v = i0 + k < count ? (uint32_t)reinterpret_cast<const I *>(p)[k] : 0u;
        if (EW == 4) raw[k] = v; else raw[(k * EW) >> 2] |= v << (8 * ((k * EW) & 3));
      }
    }
  }
  auto index_of = [&](int k) -> uint32_t {
    if (EW == 4) return raw[k];
    if (EW == 2) return (raw[k >> 1] >> (16 * (k & 1))) & 0xffffu;
    return (raw[k >> 2] >> (8 * (k & 3))) & 0xffu;
  };
  uint32_t vbits = 0u;
  if (i0 < count) {
    vbits = mask ? (uint32_t)__ldg(reinterpret_cast<const uint8_t *>(mask) + tid) : 0xffu;  // byte t of the mask = rows 8t .. 8t + 7
    if (count - i0 < kR) vbits &= (1u << (count - i0)) - 1u;
  }
  // the labels as string_t, once per CTA (the index loads above are in flight meanwhile).  Word 0 of an entry is the label's
  // length; a label too long for this kernel reads as length 0 + bit 30, and entry dict_size -- where every index past the
  // dictionary is sent -- as length 0 + bit 31: the row loop needs no comparisons
  for (uint32_t t = tid; t <= ej.dict_size; t += kThreads) {
    uint4 e = make_uint4(0x80000000u, 0u, 0u, 0u);
    if (t < ej.dict_size) {
      e = enum_entry(ej, t);
      if (e.x > 12u) e = make_uint4(0x40000000u, 0u, 0u, 0u);
    }
    s_tab[t] = e;
  }
  __syncthreads();

  // ---- lengths (4 bits per row), the thread's sum, block scan
  uint32_t lens = 0u, mine = 0u, seen = 0u;
  unsigned bad_idx = 0;
#pragma unroll
  for (int k = 0; k < kR; ++k) {
    const uint32_t ix = index_of(k);
    uint32_t t = s_tab[ix < ej.dict_size ? ix : ej.dict_size].x;
    t = ((vbits >> k) & 1u) ? t : 0u;  // (the index under a NULL row is looked up and dropped)
    seen |= t;
    bad_idx += t >> 31;  // an index past the dictionary: reported, rendered as the empty string
    const uint32_t l = t & 15u;
    lens |= l << (4 * k);
    mine += l;
  }
  const int bad = (seen >> 30) & 1;  // a label too long for this kernel (the host sends such dictionaries the two-step way)
  uint32_t incl = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t n = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += n;
  }
  if (lane == 31) warp_sum[warp] = incl;
  if (bad_idx && ej.bad_index) atomicAdd(ej.bad_index, (unsigned long long)bad_idx);
  const int any_bad = __syncthreads_or(bad);
  uint32_t wincl = lane < kWarps ? warp_sum[lane] : 0u;
  const uint32_t wown = wincl;
#pragma unroll
  for (int d = 1; d < kWarps; d <<= 1) {
    const uint32_t n = __shfl_up_sync(0xffffffffu, wincl, d);
    if (lane >= d) wincl += n;
  }
  const uint32_t tile_total = __shfl_sync(0xffffffffu, wincl, kWarps - 1);
  const uint32_t my_off = __shfl_sync(0xffffffffu, wincl - wown, warp) + incl - mine;  // tile-local byte offset of the thread's first row
  if (tid == 0) {
    atomicExch(status + tile, (tile == 0 ? kFlagPrefix : kFlagAggregate) | (uint64_t)tile_total);
    atomicAdd(status + ntiles + (tile >> 5), kGroupOne | (unsigned long long)tile_total);
    if (any_bad) atomicOr(scratch + 1, (unsigned long long)kErrHeapRange);
  }

  // ---- the thread's bytes: one stream from stage byte my_off on.  Whole words only in the loop: the first word of a stream
  // that starts inside a word leaves with zeros in its low `head` bytes, and after the barrier the threads before write
  // those bytes -- the unfinished tail of their own stream -- over them, byte by byte.
  uint32_t *sw = reinterpret_cast<uint32_t *>(stage);
  const uint32_t head = my_off & 3u;
  uint32_t wp = my_off >> 2, fill = head, acc = 0u;
  const uint32_t wp0 = wp;
#pragma unroll
  for (int k = 0; k < kR; ++k) {
    const uint32_t l = (lens >> (4 * k)) & 15u;
    if (l == 0u) continue;
    const uint4 ent = s_tab[index_of(k)];
    const uint32_t sft = 8u * fill;
    const uint32_t x0 = acc | (ent.y << sft);
    const uint32_t x1 = __funnelshift_l(ent.y, ent.z, sft);
    const uint32_t x2 = __funnelshift_l(ent.z, ent.w, sft);
    const uint32_t x3 = __funnelshift_l(ent.w, 0u, sft);
    const uint32_t n = fill + l, nw = n >> 2;  // n <= 15: at most three words complete
    if (nw >= 1u) sw[wp] = x0;
    if (nw >= 2u) sw[wp + 1] = x1;
    if (nw >= 3u) sw[wp + 2] = x2;
    // bytes of the label past its length never leave: whole words hold only the first 4 nw <= n bytes, the rest is masked here
    acc = ((nw & 2u) ? ((nw & 1u) ? x3 : x2) : ((nw & 1u) ? x1 : x0)) & low_bytes3(n & 3u);
    wp += nw;
    fill = n & 3u;
  }
  __syncthreads();
  // the stream's unfinished tail: bytes [0, fill) of word wp, or [head, fill) when the whole stream lies inside its first word
  if (fill) store_bytes(sw + wp, acc, wp == wp0 ? head : 0u, fill);
  // ---- decoupled look-back (warp 0), after its own bytes are placed: the later it starts, the shorter it is
  if (warp == 0) {
    const uint64_t prefix = lookback_groups(status, status + ntiles, status + ntiles + ((ntiles + 31) >> 5), tile, lane, status - 1,
                                            (unsigned long long)kErrTimeout, g_lookback_limit_ns);
    if (lane == 0) {
      if (tile > 0) atomicExch(status + tile, kFlagPrefix | ((prefix + tile_total) & kValueMask));
      if ((tile & 31) == 31) atomicExch(status + ntiles + ((ntiles + 31) >> 5) + (tile >> 5), kFlagPrefix | ((prefix + tile_total) & kValueMask));
      base_sh = prefix;
    }
  }
  __syncthreads();
  const uint64_t base = base_sh;
  if (tid == 0) {
    if (!LARGE && base + tile_total > 0x7fffffffull) atomicOr(scratch + 1, (unsigned long long)kErrOffsetOverflow);
    if (tile == ntiles - 1) {
      if (LARGE) reinterpret_cast<long long *>(job.out_offsets)[b.nrows] = (long long)(base + tile_total);
      else reinterpret_cast<int32_t *>(job.out_offsets)[b.nrows] = (int32_t)(base + tile_total);
      if (job.total_bytes) *job.total_bytes = base + tile_total;
    }
  }
  // ---- offsets: 8 consecutive values per thread
  if (i0 < count) {
    uint64_t o = base + my_off;
    if (LARGE) {
      long long *oo = reinterpret_cast<long long *>(job.out_offsets) + out_row0 + i0;
      if (i0 + kR <= count && (reinterpret_cast<uintptr_t>(oo) & 15u) == 0u) {
#pragma unroll
        for (int k = 0; k < kR; k += 2) {
          const uint64_t o1 = o + ((lens >> (4 * k)) & 15u);
          __stcs(reinterpret_cast<longlong2 *>(oo + k), make_longlong2((long long)o, (long long)o1));
          o = o1 + ((lens >> (4 * k + 4)) & 15u);
        }
      } else {
#pragma unroll
        for (int k = 0; k < kR; ++k) {
          if (i0 + k < count) __stcs(oo + k, (long long)o);
          o += (lens >> (4 * k)) & 15u;
        }
      }
    } else {
      int32_t *oo = reinterpret_cast<int32_t *>(job.out_offsets) + out_row0 + i0;
      uint32_t o32 = (uint32_t)o;
      if (i0 + kR <= count && (reinterpret_cast<uintptr_t>(oo) & 15u) == 0u) {
#pragma unroll
        for (int k = 0; k < kR; k += 4) {
          const uint32_t o1 = o32 + ((lens >> (4 * k)) & 15u), o2 = o1 + ((lens >> (4 * k + 4)) & 15u), o3 = o2 + ((lens >> (4 * k + 8)) & 15u);
          __stcs(reinterpret_cast<int4 *>(oo + k), make_int4((int)o32, (int)o1, (int)o2, (int)o3));
          o32 = o3 + ((lens >> (4 * k + 12)) & 15u);
        }
      } else {
#pragma unroll
        for (int k = 0; k < kR; ++k) {
          if (i0 + k < count) __stcs(oo + k, (int32_t)o32);
          o32 += (lens >> (4 * k)) & 15u;
        }
      }
    }
  }
  if (tile_total == 0) return;
  if (job.out_data_cap && base + tile_total > job.out_data_cap) {
    if (tid == 0) atomicOr(scratch + 1, (unsigned long long)kErrDataCap);
    return;
  }
  // ---- stage -> out_data: destination-aligned 16-byte vectors; vector v holds tile bytes [16v - mis, 16v - mis + 16)
  uint8_t *gdst = job.out_data + base;
  const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(gdst) & 15u);
  const uint32_t end = mis + tile_total;
  const uint32_t v0 = mis ? 1u : 0u, v1 = end >> 4;  // whole vectors [v0, v1)
  for (uint32_t v = v0 + tid; v < v1; v += kThreads) {
    const uint32_t q = 16u * v - mis, sh = 8u * (q & 3u);
    const uint32_t *s = sw + (q >> 2);
    const uint32_t a0 = s[0], a1 = s[1], a2 = s[2], a3 = s[3], a4 = s[4];  // s[4]: inside the stage's 32 bytes of slack
    uint4 o;
    o.x = __funnelshift_r(a0, a1, sh);
    o.y = __funnelshift_r(a1, a2, sh);
    o.z = __funnelshift_r(a2, a3, sh);
    o.w = __funnelshift_r(a3, a4, sh);
    st_stream(reinterpret_cast<uint4 *>(gdst - mis) + v, o);
  }
  // the ragged first / last vector: the neighbouring tiles own their other bytes
  if (warp == kWarps - 1) {
    const uint32_t h1 = v1 > v0 ? 16u * v0 : end;  // (no whole vector: everything is ragged)
    for (uint32_t q = mis + lane; q < h1; q += 32u) gdst[q - mis] = stage[q - mis];
    if (v1 > v0)
      for (uint32_t q = 16u * v1 + lane; q < end; q += 32u) gdst[q - mis] = stage[q - mis];
  }
}

// bench/test helper: DuckDB-shaped string_t from lengths + heap offsets
__global__ void __launch_bounds__(kThreads)
make_string_t_kernel(const uint32_t *__restrict__ lengths, const uint64_t *__restrict__ heap_off,
                     const uint8_t *__restrict__ heap_dev, uint64_t heap_host_base,
                     dmb_string_t *__restrict__ out, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads) {
    uint32_t l = lengths[i];
    uint64_t ho = heap_off[i];
    uint4 e = make_uint4(l, 0, 0, 0);
    uint8_t *eb = reinterpret_cast<uint8_t *>(&e);
    if (l <= 12u) {
      for (uint32_t k = 0; k < l; ++k) eb[4 + k] = heap_dev[ho + k];
    } else {
      for (uint32_t k = 0; k < 4; ++k) eb[4 + k] = heap_dev[ho + k];
      uint64_t p = heap_host_base + ho;
      e.z = (uint32_t)p;
      e.w = (uint32_t)(p >> 32);
    }
    reinterpret_cast<uint4 *>(out)[i] = e;
  }
}

}  // namespace dmb

using namespace dmb;

extern "C" int32_t dmb_dev_set_lookback_limit_ns(unsigned long long ns) {
  return check_cuda(cudaMemcpyToSymbol(g_lookback_limit_ns, &ns, sizeof(ns)), "set look-back limit");
}

// [0] ticket  [1] error flags  [2, 2 + ntiles) tile status  then, for the pack kernel, one sum word and one prefix word per group of 32 tiles
extern "C" size_t dmb_dev_string_scratch_bytes(int64_t nchunks) {
  const int64_t nt = (int64_t)kStrTilesPerChunk * (nchunks > 0 ? nchunks : 0);
  return (size_t)(2 + nt + 2 * ((nt + 31) / 32)) * sizeof(unsigned long long);
}

extern "C" int32_t dmb_dev_enum_utf8(const dmb_enum_job *ejob, const dmb_string_job *job, const uint32_t *counts,
                                     const int64_t *row_off, int64_t nchunks, int64_t nrows,
                                     void *scratch, void *stream) {
  if (!ejob || !job) { set_error("dmb_dev_enum_utf8: job is null"); return -1; }
  if (job->mode != DMB_STR_ARROW_UTF8 && job->mode != DMB_STR_ARROW_LARGE) { set_error("dmb_dev_enum_utf8: Arrow modes only (mode %d)", job->mode); return -1; }
  if (ejob->dict_size > DMB_ENUM_FUSED_MAX_LABELS) {
    set_error("dmb_dev_enum_utf8: %u labels, the fused kernel takes up to %d (use dmb_dev_enum_to_string_t + dmb_dev_string_batch)", ejob->dict_size, DMB_ENUM_FUSED_MAX_LABELS);
    return -1;
  }
  if (ejob->dict_size && (!ejob->dict_offsets || !ejob->dict_data)) { set_error("dmb_dev_enum_utf8: dictionary is null"); return -1; }
  cudaStream_t st = (cudaStream_t)stream;
  if (nchunks <= 0 || nrows <= 0) return 0;
  if (check_cuda(cudaMemsetAsync(scratch, 0, dmb_dev_string_scratch_bytes(nchunks), st), "string scratch memset")) return -1;
  BatchView b{counts, row_off, nchunks, nrows};
  const bool large = job->mode == DMB_STR_ARROW_LARGE;
  auto launch = [&](auto kernel) -> int32_t {
    kernel<<<(unsigned)nchunks, kThreads, 0, st>>>(*job, b, (unsigned long long *)scratch, nchunks, *ejob);
    return check_cuda(cudaGetLastError(), "enum_pack_kernel launch");
  };
  switch (ejob->phys) {
    case DMB_PHYS_U8: return large ? launch(enum_pack_kernel<true, 1>) : launch(enum_pack_kernel<false, 1>);
    case DMB_PHYS_U16: return large ? launch(enum_pack_kernel<true, 2>) : launch(enum_pack_kernel<false, 2>);
    case DMB_PHYS_U32: return large ? launch(enum_pack_kernel<true, 4>) : launch(enum_pack_kernel<false, 4>);
    default: set_error("dmb_dev_enum_utf8: ENUM indices are uint8/uint16/uint32, not physical type %d", ejob->phys); return -1;
  }
}

extern "C" int32_t dmb_dev_string_batch(const dmb_string_job *job, const uint32_t *counts,
                                        const int64_t *row_off, int64_t nchunks, int64_t nrows,
                                        void *scratch, void *stream) {
  if (!job) { set_error("dmb_dev_string_batch: job is null"); return -1; }
  cudaStream_t st = (cudaStream_t)stream;
  if (nchunks <= 0 || nrows <= 0) return 0;
  const int64_t ntiles = (int64_t)kStrTilesPerChunk * nchunks;
  if (check_cuda(cudaMemsetAsync(scratch, 0, dmb_dev_string_scratch_bytes(nchunks), st), "string scratch memset")) return -1;
  BatchView b{counts, row_off, nchunks, nrows};
  auto launch = [&](auto kernel) -> int32_t {
    kernel<<<(unsigned)ntiles, kThreads, 0, st>>>(*job, b, (unsigned long long *)scratch, ntiles);
    return check_cuda(cudaGetLastError(), "string_batch_kernel launch");
  };
  // Arrow modes: the TMA-staged pack kernel, unless the strings are long (long runs: the run-gather is
  // the better fit) or the heap is beyond 32-bit 16-byte units
  if ((job->mode == DMB_STR_ARROW_UTF8 || job->mode == DMB_STR_ARROW_LARGE) && job->heap_len < (1ull << 35)) {
    const bool large = job->mode == DMB_STR_ARROW_LARGE;
    // persistent grid: as many CTAs as are resident at once (tiles are claimed from a ticket)
    auto launch_pack = [&](auto kernel, int rows_per_tile, int threads, uint32_t ob, uint32_t hb, bool unify = true) -> int32_t {
      const int64_t nt = (int64_t)(kVec / rows_per_tile) * nchunks;
      const size_t smem = (size_t)kPackTail + 2u * (size_t)rows_per_tile * 16u + ob + 2u * ((size_t)hb + 16u) + (unify ? (size_t)(threads - 64) * kPackScratchPerThread : 0u) + 128u;
      if (check_cuda(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "string_pack_kernel smem attribute")) return -1;
      int per_sm = 0;
      if (check_cuda(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem), "string_pack_kernel occupancy")) return -1;
      if (per_sm < 1) { set_error("string_pack_kernel does not fit an SM (%zu bytes of shared memory)", smem); return -1; }
      int dev = 0, sms = kNumSMs;
      if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
      int64_t grid = (int64_t)per_sm * sms;
      if (grid > nt) grid = nt;
      kernel<<<(unsigned)grid, threads, smem, st>>>(*job, b, (unsigned long long *)scratch, nt, ob, hb);
      return check_cuda(cudaGetLastError(), "string_pack_kernel launch");
    };
    // columns without a heap: the pipeline's lean form on whole-vector tiles (16 worker warps x 4 rows) --
    // 0.270 / 0.313 ms per 60 M one-byte / l_shipmode-shaped rows, against 0.287 / 0.334 for a one-CTA-per-tile
    // kernel and 0.297 / 0.336 for 8 worker warps
    if (job->heap_len == 0) {
      constexpr int threads = pack_warps(false) * 32 + 64;
      const uint32_t ob = ((2048u * 12u + 64u) + 127u) & ~127u;
      return large ? launch_pack(string_pack_kernel<true, 4, false>, 2048, threads, ob, 0u) : launch_pack(string_pack_kernel<false, 4, false>, 2048, threads, ob, 0u);
    }
    const double heap_per_row = (double)job->heap_len / (double)nrows;
    // the pipeline needs three CTAs per SM to hide its latencies: S[2] + O + H[2] <= ~72 KiB, i.e. a heap span of
    // <= 18 KiB per 512-row tile.  Longer strings come in long runs, which is what the run-gather is good at.
    // Largest heap stage of a 512-row tile that still leaves three CTAs per SM (228 KiB of shared memory, 1 KiB
    // reserved per CTA; smem = tail + S[2] + O (= hb + 2048) + H[2]).  Measured on the C3 shape (30.8 heap bytes per
    // row): three CTAs 0.98 ms, two CTAs 1.21 ms, the run-gather kernel 1.17 ms per 50 M rows.
    // kHb3u: the same with the unified kernel's scratch area (12 bytes per worker thread); columns whose stage would have to
    // shrink for it (C3: 30.8 heap bytes per row) keep the two-path kernel and the larger stage
    constexpr uint32_t kHb3 = ((233472u / 3u - 1024u - kPackTail - 2u * 512u * 16u - 2048u - 32u - 128u) / 3u) & ~127u;
    constexpr uint32_t kHb3u = ((233472u / 3u - 1024u - kPackTail - 2u * 512u * 16u - 2048u - 32u - 128u - 256u * kPackScratchPerThread) / 3u) & ~127u;
    constexpr double kSlack = 1.15;     // heap stage of a tile: its expected span times kSlack, + 1 KiB
    // a stage a little tighter than kSlack asks for rather than a third CTA lost (tiles that overflow the stage are copied
    // row by row: kMinSlack keeps them rare)
    constexpr double kMinSlack = 1.04;
    constexpr double kHprLimit = ((double)kHb3 - 1024.0 - 128.0) / (512.0 * kMinSlack);  // heap bytes per row the pipeline takes
    constexpr double kR4Limit = 9.5;    // few heap bytes per row (codes, short names): 1024-row tiles, 4 rows per thread, halve the per-tile costs
    constexpr int threads = pack_warps(true) * 32 + 64;
    if (heap_per_row <= kHprLimit) {
      if (heap_per_row <= kR4Limit) {
        uint32_t hb4 = ((uint32_t)(heap_per_row * 1024.0 * kSlack) + 1024u + 127u) & ~127u;
        if (hb4 < 2048u) hb4 = 2048u;
        const uint32_t ob4 = hb4 + 4096u + 2048u;  // inlined rows add at most 12 bytes each: room for 6 bytes per row (the scratch area took the rest of what three CTAs per SM leave)
        return large ? launch_pack(string_pack_kernel<true, 4, true>, 1024, threads, ob4, hb4)
                     : launch_pack(string_pack_kernel<false, 4, true>, 1024, threads, ob4, hb4);
      }
      // 512-row tiles, 2 rows per thread
      uint32_t hb = ((uint32_t)(heap_per_row * 512 * kSlack) + 1024u + 127u) & ~127u;
      if (hb < 2048u) hb = 2048u;
      if (hb > kHb3 && (double)kHb3 >= heap_per_row * 512 * kMinSlack + 1024.0) hb = kHb3;
      const uint32_t ob = hb + 2048u;  // inlined rows add at most 12 bytes each; a tile that exceeds the stage is copied row by row
      if (hb <= kHb3u) return large ? launch_pack(string_pack_kernel<true, 2, true, true>, 512, threads, ob, hb, true) : launch_pack(string_pack_kernel<false, 2, true, true>, 512, threads, ob, hb, true);
      return large ? launch_pack(string_pack_kernel<true, 2, true, false>, 512, threads, ob, hb, false) : launch_pack(string_pack_kernel<false, 2, true, false>, 512, threads, ob, hb, false);
    }
  }
  if (job->heap_len == 0 && job->mode == DMB_STR_REF_BLOB) {  // no heap: inlined strings only, whole-vector tiles
    string_inline_kernel<DMB_STR_REF_BLOB><<<(unsigned)nchunks, kThreads, 0, st>>>(*job, b, (unsigned long long *)scratch, nchunks);
    return check_cuda(cudaGetLastError(), "string_inline_kernel launch");
  }
  switch (job->mode) {
    case DMB_STR_ARROW_UTF8: return launch(string_batch_kernel<DMB_STR_ARROW_UTF8>);
    case DMB_STR_ARROW_LARGE: return launch(string_batch_kernel<DMB_STR_ARROW_LARGE>);
    case DMB_STR_REF_BLOB: return launch(string_batch_kernel<DMB_STR_REF_BLOB>);
    default: set_error("dmb_dev_string_batch: bad mode %d", job->mode); return -1;
  }
}

// error flags of the last string launch that used `scratch` (host reads after a sync)
extern "C" int32_t dmb_dev_string_error(const void *scratch, void *stream) {
  unsigned long long flags = 0;
  if (check_cuda(cudaMemcpyAsync(&flags, (const unsigned long long *)scratch + 1, sizeof(flags), cudaMemcpyDeviceToHost, (cudaStream_t)stream), "string error copy")) return -1;
  if (check_cuda(cudaStreamSynchronize((cudaStream_t)stream), "string error sync")) return -1;
  if (flags & kErrTimeout) set_error("a string tile's look-back gave up waiting for its predecessors; the outputs are not valid");
  else if (flags & kErrHeapRange) set_error("string_t pointer outside the registered heap");
  else if (flags & kErrDataCap) set_error("the column's strings total more bytes than out_data_cap (aliased string_t pointers?)");
  else if (flags & kErrOffsetOverflow) set_error("utf8 data exceeds int32 offsets; use large offsets or smaller batches");
  else if (flags & kErrTileTooBig) set_error("a 1024-row tile holds more than 4 GiB of string bytes");
  return (int32_t)flags;
}

extern "C" int32_t dmb_dev_make_string_t(const uint32_t *lengths, const uint64_t *heap_off,
                                         const uint8_t *heap_dev, uint64_t heap_host_base,
                                         dmb_string_t *out, int64_t n, void *stream) {
  if (n <= 0) return 0;
  int64_t blocks = (n + kThreads - 1) / kThreads;
  int grid = (int)(blocks < (int64_t)kNumSMs * 16 ? blocks : (int64_t)kNumSMs * 16);
  make_string_t_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(lengths, heap_off, heap_dev, heap_host_base, out, n);
  return check_cuda(cudaGetLastError(), "make_string_t_kernel launch");
}
