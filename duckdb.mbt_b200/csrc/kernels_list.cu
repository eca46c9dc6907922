// K9 list_to_arrow: DuckDB LIST vectors -> Arrow list<child> (SURVEY.md §8f item 3, "nested offsets kernels").
//
// DuckDB side, per chunk: a vector of duckdb_list_entry {uint64 offset, uint64 length} (what
// duckdb_vector_get_data returns for a LIST vector) + its validity mask, and ONE child vector per chunk
// (duckdb_list_vector_get_child / _get_size) that the entries index.  Entries need not be in row order or
// contiguous (slices, selections), and the entry of a NULL row is unspecified.
// Arrow side: offsets[n+1] (int32, or int64 for large_list) = running sum of the valid rows' lengths, the
// child values gathered in row order, the child validity bitmap gathered with them (payload under a NULL
// child element zeroed, like every other export of this library).
//
// The reference rejects LIST on its chunk path (src/duckdb_native.c:271-303) and its README lists
// List/Struct/Map as "not yet supported" for Arrow: there is no reference output to match; the contract is
// the Arrow format (validated with pyarrow) and the oracle's restatement of the loops above.
//
// One launch, a persistent grid no larger than what is resident at once (CTA b takes chunks b, b + grid, ...), software
// pipelined inside the CTA like string_pack_kernel:
//   workers (8 warps)  front(next chunk): entries striped into shared memory (NULL rows: length 0), block scan of the lengths,
//                      the chunk's AGGREGATE published, row starts + the contiguity test left in shared memory (two buffers);
//                      back(this chunk): offsets, then the chunk's child elements.  A chunk whose entries are one run in row
//                      order (what a scan produces; detected from entry.offset - start being the same for every non-empty
//                      row) is copied as aligned 16-byte output vectors (source misaligned by whole elements: two aligned
//                      loads + funnel shift), NULL elements zeroed from the mask bits, the child bitmap as a shifted word copy.
//                      Any other chunk is gathered output-centric, one element per lane: row of an output element by binary
//                      search over the chunk's 2048 row starts in shared memory, child validity by warp ballot over
//                      32-aligned groups of OUTPUT elements.  Whole bitmap words are stored; the ragged first / last word of
//                      a chunk is merged with atomicOr into the pre-zeroed bitmap.
//   L (1 warp)         the chunk's base by the two-level decoupled look-back (dmb_common.cuh) WHILE the workers are in
//                      front(next chunk): as one serial chain per chunk (scan -> look-back -> copy, round 1) the other seven
//                      warps spent 19 % of their stall samples at the barrier behind the look-back, and with every CTA at the
//                      same point of its chunk the nearest published PREFIX is a whole grid (~600 chunks) back.
// front(j + 1) needs nothing from other CTAs and back(j) only look-backs over aggregates published in fronts, so the
// resident grid cannot deadlock.  Hand-offs are named barriers (F: worker warp 0 -> L, B: L -> workers), alternating pairs.

#include "dmb_common.cuh"

namespace dmb {

constexpr int kListRpt = kVec / kThreads;    // rows per worker thread: 8
constexpr int kListCta = kThreads + 32;      // 8 worker warps + L
constexpr int kListCtas = 4;                 // CTAs per SM (launch bound)
constexpr int kListCopyUnroll = 4;           // 16-byte vectors of the contiguous copy in flight per thread

struct ListEntry {
  uint64_t offset, length;
};

enum { kLBarWorkers = 1, kLBarF0 = 2, kLBarF1 = 3, kLBarB0 = 4, kLBarB1 = 5 };
__device__ __forceinline__ void lbar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void lbar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// [p, p + bytes) -> L2, trimmed to the whole 16-byte units inside the range (a hint: nothing outside the range is touched)
__device__ __forceinline__ void l2_prefetch(const void *p, uint32_t bytes) {
  const uintptr_t a = (reinterpret_cast<uintptr_t>(p) + 15u) & ~(uintptr_t)15, e = (reinterpret_cast<uintptr_t>(p) + bytes) & ~(uintptr_t)15;
  if (e > a) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a), "r"((uint32_t)(e - a)) : "memory");
}

// exclusive scan over the kThreads worker threads of one value each; returns the exclusive prefix, *total = sum
__device__ __forceinline__ uint64_t workers_exscan(uint64_t v, uint64_t *total, uint64_t *s_warp /* [kThreads / 32 + 1] */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint64_t inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint64_t t = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += t;
  }
  if (lane == 31) s_warp[warp] = inc;
  lbar_sync(kLBarWorkers, kThreads);
  // every warp scans the 8 warp sums itself (one load per lane + 3 shuffle steps): no second barrier for a warp-0 pass
  const uint64_t w = lane < kThreads / 32 ? s_warp[lane] : 0ull;
  uint64_t winc = w;
#pragma unroll
  for (int d = 1; d < kThreads / 32; d <<= 1) {
    const uint64_t t = __shfl_up_sync(0xffffffffu, winc, d);
    if (lane >= d) winc += t;
  }
  const uint64_t warp_excl = __shfl_sync(0xffffffffu, winc - w, warp);
  *total = __shfl_sync(0xffffffffu, winc, kThreads / 32 - 1);
  return warp_excl + inc - v;
}

struct ListShared {
  alignas(16) uint32_t start[2][kVec + 4];  // row -> first output element of the row, relative to the chunk; [count] = the chunk's total
  alignas(16) uint32_t src[2][kVec];        // row -> entry.offset (elements of the chunk's child vector: < 2^32, checked)
  uint64_t warp[2][kThreads / 32 + 1];
  uint32_t wmin[2][kThreads / 32], wmax[2][kThreads / 32];
  unsigned long long csum[2], cbase[2];
  unsigned nulls;
};

template <int W, bool LARGE>
__global__ void __launch_bounds__(kListCta, kListCtas)
list_emit_kernel(dmb_list_job job, BatchView b, unsigned long long *status, unsigned long long *flags) {
  __shared__ ListShared sm;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned long long *gsum = status + 2 * b.nchunks, *gpre = gsum + ((b.nchunks + 31) >> 5);

  if (warp == kThreads / 32) {
    // ------------------------------------------------------------ L: chunk bases
    int j = 0;
    for (int64_t c = blockIdx.x; c < b.nchunks; c += gridDim.x, ++j) {
      const int buf = j & 1;
      lbar_sync(kLBarF0 + buf, 64);  // the chunk is scanned, its aggregate is out
      const uint64_t csum = sm.csum[buf];
      const uint64_t base = lookback_groups(status, gsum, gpre, c, lane, flags, 4ull, 2000000000ull);
      if (lane == 0) {
        if (c > 0) atomicExch(status + c, kFlagPrefix | ((base + csum) & kValueMask));
        if ((c & 31) == 31) atomicExch(gpre + (c >> 5), kFlagPrefix | ((base + csum) & kValueMask));
        sm.cbase[buf] = base;
        if (c == b.nchunks - 1) {
          if (job.total) *job.total = base + csum;
          if (!LARGE && base + csum > 0x7fffffffull) atomicOr(flags, 1ull);  // int32 offsets overflow: use large_list
        }
      }
      __syncwarp();
      lbar_arrive(kLBarB0 + buf, kThreads + 32);
      // L has time to spare: pull what the workers will read next into L2 (bulk prefetches, one instruction each) -- the entries
      // (+ mask) of the chunk after next, whose front() starts an iteration from now, and the child vector (+ its mask) of the
      // next chunk, whose back() follows that.  The workers' loads then wait for L2, not for DRAM.
      if (lane == 0) {
        const int64_t c2 = c + 2 * (int64_t)gridDim.x, c1 = c + (int64_t)gridDim.x;
        if (c2 < b.nchunks) {
          const uint32_t cnt = __ldg(b.counts + c2);
          const dmb_vec_desc vd = job.vecs[c2];
          if (cnt) l2_prefetch(reinterpret_cast<const uint8_t *>(job.in_entries) + vd.data_off, cnt * 16u);
          if (vd.val_off >= 0) l2_prefetch(job.in_validity + vd.val_off, ((cnt + 63u) >> 6) * 8u);
        }
        if (c1 < b.nchunks && job.child_sizes) {
          const uint64_t child1 = __ldg(job.child_base + c1), n1 = __ldg(job.child_sizes + c1);
          const uint64_t bytes = n1 * W < 65536ull ? n1 * W : 65536ull;
          l2_prefetch(reinterpret_cast<const uint8_t *>(job.child_data) + child1 * W, (uint32_t)bytes);
          if (job.child_validity) {
            const bool dense = (job.large & DMB_LIST_DENSE_CHILD_BITS) != 0;
            const int64_t cvo = dense ? (int64_t)(child1 >> 6) : (job.child_val_off ? __ldg(job.child_val_off + c1) : -1);
            const uint64_t mb = ((n1 + 63ull) >> 6) * 8ull;
            if (cvo >= 0) l2_prefetch(job.child_validity + cvo, (uint32_t)(mb < 8192ull ? mb : 8192ull));
          }
        }
      }
    }
    return;
  }

  // -------------------------------------------------------------- workers
  // front: entries -> shared memory, scan, aggregate, contiguity test
  auto front = [&](int64_t c, int buf) {
    const int count = (int)__ldg(b.counts + c);
    const dmb_vec_desc vd = job.vecs[c];
    const ListEntry *ent = reinterpret_cast<const ListEntry *>(reinterpret_cast<const uint8_t *>(job.in_entries) + vd.data_off);
    const uint64_t *mask = vd.val_off < 0 ? nullptr : job.in_validity + vd.val_off;
    uint32_t *s_start = sm.start[buf], *s_src = sm.src[buf];
    // elements in this chunk's child vector; offsets are kept as 32-bit values, so a child vector of 4 G elements or more
    // (or an unknown size) is cut there: what reaches past it is reported like any entry outside its child vector
    uint64_t csize = job.child_sizes ? __ldg(job.child_sizes + c) : 0xfffffffeull;
    const bool big = csize > 0xfffffffeull;
    csize = big ? 0xfffffffeull : csize;
    // the validity bits of this thread's 8 CONSECUTIVE rows (used after the barrier): byte t of the mask = rows 8t .. 8t + 7
    const int i0 = tid * kListRpt;
    uint32_t vbits = 0u;
    if (i0 < count) {
      vbits = mask ? (uint32_t)__ldg(reinterpret_cast<const uint8_t *>(mask) + tid) : 0xffu;
      if (count - i0 < kListRpt) vbits &= (1u << (count - i0)) - 1u;
    }
    // striped (consecutive lanes, consecutive 16-byte entries), a thread's loads in flight together.  Validity is applied
    // after the barrier (one mask byte per thread instead of a mask word per row here); the entry of a NULL row is read and
    // dropped: it is storage of the vector, only its content is unspecified.  An entry that reaches outside the child
    // vector is marked with the length 0xffffffff (no real length: the child vector has fewer elements).
#pragma unroll
    for (int h = 0; h < kListRpt; h += 4) {
      ulonglong2 e[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int i = tid + (h + k) * kThreads;
        e[k] = i < count ? ld_stream(reinterpret_cast<const ulonglong2 *>(ent) + i) : make_ulonglong2(0ull, 0ull);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int i = tid + (h + k) * kThreads;
        const bool inside = e[k].x <= csize && e[k].y <= csize - e[k].x;
        s_src[i] = (uint32_t)e[k].x;
        s_start[i] = inside ? (uint32_t)e[k].y : 0xffffffffu;
      }
    }
    if (big && tid == 0) atomicOr(flags, 2ull);
    lbar_sync(kLBarWorkers, kThreads);
    // this thread's kListRpt consecutive rows: block scan of the lengths, starts written back in place
    uint32_t len[kListRpt], src[kListRpt];
    {
      const uint4 a = *reinterpret_cast<const uint4 *>(s_start + i0), c4 = *reinterpret_cast<const uint4 *>(s_start + i0 + 4);
      len[0] = a.x; len[1] = a.y; len[2] = a.z; len[3] = a.w; len[4] = c4.x; len[5] = c4.y; len[6] = c4.z; len[7] = c4.w;
      const uint4 p = *reinterpret_cast<const uint4 *>(s_src + i0), q = *reinterpret_cast<const uint4 *>(s_src + i0 + 4);
      src[0] = p.x; src[1] = p.y; src[2] = p.z; src[3] = p.w; src[4] = q.x; src[5] = q.y; src[6] = q.z; src[7] = q.w;
    }
    bool outside = false;
#pragma unroll
    for (int k = 0; k < kListRpt; ++k) {
      const bool valid = (vbits >> k) & 1u;
      if (valid && len[k] == 0xffffffffu) outside = true;  // a malformed / stale entry: never read outside the child vector
      if (!valid || len[k] == 0xffffffffu) len[k] = 0u;    // (contributes no elements; the error flag makes the host discard the output)
    }
    if (outside) atomicOr(flags, 8ull);
    uint64_t mine = 0;
#pragma unroll
    for (int k = 0; k < kListRpt; ++k) mine += len[k];
    uint64_t total;
    const uint64_t ex64 = workers_exscan(mine, &total, sm.warp[buf]);
    if (tid == 0) {
      if (total > 0xffffffffull) atomicOr(flags, 2ull);  // one chunk with more than 4 G child elements: reported, the output is not usable
      sm.csum[buf] = total;
      atomicExch(status + c, (c == 0 ? kFlagPrefix : kFlagAggregate) | (total & kValueMask));
      atomicAdd(gsum + (c >> 5), kGroupOne | (total & kGroupSumMask));
    }
    // contiguity: the chunk's entries are one run in row order iff entry.offset - start is the same for every non-empty row
    uint32_t ex = (uint32_t)ex64, dmin = 0xffffffffu, dmax = 0u, st[kListRpt];
    bool any = false;
#pragma unroll
    for (int k = 0; k < kListRpt; ++k) {
      st[k] = ex;
      if (len[k]) {
        const uint32_t d = src[k] - ex;  // (mod 2^32: a run that starts before its output position is a run all the same)
        dmin = any ? (d < dmin ? d : dmin) : d;
        dmax = any ? (d > dmax ? d : dmax) : d;
        any = true;
      }
      ex += len[k];
    }
    *reinterpret_cast<uint4 *>(s_start + i0) = make_uint4(st[0], st[1], st[2], st[3]);
    *reinterpret_cast<uint4 *>(s_start + i0 + 4) = make_uint4(st[4], st[5], st[6], st[7]);
    if (tid == kThreads - 1) s_start[kVec] = ex;  // (= the chunk's total; rows past `count` are empty, so s_start[count] holds it too)
    // one slot per warp; a warp without a non-empty row leaves (0xffffffff, 0): neutral for min / max
    if (!any) { dmin = 0xffffffffu; dmax = 0u; }
    dmin = __reduce_min_sync(0xffffffffu, dmin);
    dmax = __reduce_max_sync(0xffffffffu, dmax);
    if (lane == 0) { sm.wmin[buf][warp] = dmin; sm.wmax[buf][warp] = dmax; }
    if (warp == 0) {
      __syncwarp();
      lbar_arrive(kLBarF0 + buf, 64);
    }
  };

  // back: offsets + the chunk's child elements + child bitmap
  auto back = [&](int64_t c, int buf) {
    const int count = (int)__ldg(b.counts + c);
    const int64_t row0 = __ldg(b.row_off + c);
    const uint64_t child0 = __ldg(job.child_base + c);  // element index of the chunk's child vector in the staged slab
    // child validity: one padded mask per chunk (bit = element index inside the chunk's child vector), or, for a
    // second-level gather, ONE bitmap over the whole slab (bit = element index in the slab: cbit0 = the chunk's first element)
    const bool dense_bits = (job.large & DMB_LIST_DENSE_CHILD_BITS) != 0;
    const int64_t cvo = dense_bits ? 0 : (job.child_val_off ? __ldg(job.child_val_off + c) : -1);
    const uint32_t *s_start = sm.start[buf], *s_src = sm.src[buf];
    lbar_sync(kLBarB0 + buf, kThreads + 32);  // L has resolved the chunk's base
    const uint64_t cbase = sm.cbase[buf];
    const uint64_t csum = sm.csum[buf] > 0xffffffffull ? 0ull : sm.csum[buf];  // (flagged: nothing of the chunk is emitted)
    if (tid == 0 && row0 + count == b.nrows) {  // the last chunk writes offsets[nrows]
      const uint64_t o = cbase + csum;
      if (LARGE) reinterpret_cast<long long *>(job.out_offsets)[b.nrows] = (long long)o;
      else reinterpret_cast<int32_t *>(job.out_offsets)[b.nrows] = (int32_t)o;
    }
    for (int i = tid; i < count; i += kThreads) {  // offsets: coalesced
      const uint64_t o = cbase + s_start[i];
      if (LARGE) __stcs(reinterpret_cast<long long *>(job.out_offsets) + row0 + i, (long long)o);
      else __stcs(reinterpret_cast<int32_t *>(job.out_offsets) + row0 + i, (int32_t)o);
    }
    uint32_t cmin = 0xffffffffu, cmax = 0u;
    {
      const uint32_t a = lane < kThreads / 32 ? sm.wmin[buf][lane] : 0xffffffffu, z = lane < kThreads / 32 ? sm.wmax[buf][lane] : 0u;
      cmin = __reduce_min_sync(0xffffffffu, a);
      cmax = __reduce_max_sync(0xffffffffu, z);
    }
    const bool contiguous = cmin == cmax;
    const uint32_t run_d = cmin;  // source element of output element e of a contiguous chunk: run_d + e (mod 2^32)
    const uint64_t *cmask = (job.child_validity && cvo >= 0) ? job.child_validity + cvo : nullptr;
    const uint64_t cbit0 = dense_bits ? child0 : 0ull;
    const uint64_t first = cbase & ~31ull, end = cbase + csum, stop = (end + 31ull) & ~31ull;
    uint32_t *bm32 = reinterpret_cast<uint32_t *>(job.out_child_validity);
    unsigned nulls = 0;
    if (contiguous) {
      // ---- the chunk's output is one run of its child vector: out[cbase + e] = child[run0 + e].  Aligned 16-byte output
      // vectors (source misaligned by whole elements: two aligned loads + funnel shift), NULL elements zeroed from the mask
      // bits read as aligned 32-bit words; the bitmap is a shifted word copy, one output word per thread.
      constexpr int R = 16 / W;
      const uint64_t run0 = (uint64_t)run_d;  // csum > 0: run_d is the first non-empty row's offset minus its (smaller) start, so no wrap
      const uint8_t *srcb = reinterpret_cast<const uint8_t *>(job.child_data) + (child0 + run0) * W;
      uint8_t *dstb = reinterpret_cast<uint8_t *>(job.out_child) + cbase * W;
      const uintptr_t d0 = reinterpret_cast<uintptr_t>(dstb);
      const uintptr_t dA = (d0 + 15u) & ~(uintptr_t)15, dE = (d0 + csum * W) & ~(uintptr_t)15;
      const uint32_t *cm32 = reinterpret_cast<const uint32_t *>(cmask);
      uint32_t head = (uint32_t)csum, tail0 = (uint32_t)csum;  // elements [0, head) and [tail0, csum) are copied one by one
      if (dE > dA) {
        head = (uint32_t)((dA - d0) / W);
        tail0 = (uint32_t)((dE - d0) / W);
        const uint32_t nvec = (uint32_t)((dE - dA) >> 4);
        const uint8_t *s0 = srcb + (dA - d0);
        const int m = (int)(reinterpret_cast<uintptr_t>(s0) & 15u);
        const uint4 *sal = reinterpret_cast<const uint4 *>(s0 - m);
        const int ws = m >> 2;
        const uint32_t sh = (uint32_t)(m & 3) * 8u;
        const uint64_t sbit0 = cbit0 + run0 + head;  // mask bit of the first element of vector 0
        uint4 *dal = reinterpret_cast<uint4 *>(dA);
#pragma unroll(kListCopyUnroll)
        for (uint32_t v = tid; v < nvec; v += kThreads) {
          const uint4 a = ld_stream(sal + v);
          uint4 o = a;
          if (m) o = shift_words(a, __ldg(sal + v + 1), ws, sh);
          if (cm32) {
            const uint32_t bits = load_bits32(cm32, (int64_t)(sbit0 + (uint64_t)v * R), R);
            o.x &= word_keep<W>(bits, 0);
            o.y &= word_keep<W>(bits, 1);
            o.z &= word_keep<W>(bits, 2);
            o.w &= word_keep<W>(bits, 3);
          }
          st_stream(dal + v, o);
        }
      }
      // the elements in front of / behind the aligned vectors (fewer than 16 / W each; a tiny chunk: all of them)
      {
        using T = typename RawVec<W>::type;
        const uint32_t ntail = (uint32_t)csum - tail0;
        uint32_t e = 0xffffffffu;
        if ((uint32_t)tid < head) e = tid;
        else if (tid >= 32 && (uint32_t)(tid - 32) < ntail && tail0 >= head) e = tail0 + (tid - 32);
        if (head == (uint32_t)csum) {  // no aligned vector at all: walk the elements
          for (uint32_t q = tid; q < (uint32_t)csum; q += kThreads) {
            const uint64_t s = run0 + q;
            const bool valid = cm32 ? (load_bits32(cm32, (int64_t)(cbit0 + s), 1) != 0u) : true;
            T v;
            memset(&v, 0, sizeof(T));
            if (valid) v = *reinterpret_cast<const T *>(srcb + (uint64_t)q * W);
            *reinterpret_cast<T *>(dstb + (uint64_t)q * W) = v;
          }
        } else if (e != 0xffffffffu) {
          const uint64_t s = run0 + e;
          const bool valid = cm32 ? (load_bits32(cm32, (int64_t)(cbit0 + s), 1) != 0u) : true;
          T v;
          memset(&v, 0, sizeof(T));
          if (valid) v = *reinterpret_cast<const T *>(srcb + (uint64_t)e * W);
          *reinterpret_cast<T *>(dstb + (uint64_t)e * W) = v;
        }
      }
      // bitmap: output word Ew holds the mask bits of elements [Ew, Ew + 32) of the run
      for (uint64_t Ew = first + 32ull * tid; Ew < stop; Ew += 32ull * kThreads) {
        const uint64_t lo = Ew > cbase ? Ew : cbase, hi = Ew + 32 < end ? Ew + 32 : end;
        if (hi <= lo) continue;
        const int nb = (int)(hi - lo);
        const uint32_t bits = cm32 ? load_bits32(cm32, (int64_t)(cbit0 + run0 + (lo - cbase)), nb) : (nb == 32 ? 0xffffffffu : ((1u << nb) - 1u));
        nulls += (unsigned)(nb - __popc(bits));
        if (bm32) {
          if (nb == 32) bm32[Ew >> 5] = bits;
          else if (bits) atomicOr(bm32 + (Ew >> 5), bits << (unsigned)(lo - Ew));  // ragged first / last word: shared with the neighbouring chunks
        }
      }
    } else {
      constexpr int U = 4;  // output elements per thread in flight
      using T = typename RawVec<W>::type;
      for (uint64_t E0 = first + tid; E0 < stop; E0 += (uint64_t)U * kThreads) {  // a warp's 32 elements share one bitmap word
        T v[U];
        bool valid[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const uint64_t E = E0 + (uint64_t)u * kThreads;
          valid[u] = false;
          memset(&v[u], 0, sizeof(T));
          if (E >= cbase && E < end) {
            const uint32_t e = (uint32_t)(E - cbase);
            int lo = 0, hi = count;  // the last row whose start is <= e: rows after it start later, empty rows before it are skipped
            while (hi - lo > 1) {
              const int mid = (lo + hi) >> 1;
              if (s_start[mid] <= e) lo = mid; else hi = mid;
            }
            const uint64_t s = (uint64_t)s_src[lo] + (e - s_start[lo]);
            // the element is read whether or not it is NULL (it is storage of the child vector): mask word and element in flight together
            const uint64_t cw = cmask ? __ldg(cmask + ((cbit0 + s) >> 6)) : ~0ull;
            v[u] = *reinterpret_cast<const T *>(reinterpret_cast<const uint8_t *>(job.child_data) + (child0 + s) * W);
            valid[u] = (cw >> ((cbit0 + s) & 63)) & 1ull;
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const uint64_t E = E0 + (uint64_t)u * kThreads;
          if (E >= cbase && E < end && !valid[u]) {
            memset(&v[u], 0, sizeof(T));
            ++nulls;
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const uint64_t E = E0 + (uint64_t)u * kThreads;
          if (E >= cbase && E < end) *reinterpret_cast<T *>(reinterpret_cast<uint8_t *>(job.out_child) + E * W) = v[u];
          const uint32_t word = __ballot_sync(0xffffffffu, valid[u]);
          if (lane == 0 && bm32 && E < stop) {
            if (E >= cbase && E + 32 <= end) bm32[E >> 5] = word;   // lane 0's E is 32-aligned
            else if (word) atomicOr(bm32 + (E >> 5), word);         // ragged first / last word: shared with the neighbouring chunks
          }
        }
      }
    }
    if (job.child_null_count) {  // one global atomic per chunk
      nulls = __reduce_add_sync(0xffffffffu, nulls);
      if (lane == 0 && nulls) atomicAdd(&sm.nulls, nulls);
    }
    lbar_sync(kLBarWorkers, kThreads);  // (also: every worker has left this chunk's buffers, front(j + 2) may fill them)
    if (tid == 0 && job.child_null_count && sm.nulls) {
      atomicAdd(job.child_null_count, (unsigned long long)sm.nulls);
      sm.nulls = 0u;  // (the next back()'s first add comes after a workers' barrier of the front() in between)
    }
  };

  if (tid == 0) sm.nulls = 0u;
  int64_t c = blockIdx.x;  // (the grid is no larger than the number of chunks)
  front(c, 0);
  for (int j = 0;; ++j) {
    const int64_t next = c + gridDim.x;
    if (next < b.nchunks) front(next, (j + 1) & 1);
    back(c, j & 1);
    if (next >= b.nchunks) break;
    c = next;
  }
}

}  // namespace dmb

using namespace dmb;

extern "C" size_t dmb_dev_list_scratch_bytes(int64_t nchunks) {
  const int64_t n = nchunks > 0 ? nchunks : 0;
  return (size_t)(2 * n + 2 + 2 * ((n + 31) / 32)) * sizeof(unsigned long long);
}

// scratch: [0] error flags (1: int32 offsets overflow, 2: a chunk with > 4 G child elements, 4: a look-back gave up
// waiting, 8: a list entry reaches outside its chunk's child vector), [1] unused,
// then one look-back status word per chunk (aggregate / inclusive prefix), nchunks words that are no longer used (round 1's
// precomputed chunk bases; the size function is part of the ABI), and a sum word + a prefix word per group of 32 chunks (the
// two-level look-back).  out_child_validity must hold ceil(total / 64) + 1 words.
extern "C" int32_t dmb_dev_list_batch(const dmb_list_job *job, const uint32_t *counts, const int64_t *row_off, int64_t nchunks,
                                      int64_t nrows, int64_t child_capacity, void *scratch, void *stream) {
  if (!job) { set_error("dmb_dev_list_batch: job is null"); return -1; }
  cudaStream_t st = (cudaStream_t)stream;
  if (nchunks <= 0 || nrows <= 0) return 0;
  const int w = job->child_width;
  if (w != 1 && w != 2 && w != 4 && w != 8 && w != 16) { set_error("dmb_dev_list_batch: child width %d (fixed-width children of 1/2/4/8/16 bytes)", w); return -1; }
  unsigned long long *flags = (unsigned long long *)scratch;
  unsigned long long *status = flags + 2;
  if (check_cuda(cudaMemsetAsync(scratch, 0, dmb_dev_list_scratch_bytes(nchunks), st), "list scratch memset")) return -1;
  if (job->out_child_validity && child_capacity > 0 &&
      check_cuda(cudaMemsetAsync(job->out_child_validity, 0, (size_t)((child_capacity + 63) / 64 + 1) * 8, st), "list child bitmap memset")) return -1;
  if (job->child_null_count && check_cuda(cudaMemsetAsync(job->child_null_count, 0, 8, st), "list null count memset")) return -1;
  BatchView b{counts, row_off, nchunks, nrows};
  auto launch = [&](auto kernel) -> int32_t {
    // persistent grid, no larger than what is resident at once (the look-back relies on it)
    int per_sm = 0, dev = 0, sms = kNumSMs;
    cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (check_cuda(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kListCta, 0), "list_emit_kernel occupancy")) return -1;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (per_sm < 1) { set_error("list_emit_kernel does not fit an SM"); return -1; }
    const int64_t resident = (int64_t)per_sm * sms;
    const int g1 = (int)(nchunks < resident ? nchunks : resident);
    kernel<<<g1, kListCta, 0, st>>>(*job, b, status, flags);
    return 0;
  };
#define DMB_LIST_LAUNCH(W)                                                        \
  do {                                                                            \
    if (job->large & 1) { if (launch(list_emit_kernel<W, true>)) return -1; }     \
    else { if (launch(list_emit_kernel<W, false>)) return -1; }                   \
  } while (0)
  switch (w) {
    case 1: DMB_LIST_LAUNCH(1); break;
    case 2: DMB_LIST_LAUNCH(2); break;
    case 4: DMB_LIST_LAUNCH(4); break;
    case 8: DMB_LIST_LAUNCH(8); break;
    default: DMB_LIST_LAUNCH(16); break;
  }
#undef DMB_LIST_LAUNCH
  return check_cuda(cudaGetLastError(), "list kernels launch");
}
