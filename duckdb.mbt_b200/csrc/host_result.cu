// L1 host API (duckdb_mb_gpu_result_*) and L2 drop-in symbols (duckdb_mb_arrow_*).
//
// A result holds what the reference keeps in `duckdb_mb_arrow_result` (src/duckdb_native.c:2211-2217:
// the duckdb_result plus int32 column/row counts) in DataChunk form: per column, the pointers
// duckdb_vector_get_data / duckdb_vector_get_validity return for each chunk.  Every export
//   * stages the column to HBM (a few large cudaMemcpyAsync on the copy-in stream),
//   * runs the conversion kernel of kernels_fixed.cu / kernels_string.cu on the compute stream,
//   * copies the result into page-locked host memory on the copy-out stream,
// column by column, so that copy-in of column j+1, the kernel of column j and copy-out of column
// j-1 overlap (PCIe is full duplex; the kernels are ~100x faster than the link).
//
// There is no CPU fallback: without a CUDA device every entry point fails with an error string.

#include <algorithm>
#include <chrono>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "host_common.hpp"

namespace dmb {
namespace {

double now_ms() {
  using namespace std::chrono;
  return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

// page-locked Arrow buffers of one column; exported ArrowArrays share ownership, so an exported
// array stays valid after duckdb_mb_arrow_destroy / duckdb_mb_gpu_ctx_destroy
// an ENUM type's dictionary (dmb_enum_dict copied at result_from_chunks); shared with exported Arrow dictionaries
struct EnumDict {
  std::vector<uint32_t> offsets;  // size + 1
  std::vector<char> data;
  uint32_t max_len = 0;
  uint32_t *d_offsets = nullptr;  // device copies, staged on first use, owned by the result
  uint8_t *d_data = nullptr;
  uint32_t size() const { return (uint32_t)(offsets.size() - 1); }
};

struct ArrowColOut {
  std::shared_ptr<CtxCore> core;
  std::shared_ptr<EnumDict> dict;  // dictionary-encoded export (ENUM)
  std::vector<std::shared_ptr<ArrowColOut>> children;  // list<child> / map<entries>: one; struct<...>: one per field
  int64_t flags = 2;                   // ARROW_FLAG_NULLABLE (map keys: 0)
  bool no_values = false;              // struct: the validity buffer only
  std::string name, format;
  int64_t length = 0, null_count = 0;
  void *validity = nullptr, *values = nullptr, *data = nullptr;  // values = offsets for utf8
  size_t validity_bytes = 0, values_bytes = 0, data_bytes = 0;
  ~ArrowColOut() {
    if (!core) return;
    core->pin.free(validity);
    core->pin.free(values);
    core->pin.free(data);
  }
};

struct TypedOut {
  bool ready = false;
  int32_t tag = DMB_VALUE_NULL, width = 0;
  int64_t null_count = 0;
  void *values = nullptr, *valid = nullptr, *offsets = nullptr, *data = nullptr;  // pinned
};

// the type of a column or of a nested leaf: what arrow_map needs of either
struct ColType {
  std::string name;
  int32_t type_id = 0, phys = 0, dec_width = 0, dec_scale = 0, width = 0;
};

// ---- nested types (SURVEY.md 8f item 3).  The child level of a LIST / MAP column, in whichever form dmb_host_list gave
// it (flat fixed-width fields or child_col): every "leaf" is one vector family (one child vector per chunk, sizes[k]
// elements of it), staged as one flat slab.
struct ListNode;
struct Leaf : ColType {
  std::vector<const void *> data;      // [nchunks]
  std::vector<const void *> validity;  // [nchunks] or empty (no masks at all)
  // staged
  uint8_t *d_data = nullptr;
  uint64_t *d_validity = nullptr;      // per-chunk padded masks (word offsets d_val_off), or one dense bitmap over the slab
  int64_t *d_val_off = nullptr;
  uint8_t *d_heap = nullptr;           // VARCHAR / BLOB leaves: the child vectors' strings, gathered by the stager
  uint64_t heap_len = 0;
};
struct ListNode {
  enum Kind { kLeaf = 0, kStruct = 1, kList = 2 };
  int kind = kLeaf;
  std::vector<uint64_t> sizes, base;   // per chunk; base has nchunks + 1 entries
  std::vector<Leaf> leaves;            // kLeaf: one; kStruct: one per field; kList: the inner list's entries (16 bytes, rebased)
  Leaf struct_validity;                // kStruct: the struct vectors' own masks (width 1 dummy payload)
  bool has_struct_validity = false;
  std::shared_ptr<ListNode> inner;     // kList: the level below
  uint64_t *d_base = nullptr, *d_sizes = nullptr;
  bool staged = false;
};

struct Col : ColType {
  std::vector<const void *> data;
  std::vector<const void *> validity;  // entries may be NULL; empty = no masks at all
  bool any_validity = false;
  const uint8_t *heap_base = nullptr;
  uint64_t heap_len = 0;
  bool force_large = false;  // export as large_utf8 / large_binary whatever the size (all parts of a sharded table agree)
  std::shared_ptr<EnumDict> dict;  // ENUM
  // STRUCT: the fields are columns of their own, appended behind the visible ones (indices into Result::cols)
  bool is_struct = false;
  std::vector<int> kids;
  // LIST / MAP: the child level
  std::shared_ptr<ListNode> node;
  bool is_map = false;
  // device copy (lives as long as the result)
  bool staged = false;
  uint8_t *d_data = nullptr;
  uint64_t *d_validity = nullptr;
  dmb_vec_desc *d_vecs = nullptr;
  uint8_t *d_heap = nullptr;
  uint64_t heap_host_base = 0, d_heap_len = 0;
  cudaEvent_t ev_staged = nullptr;
  std::shared_ptr<ArrowColOut> arrow;
  // reference packed blob of this column, complete in pinned memory (getter prefetch): kind = GetterKind or 4 = string
  int gc_kind = -1;
  bool gc_nullable = false;
  uint8_t *gc_blob = nullptr;
  size_t gc_bytes = 0;
  TypedOut typed;
  TypedOut text;  // VARCHAR rendering of the column (QueryResult's string form)
};

}  // namespace
}  // namespace dmb

using namespace dmb;

struct duckdb_mb_arrow_result {
  std::shared_ptr<CtxCore> core;
  int64_t nchunks = 0, nrows = 0;
  int32_t column_count = 0, row_count = 0;  // (int32_t) casts like src/duckdb_native.c:2264-2265
  bool pinned_input = false;
  std::vector<uint32_t> counts;
  std::vector<int64_t> row_off;
  uint32_t *d_counts = nullptr;
  int64_t *d_row_off = nullptr;
  bool meta_staged = false;
  std::vector<Col> cols;
  std::vector<void *> dev_keep, pin_keep;  // staged inputs / typed outputs: freed when the result dies
  std::vector<cudaEvent_t> events;
  bool arrow_ready = false;
  bool getters_prefetched = false;
  std::shared_ptr<void> owner;  // the glue's duckdb_result + chunk handles: shared with the result's slices (shards, stream parts)
  double t_h2d = 0, t_kernels = 0, t_d2h = 0, t_total = 0;
  uint64_t bytes_h2d = 0, bytes_d2h = 0;
};

namespace dmb {
namespace {

typedef duckdb_mb_arrow_result Result;
static_assert(sizeof(dmb_string_t) == 16, "duckdb_string_t is 16 bytes");

void *keep_dev(Result *r, size_t bytes) {
  void *p = r->core->dev.alloc(bytes + 64);
  if (p) r->dev_keep.push_back(p);
  return p;
}
void *keep_pin(Result *r, size_t bytes) {
  void *p = r->core->pin.alloc(bytes + 64);
  if (p) r->pin_keep.push_back(p);
  return p;
}

void free_result(Result *r) {
  if (!r) return;
  CtxCore &c = *r->core;
  {
    std::lock_guard<std::mutex> g(c.mu);
    c.bind();
    cudaStreamSynchronize(c.s_in);
    cudaStreamSynchronize(c.s_compute);
    cudaStreamSynchronize(c.s_out);
    for (void *p : r->dev_keep) c.dev.free(p);
    for (void *p : r->pin_keep) c.pin.free(p);
    for (cudaEvent_t e : r->events) cudaEventDestroy(e);
    r->cols.clear();  // ArrowColOut buffers go back to the pinned pool unless an export still holds them
  }
  delete r;  // (drops the owner reference: after the last use of the host chunk pointers)
}

int32_t ensure_meta(Result *r) {
  if (r->meta_staged) return 0;
  CtxCore &c = *r->core;
  const size_t nb_counts = sizeof(uint32_t) * (size_t)(r->nchunks > 0 ? r->nchunks : 1);
  const size_t nb_off = sizeof(int64_t) * (size_t)(r->nchunks + 1);
  r->d_counts = (uint32_t *)keep_dev(r, nb_counts);
  r->d_row_off = (int64_t *)keep_dev(r, nb_off);
  uint8_t *pin = (uint8_t *)keep_pin(r, nb_counts + nb_off);
  if (!r->d_counts || !r->d_row_off || !pin) return -1;
  if (r->nchunks) memcpy(pin, r->counts.data(), sizeof(uint32_t) * (size_t)r->nchunks);
  memcpy(pin + nb_counts, r->row_off.data(), nb_off);
  if (check_cuda(cudaMemcpyAsync(r->d_counts, pin, nb_counts, cudaMemcpyHostToDevice, c.s_in), "counts H2D")) return -1;
  if (check_cuda(cudaMemcpyAsync(r->d_row_off, pin + nb_counts, nb_off, cudaMemcpyHostToDevice, c.s_in), "row_off H2D")) return -1;
  r->bytes_h2d += nb_counts + nb_off;
  r->meta_staged = true;
  return 0;
}

// String columns whose heap nobody registered: the pointed-to bytes are compacted into pinned arena segments while the
// string_t are staged.  A gather task (64 chunk vectors, 2 MB of string_t that are still in the core's cache) sums the bytes
// of its pointer strings, reserves that many bytes of the arena, copies the strings there and rewrites the pointers -- one
// pass over the string_t.  (Round 2 first sized the arena with a pass of its own over every string_t of the column, 59 ms of
// a 355 ms step for the two text columns of the C2 table; a per-ring-buffer plan with a second pass over the buffer moved
// those 59 ms into the gather instead of removing them: the 32 MiB buffer is no longer cached when the second pass comes.)
// Arena positions are logical: segment s covers [base_s, base_s + cap_s) of one address range per column, the device heap is
// allocated when the column is through and every segment's used bytes are copied to base_s in it.
struct ArenaSeg {
  uint8_t *pin;
  uint64_t base, used, cap;
};
struct CompactCtx {
  Result *r = nullptr;
  const Col *col = nullptr;
  int64_t nchunks = 0;
  std::mutex mu;
  std::vector<ArenaSeg> segs;
  uint64_t fake_base = 0;
  bool failed = false;
};
constexpr uint64_t kArenaSegMax = 256ull << 20, kArenaSegMin = 1ull << 20;

inline bool host_row_valid(const void *mask, uint32_t row) {
  if (!mask) return true;
  return (reinterpret_cast<const uint64_t *>(mask)[row >> 6] >> (row & 63)) & 1ull;
}

// `bytes` of the arena for a task that covers `nch_task` chunks: logical position + where that is in pinned memory
bool compact_reserve(CompactCtx *cc, uint64_t bytes, int64_t nch_task, uint64_t *pos, uint8_t **at) {
  std::lock_guard<std::mutex> g(cc->mu);
  if (cc->failed) return false;
  if (cc->segs.empty() || cc->segs.back().used + bytes > cc->segs.back().cap) {
    // a new segment: what the whole column needs if it goes on like this task (+ 10 %), between 1 MiB and 256 MiB; a task
    // larger than that gets a segment of its own size
    uint64_t want = bytes / (uint64_t)(nch_task > 0 ? nch_task : 1) * (uint64_t)cc->nchunks;
    want += want / 10 + kArenaSegMin;
    want = want > kArenaSegMax ? kArenaSegMax : want;
    want = want < bytes ? bytes : want;
    if (!cc->r->core->bind()) { cc->failed = true; return false; }  // (a worker thread: the pinned pool may have to allocate)
    uint8_t *pin = (uint8_t *)keep_pin(cc->r, (size_t)want + 32);
    if (!pin) { cc->failed = true; return false; }
    const uint64_t base = cc->segs.empty() ? 0ull : cc->segs.back().base + cc->segs.back().cap;
    cc->segs.push_back(ArenaSeg{pin, base, 0, want});
  }
  ArenaSeg &seg = cc->segs.back();
  *pos = seg.base + seg.used;
  *at = seg.pin + seg.used;
  seg.used += bytes;
  return true;
}

void compact_task(void *user, int64_t c0, int64_t c1, uint8_t *staged0, size_t slot_bytes) {
  CompactCtx *cc = reinterpret_cast<CompactCtx *>(user);
  const Col &col = *cc->col;
  const std::vector<uint32_t> &counts = cc->r->counts;
  auto mask_of = [&](int64_t k) -> const void * { return col.validity.empty() ? nullptr : col.validity[(size_t)k]; };
  // 1: bytes of the task's pointer strings (payload under a NULL row is unspecified: not counted, never followed)
  uint64_t sum = 0;
  for (int64_t k = c0; k < c1; ++k) {
    if (!col.data[(size_t)k]) continue;
    const dmb_string_t *e = reinterpret_cast<const dmb_string_t *>(staged0 + (size_t)(k - c0) * slot_bytes);
    const void *mask = mask_of(k);
    const uint32_t n = counts[(size_t)k];
    for (uint32_t i = 0; i < n; ++i)
      if (host_row_valid(mask, i) && e[i].length > 12) sum += e[i].length;
  }
  if (!sum) return;
  // 2: that many bytes of the arena
  uint64_t pos = 0;
  uint8_t *at = nullptr;
  if (!compact_reserve(cc, sum, c1 - c0, &pos, &at)) return;
  // 3: copy + rewrite.  Pointer strings that follow each other in memory (what a scan leaves in a vector's string heap) are
  // copied as ONE run: per row that is a compare and an add instead of a ~27-byte memcpy of unpredictable size.
  uint8_t *arena = at - pos;  // arena + logical position = the byte's place in the segment
  for (int64_t k = c0; k < c1; ++k) {
    if (!col.data[(size_t)k]) continue;
    dmb_string_t *e = reinterpret_cast<dmb_string_t *>(staged0 + (size_t)(k - c0) * slot_bytes);
    const void *mask = mask_of(k);
    const uint32_t n = counts[(size_t)k];
    const uint8_t *run_src = nullptr;
    uint64_t run_pos = pos, run_len = 0;
    for (uint32_t i = 0; i < n; ++i) {
      if (!host_row_valid(mask, i)) continue;
      const uint32_t len = e[i].length;
      if (len <= 12) continue;
      const uint8_t *src = reinterpret_cast<const uint8_t *>((uintptr_t)e[i].tail.ptr);
      if ((uintptr_t)src != (uintptr_t)run_src + run_len) {  // (also the first pointer row: run_src is null)
        if (run_len) memcpy(arena + run_pos, run_src, (size_t)run_len);
        run_src = src;
        run_pos = pos;
        run_len = 0;
      }
      run_len += len;
      e[i].tail.ptr = cc->fake_base + pos;
      pos += len;
    }
    if (run_len) memcpy(arena + run_pos, run_src, (size_t)run_len);
  }
}

// copy one column's chunk vectors (payload, validity masks, descriptors, string heap) to HBM
int32_t stage_column(Result *r, int j) {
  Col &col = r->cols[(size_t)j];
  if (col.staged) return 0;
  NvtxRange nvtx("dmb::stage_column");
  if (ensure_meta(r)) return -1;
  CtxCore &c = *r->core;
  struct StageTimer { CtxCore &c; double t0; ~StageTimer() { c.t_stage += wall_ms() - t0; } } stage_timer{c, wall_ms()};
  const int64_t nch = r->nchunks;
  const size_t nslots = (size_t)(nch > 0 ? nch : 1);
  const size_t slot = (size_t)DMB_VECTOR_SIZE * (size_t)col.width;
  col.d_data = (uint8_t *)keep_dev(r, slot * nslots + 16);
  if (!col.d_data) return -1;
  if (col.any_validity) {
    col.d_validity = (uint64_t *)keep_dev(r, 8 * (size_t)DMB_VALIDITY_WORDS * nslots + 16);
    if (!col.d_validity) return -1;
  }
  dmb_vec_desc *pv = (dmb_vec_desc *)keep_pin(r, sizeof(dmb_vec_desc) * nslots);
  col.d_vecs = (dmb_vec_desc *)keep_dev(r, sizeof(dmb_vec_desc) * nslots);
  if (!pv || !col.d_vecs) return -1;
  for (int64_t k = 0; k < nch; ++k) {
    pv[k].data_off = (uint64_t)k * slot;
    pv[k].val_off = (col.any_validity && col.validity[(size_t)k]) ? k * DMB_VALIDITY_WORDS : -1;
  }
  if (nch && check_cuda(cudaMemcpyAsync(col.d_vecs, pv, sizeof(dmb_vec_desc) * (size_t)nch, cudaMemcpyHostToDevice, c.s_in), "vec desc H2D")) return -1;
  r->bytes_h2d += sizeof(dmb_vec_desc) * (size_t)nch;

  StageFixup fixup{compact_task, nullptr};
  CompactCtx cc;
  bool compact = false;
  if (col.phys == DMB_PHYS_STRING) {
    if (col.heap_base == (const uint8_t *)DMB_HEAP_INLINE_ONLY && col.heap_len == 0) {
      // the caller vouches for an all-inlined column: nothing to stage, the heap-less kernel checks every entry
      col.d_heap = nullptr;
      col.heap_host_base = 0;
      col.d_heap_len = 0;
    } else if (col.heap_len > 0 && col.heap_base) {
      // contiguous heap registered by the caller: copy wholesale, rebase pointers in the kernel
      col.d_heap = (uint8_t *)keep_dev(r, (size_t)col.heap_len + 32);
      if (!col.d_heap) return -1;
      if (stage_contiguous(c, c.s_in, col.d_heap, col.heap_base, (size_t)col.heap_len, r->pinned_input ? 1 : 0, &r->bytes_h2d)) return -1;
      col.heap_host_base = (uint64_t)(uintptr_t)col.heap_base;
      col.d_heap_len = col.heap_len;
    } else {
      // scattered heap: gathered into pinned arena segments while the string_t are staged (CompactCtx)
      cc.r = r;
      cc.col = &col;
      cc.nchunks = nch > 0 ? nch : 1;
      cc.fake_base = 1ull << 40;
      fixup.user = &cc;
      compact = true;
    }
  }
  if (nch && !col.is_struct &&  // (a STRUCT vector has no payload of its own: validity + descriptors only)
      stage_pieces(c, c.s_in, col.data.data(), r->counts.data(), (size_t)col.width, slot, nch, col.d_data,
                   r->pinned_input, compact ? &fixup : nullptr, &r->bytes_h2d)) return -1;
  if (compact) {
    // every piece was gathered (host side) before its ring copy was issued, so the segments are complete
    if (cc.failed) return -1;
    const uint64_t total = cc.segs.empty() ? 0ull : cc.segs.back().base + cc.segs.back().used;
    col.heap_host_base = cc.fake_base;
    col.d_heap_len = total;
    col.d_heap = (uint8_t *)keep_dev(r, (size_t)total + 32);
    if (!col.d_heap) return -1;
    for (const ArenaSeg &seg : cc.segs) {
      if (seg.used && check_cuda(cudaMemcpyAsync(col.d_heap + seg.base, seg.pin, (size_t)seg.used, cudaMemcpyHostToDevice, c.s_in), "string arena H2D")) return -1;
      r->bytes_h2d += seg.used;
    }
  }
  if (col.any_validity && nch) {
    if (stage_pieces(c, c.s_in, col.validity.data(), nullptr, 0, 8 * (size_t)DMB_VALIDITY_WORDS, nch,
                     (uint8_t *)col.d_validity, r->pinned_input, nullptr, &r->bytes_h2d)) return -1;
  }
  cudaEvent_t e = nullptr;
  if (check_cuda(cudaEventCreateWithFlags(&e, cudaEventDisableTiming), "cudaEventCreate")) return -1;
  r->events.push_back(e);
  col.ev_staged = e;
  if (check_cuda(cudaEventRecord(col.ev_staged, c.s_in), "event record")) return -1;
  col.staged = true;
  return 0;
}

// upload one job struct; the device copy is consumed by the next launch on s_compute
void *upload_job(Scope &sc, const void *job, size_t bytes) {
  void *hp = sc.palloc(bytes), *dp = sc.dalloc(bytes);
  if (!hp || !dp) return nullptr;
  memcpy(hp, job, bytes);
  if (check_cuda(cudaMemcpyAsync(dp, hp, bytes, cudaMemcpyHostToDevice, sc.c.s_compute), "job H2D")) return nullptr;
  return dp;
}

struct FixedRun {
  uint8_t *d_values = nullptr;
  size_t values_bytes = 0;
  uint64_t *d_bitmap = nullptr;
  size_t bitmap_bytes = 0;
  uint8_t *d_valid_bytes = nullptr;
  unsigned long long *d_null_count = nullptr;
  cudaEvent_t done = nullptr;
};

// launch one fixed-width conversion of column j on the compute stream (after its staging).
// op == DMB_OP_VALIDITY_ONLY or an unsupported (phys,dst) pair with zero_width > 0: only the
// validity outputs are produced and the values are `zero_width` zero bytes per row.
int32_t run_fixed(Result *r, Scope &sc, int j, int32_t op, int zero_width, bool want_bitmap, bool want_valid_bytes,
                  FixedRun *out, int32_t param = 0) {
  if (stage_column(r, j)) return -1;
  CtxCore &c = *r->core;
  Col &col = r->cols[(size_t)j];
  const int64_t n = r->nrows;
  int32_t w = -2;
  if (op != DMB_OP_VALIDITY_ONLY) {
    w = dmb_op_out_width(op);
    if (w < 0 && zero_width <= 0) { set_error("unsupported conversion op 0x%x for column %d", op, j); return -1; }
  }
  if (w >= 0) {
    out->values_bytes = w == 0 ? (size_t)((n + 7) / 8) : (size_t)n * (size_t)w;
    out->d_values = (uint8_t *)sc.dalloc(out->values_bytes + 64);
    if (!out->d_values) return -1;
  } else if (zero_width > 0) {
    out->values_bytes = (size_t)n * (size_t)zero_width;
    out->d_values = (uint8_t *)sc.dalloc(out->values_bytes + 64);
    if (!out->d_values) return -1;
    if (check_cuda(cudaMemsetAsync(out->d_values, 0, out->values_bytes, c.s_compute), "zero values")) return -1;
    op = DMB_OP_VALIDITY_ONLY;
  }
  if (want_bitmap) {
    out->bitmap_bytes = (size_t)((n + 63) / 64) * 8;
    out->d_bitmap = (uint64_t *)sc.dalloc(out->bitmap_bytes + 64);
    if (!out->d_bitmap) return -1;
  }
  if (want_valid_bytes) {
    out->d_valid_bytes = (uint8_t *)sc.dalloc((size_t)n + 64);
    if (!out->d_valid_bytes) return -1;
  }
  out->d_null_count = (unsigned long long *)sc.dalloc(8);
  if (!out->d_null_count) return -1;
  if (check_cuda(cudaMemsetAsync(out->d_null_count, 0, 8, c.s_compute), "counter memset")) return -1;
  dmb_fixed_job job;
  memset(&job, 0, sizeof(job));
  job.in_data = col.d_data;
  job.in_validity = col.d_validity;
  job.vecs = col.d_vecs;
  job.out_values = op == DMB_OP_VALIDITY_ONLY ? nullptr : out->d_values;
  job.out_validity = out->d_bitmap;
  job.out_valid_bytes = out->d_valid_bytes;
  job.null_count = out->d_null_count;
  job.op = op;
  job.param = param;
  if (check_cuda(cudaStreamWaitEvent(c.s_compute, col.ev_staged, 0), "wait staged")) return -1;
  void *jd = upload_job(sc, &job, sizeof(job));
  if (!jd) return -1;
  cudaEvent_t k0 = sc.event(true), k1 = sc.event(true);
  if (!k0 || !k1) return -1;
  cudaEventRecord(k0, c.s_compute);
  if (dmb_dev_fixed_batch((const dmb_fixed_job *)jd, &job, 1, r->d_counts, r->d_row_off, r->nchunks, n, c.s_compute)) return -1;
  cudaEventRecord(k1, c.s_compute);
  sc.kernel_spans.emplace_back(k0, k1);
  out->done = k1;
  return 0;
}

struct StringRun {
  void *d_offsets = nullptr;
  size_t offsets_bytes = 0;
  uint8_t *d_data = nullptr;
  size_t data_cap = 0;
  FixedRun validity;  // bitmap / valid bytes / null count come from the fixed kernel's tile phase
  void *d_scratch = nullptr;
  unsigned long long *d_total = nullptr;
  unsigned long long *h_ctr = nullptr;  // pinned: [0] total bytes [1] error flags [2] null count [3] ENUM indices past the dictionary
  int mode = 0;
  bool exact = false;          // data_cap was sized from a first launch's total
  cudaEvent_t done = nullptr;  // kernel + the small counter copies
};

// where the string kernel reads a column from: the staged VARCHAR / BLOB column itself, or the text
// rendering of a fixed-width column (kernels_render.cu) produced on the compute stream
struct StringSource {
  const dmb_string_t *in = nullptr;
  const dmb_vec_desc *vecs = nullptr;
  const uint8_t *heap = nullptr;
  uint64_t heap_host_base = 0, heap_len = 0;
  const unsigned long long *d_bad = nullptr;  // ENUM: device count of indices past the dictionary
  size_t max_row_bytes = 0;                   // ENUM: longest label
  bool fused_enum = false;                    // ENUM with a small dictionary of short labels: indices -> utf8 in one launch (dmb_dev_enum_utf8)
  dmb_enum_job ejob{};
  // a source that is not laid out in the result's chunks (BLOB text: dense rows cut into 2048-row pseudo chunks)
  const uint32_t *counts = nullptr;
  const int64_t *row_off = nullptr;
  const uint64_t *validity = nullptr;
  int64_t nchunks = -1;
};

int32_t run_string(Result *r, Scope &sc, int j, int mode, bool want_bitmap, bool want_valid_bytes, struct StringRun *out, size_t exact_cap, bool as_text);

// a column whose VARCHAR form the device produces: strings, the rendered scalar types, ENUM with its dictionary
bool text_supported(const Col &col) {
  if (col.phys == DMB_PHYS_STRING) return true;
  if (col.type_id == DMB_TYPE_ENUM) return col.dict != nullptr;
  return dmb_render_supported(col.type_id, col.phys) != 0;
}

// BLOB as text (getters, per-cell symbols, typed Value::String): the VARCHAR cast escapes the bytes.  Pass 1 turns the
// column into its dense raw form (offsets + data), the escape kernel writes one string_t per row over a 4x heap, and the
// caller's string pass runs over those rows as 2048-row pseudo chunks with pass 1's bitmap as their masks.
int32_t blob_text_source(Result *r, Scope &sc, int j, StringSource *src);

int32_t string_source(Result *r, Scope &sc, int j, bool arrow_mode, bool as_text, StringSource *src) {
  if (stage_column(r, j)) return -1;
  CtxCore &c = *r->core;
  Col &col = r->cols[(size_t)j];
  if (col.phys == DMB_PHYS_STRING && col.type_id == DMB_TYPE_BLOB && as_text) return blob_text_source(r, sc, j, src);
  if (col.phys == DMB_PHYS_STRING) {
    src->in = (const dmb_string_t *)col.d_data;
    src->vecs = col.d_vecs;
    src->heap = col.d_heap;
    src->heap_host_base = col.heap_host_base;
    src->heap_len = col.d_heap_len;
    return 0;
  }
  if (col.type_id == DMB_TYPE_ENUM && col.dict) {
    // indices -> string_t into the dictionary (kernels_enum.cu); the dictionary bytes are the string heap
    EnumDict &d = *col.dict;
    const int64_t nch = r->nchunks;
    const size_t nslots = (size_t)(nch > 0 ? nch : 1) * DMB_VECTOR_SIZE;
    if (!d.d_offsets) {
      d.d_offsets = (uint32_t *)keep_dev(r, d.offsets.size() * sizeof(uint32_t));
      d.d_data = (uint8_t *)keep_dev(r, d.data.size() + 64);
      if (!d.d_offsets || !d.d_data) return -1;
      // once per result, through a pinned copy on the stream of the kernels that read it (a pageable cudaMemcpy on the
      // legacy stream is not ordered with the non-blocking compute stream)
      const size_t ob = d.offsets.size() * sizeof(uint32_t);
      uint8_t *hp = (uint8_t *)keep_pin(r, ob + d.data.size());
      if (!hp) return -1;
      memcpy(hp, d.offsets.data(), ob);
      if (!d.data.empty()) memcpy(hp + ob, d.data.data(), d.data.size());
      if (check_cuda(cudaMemcpyAsync(d.d_offsets, hp, ob, cudaMemcpyHostToDevice, c.s_compute), "enum dictionary offsets H2D")) return -1;
      if (!d.data.empty() && check_cuda(cudaMemcpyAsync(d.d_data, hp + ob, d.data.size(), cudaMemcpyHostToDevice, c.s_compute), "enum dictionary data H2D")) return -1;
      r->bytes_h2d += d.offsets.size() * sizeof(uint32_t) + d.data.size();
    }
    // one fused launch (indices -> utf8) when the dictionary fits its label table; otherwise the string_t intermediate
    const bool fused = arrow_mode && d.size() <= DMB_ENUM_FUSED_MAX_LABELS && d.max_len <= 12;
    dmb_string_t *d_str = fused ? nullptr : (dmb_string_t *)sc.dalloc(nslots * sizeof(dmb_string_t));
    unsigned long long *d_bad = (unsigned long long *)sc.dalloc(8);
    std::vector<dmb_vec_desc> vecs((size_t)(nch > 0 ? nch : 1));
    for (int64_t k = 0; k < nch; ++k) {
      vecs[(size_t)k].data_off = (uint64_t)k * DMB_VECTOR_SIZE * sizeof(dmb_string_t);
      vecs[(size_t)k].val_off = (col.any_validity && col.validity[(size_t)k]) ? k * DMB_VALIDITY_WORDS : -1;
    }
    if ((!fused && !d_str) || !d_bad) return -1;
    if (check_cuda(cudaStreamWaitEvent(c.s_compute, col.ev_staged, 0), "wait staged")) return -1;
    dmb_vec_desc *d_vecs2 = fused ? nullptr : (dmb_vec_desc *)upload_job(sc, vecs.data(), sizeof(dmb_vec_desc) * vecs.size());
    if (!fused && !d_vecs2) return -1;
    if (check_cuda(cudaMemsetAsync(d_bad, 0, 8, c.s_compute), "enum counter memset")) return -1;
    dmb_enum_job job;
    memset(&job, 0, sizeof(job));
    job.in_data = col.d_data;
    job.in_validity = col.d_validity;
    job.vecs = col.d_vecs;
    job.out = d_str;
    job.dict_offsets = d.d_offsets;
    job.dict_data = d.d_data;
    job.dict_host_base = 1ull << 41;
    job.bad_index = d_bad;
    job.dict_size = d.size();
    job.phys = col.phys;
    src->fused_enum = fused;
    src->ejob = job;
    if (!fused && dmb_dev_enum_to_string_t(&job, r->d_counts, nch, c.s_compute)) return -1;
    src->in = d_str;
    src->vecs = d_vecs2;
    src->heap = d.d_data;
    src->heap_host_base = job.dict_host_base;
    src->heap_len = d.max_len > 12 ? (uint64_t)d.data.size() : 0;  // labels of <= 12 bytes are all inlined: the heap-less kernel
    src->d_bad = d_bad;
    src->max_row_bytes = d.max_len;
    return 0;
  }
  if (!dmb_render_supported(col.type_id, col.phys)) {
    set_error("column %d (type %d): libduckdb's text rendering of this type is not reproduced on the device", j, col.type_id);
    return -1;
  }
  const int64_t nch = r->nchunks;
  const size_t nslots = (size_t)(nch > 0 ? nch : 1) * DMB_VECTOR_SIZE;
  dmb_string_t *d_str = (dmb_string_t *)sc.dalloc(nslots * sizeof(dmb_string_t));
  const size_t slot_bytes = (size_t)dmb_render_slot_bytes(col.type_id);
  uint8_t *d_heap = (uint8_t *)sc.dalloc(nslots * slot_bytes + 64);
  std::vector<dmb_vec_desc> vecs((size_t)(nch > 0 ? nch : 1));
  for (int64_t k = 0; k < nch; ++k) {
    vecs[(size_t)k].data_off = (uint64_t)k * DMB_VECTOR_SIZE * sizeof(dmb_string_t);
    vecs[(size_t)k].val_off = (col.any_validity && col.validity[(size_t)k]) ? k * DMB_VALIDITY_WORDS : -1;
  }
  if (!d_str || !d_heap) return -1;
  if (check_cuda(cudaStreamWaitEvent(c.s_compute, col.ev_staged, 0), "wait staged")) return -1;
  dmb_vec_desc *d_vecs2 = (dmb_vec_desc *)upload_job(sc, vecs.data(), sizeof(dmb_vec_desc) * vecs.size());
  if (!d_vecs2) return -1;
  dmb_render_job job;
  memset(&job, 0, sizeof(job));
  job.in_data = col.d_data;
  job.in_validity = col.d_validity;
  job.vecs = col.d_vecs;
  job.out = d_str;
  job.out_heap = d_heap;
  job.heap_host_base = 1ull << 40;
  job.type_id = col.type_id;
  job.phys = col.phys;
  job.dec_scale = col.dec_scale;
  if (dmb_dev_render_text(&job, r->d_counts, nch, c.s_compute)) return -1;
  src->in = d_str;
  src->vecs = d_vecs2;
  src->heap = d_heap;
  src->heap_host_base = job.heap_host_base;
  src->heap_len = (uint64_t)nslots * slot_bytes;
  return 0;
}

// exact_cap != 0: the data bytes the column is known to need (a first launch reported them, see kStrFlagDataCap)
// as_text: the column's VARCHAR rendering is wanted (getters, text / typed columns): a BLOB is escaped; false: the Arrow
// export, which keeps BLOB bytes as they are
int32_t run_string(Result *r, Scope &sc, int j, int mode, bool want_bitmap, bool want_valid_bytes, StringRun *out, size_t exact_cap = 0,
                   bool as_text = true) {
  StringSource src;
  if (string_source(r, sc, j, mode != DMB_STR_REF_BLOB, as_text, &src)) return -1;
  CtxCore &c = *r->core;
  Col &col = r->cols[(size_t)j];
  const int64_t n = r->nrows;
  out->mode = mode;
  out->offsets_bytes = (size_t)(n + 1) * (mode == DMB_STR_ARROW_LARGE ? 8 : 4);
  out->d_offsets = sc.dalloc(out->offsets_bytes + 64);
  // rendered text: at most one slot per row; ENUM: at most the longest label per row
  const bool blob_text = src.nchunks >= 0;
  const size_t per_row = col.phys == DMB_PHYS_STRING ? 12 : (col.type_id == DMB_TYPE_ENUM ? (src.max_row_bytes > 12 ? src.max_row_bytes : 12) : (size_t)dmb_render_slot_bytes(col.type_id));
  // (string_t entries may alias heap bytes -- a flattened dictionary vector does -- so this is a first guess, not a bound:
  // the kernels check it and report the exact total, and the caller launches again with exact_cap)
  out->data_cap = per_row * (size_t)n + (col.phys == DMB_PHYS_STRING ? (size_t)(blob_text ? src.heap_len : col.d_heap_len) : 0) + (mode == DMB_STR_REF_BLOB ? (size_t)n : 0);
  if (exact_cap) { out->data_cap = exact_cap; out->exact = true; }
  out->d_data = (uint8_t *)sc.dalloc(out->data_cap + 64);
  out->d_scratch = sc.dalloc(dmb_dev_string_scratch_bytes(blob_text ? src.nchunks : r->nchunks));
  out->d_total = (unsigned long long *)sc.dalloc(8);
  out->h_ctr = (unsigned long long *)sc.palloc(32);
  if (!out->d_offsets || !out->d_data || !out->d_scratch || !out->d_total || !out->h_ctr) return -1;
  memset(out->h_ctr, 0, 32);
  // validity outputs + null count (the count is always needed: the reference blob's length depends on it)
  if (run_fixed(r, sc, j, DMB_OP_VALIDITY_ONLY, 0, want_bitmap, want_valid_bytes, &out->validity)) return -1;
  if (check_cuda(cudaMemsetAsync(out->d_total, 0, 8, c.s_compute), "total memset")) return -1;
  dmb_string_job job;
  memset(&job, 0, sizeof(job));
  job.in = src.in;
  job.in_validity = blob_text ? src.validity : col.d_validity;
  job.vecs = src.vecs;
  job.heap_dev = src.heap;
  job.heap_host_base = src.heap_host_base;
  job.heap_len = src.heap_len;
  job.out_offsets = out->d_offsets;
  job.out_data = out->d_data;
  job.total_bytes = out->d_total;
  job.mode = mode;
  job.out_data_cap = out->data_cap;
  cudaEvent_t k0 = sc.event(true), k1 = sc.event(true), done = sc.event(false);
  if (!k0 || !k1 || !done) return -1;
  cudaEventRecord(k0, c.s_compute);
  if (blob_text ? dmb_dev_string_batch(&job, src.counts, src.row_off, src.nchunks, n, out->d_scratch, c.s_compute)
      : src.fused_enum ? dmb_dev_enum_utf8(&src.ejob, &job, r->d_counts, r->d_row_off, r->nchunks, n, out->d_scratch, c.s_compute)
                       : dmb_dev_string_batch(&job, r->d_counts, r->d_row_off, r->nchunks, n, out->d_scratch, c.s_compute)) return -1;
  cudaEventRecord(k1, c.s_compute);
  sc.kernel_spans.emplace_back(k0, k1);
  // the data length is needed on the host to size the device->host copy; flags travel with it
  if (check_cuda(cudaMemcpyAsync(out->h_ctr + 0, out->d_total, 8, cudaMemcpyDeviceToHost, c.s_compute), "string total D2H")) return -1;
  if (n > 0 && check_cuda(cudaMemcpyAsync(out->h_ctr + 1, (unsigned long long *)out->d_scratch + 1, 8, cudaMemcpyDeviceToHost, c.s_compute), "string flags D2H")) return -1;
  if (check_cuda(cudaMemcpyAsync(out->h_ctr + 2, out->validity.d_null_count, 8, cudaMemcpyDeviceToHost, c.s_compute), "null count D2H")) return -1;
  if (src.d_bad && check_cuda(cudaMemcpyAsync(out->h_ctr + 3, src.d_bad, 8, cudaMemcpyDeviceToHost, c.s_compute), "enum counter D2H")) return -1;
  cudaEventRecord(done, c.s_compute);
  out->done = done;
  return 0;
}

constexpr unsigned long long kStrFlagOverflow = 2, kStrFlagDataCap = 8;  // kernels_string.cu kErr*
int32_t string_flags_error(unsigned long long flags) {
  if (!flags) return 0;
  if (flags & (1ull << 63)) { set_error("ENUM index outside the type's dictionary"); return -1; }
  if (flags & 16) set_error("a string tile's look-back gave up waiting for its predecessors (GPU preempted or oversubscribed?); run the call again");
  else if (flags & 4) set_error("string_t pointer outside the registered heap");
  else if (flags & kStrFlagDataCap) set_error("string bytes exceed the sized output buffer");
  else if (flags & kStrFlagOverflow) set_error("utf8 data exceeds int32 offsets");
  else set_error("a 1024-row tile holds more than 4 GiB of string bytes");
  return -1;
}

// run_string + wait; a column whose strings alias heap bytes overflows the first-guess buffer and is run again, sized exactly
int32_t run_string_sync(Result *r, Scope &sc, int j, int mode, bool want_bitmap, bool want_valid_bytes, StringRun *out) {
  size_t exact = 0;
  for (int attempt = 0; attempt < 2; ++attempt) {
    *out = StringRun();
    if (run_string(r, sc, j, mode, want_bitmap, want_valid_bytes, out, exact)) return -1;
    if (check_cuda(cudaEventSynchronize(out->done), "string kernel wait")) return -1;
    const unsigned long long flags = out->h_ctr[1];
    if ((flags & kStrFlagDataCap) && !(flags & ~(kStrFlagDataCap | kStrFlagOverflow)) && attempt == 0) {
      exact = (size_t)out->h_ctr[0];
      continue;
    }
    return string_flags_error(flags | (out->h_ctr[3] ? (1ull << 63) : 0ull));
  }
  return -1;
}

int32_t blob_text_source(Result *r, Scope &sc, int j, StringSource *src) {
  CtxCore &c = *r->core;
  const int64_t n = r->nrows;
  StringRun raw;  // pass 1: the BLOB bytes, dense (a BLOB column beyond 2 GiB cannot be one getter blob anyway)
  if (run_string(r, sc, j, DMB_STR_ARROW_UTF8, true, false, &raw, 0, /*as_text=*/false)) return -1;
  if (check_cuda(cudaEventSynchronize(raw.done), "blob pass wait")) return -1;
  if ((raw.h_ctr[1] & kStrFlagDataCap) && !(raw.h_ctr[1] & ~kStrFlagDataCap)) {  // aliased pointers: sized exactly, once more
    const size_t exact = (size_t)raw.h_ctr[0];
    raw = StringRun();
    if (run_string(r, sc, j, DMB_STR_ARROW_UTF8, true, false, &raw, exact, false)) return -1;
    if (check_cuda(cudaEventSynchronize(raw.done), "blob pass wait")) return -1;
  }
  if (string_flags_error(raw.h_ctr[1])) return -1;
  const uint64_t total = raw.h_ctr[0];
  const int64_t nck = n > 0 ? (n + DMB_VECTOR_SIZE - 1) / DMB_VECTOR_SIZE : 0;
  const size_t nslots = (size_t)(nck > 0 ? nck : 1) * DMB_VECTOR_SIZE;
  dmb_string_t *d_str = (dmb_string_t *)sc.dalloc(nslots * sizeof(dmb_string_t));
  uint8_t *d_heap = (uint8_t *)sc.dalloc((size_t)total * 4 + 64);
  // the masks of the pseudo chunks: pass 1's bitmap, copied into whole 32-word masks (the kernels fetch whole tiles of mask words)
  uint64_t *d_masks = (uint64_t *)sc.dalloc(nslots / 8 + 64);
  if (!d_str || !d_heap || !d_masks) return -1;
  if (check_cuda(cudaMemsetAsync(d_masks, 0, nslots / 8, c.s_compute), "blob masks memset")) return -1;
  if (raw.validity.bitmap_bytes && check_cuda(cudaMemcpyAsync(d_masks, raw.validity.d_bitmap, raw.validity.bitmap_bytes, cudaMemcpyDeviceToDevice, c.s_compute), "blob masks copy")) return -1;
  if (dmb_dev_blob_escape((const int32_t *)raw.d_offsets, raw.d_data, n, d_str, d_heap, 1ull << 42, c.s_compute)) return -1;
  std::vector<uint32_t> cc((size_t)(nck > 0 ? nck : 1), DMB_VECTOR_SIZE);
  std::vector<int64_t> ro((size_t)nck + 1);
  std::vector<dmb_vec_desc> vd((size_t)(nck > 0 ? nck : 1));
  if (nck) cc[(size_t)nck - 1] = (uint32_t)(n - (nck - 1) * DMB_VECTOR_SIZE);
  for (int64_t k = 0; k < nck; ++k) {
    ro[(size_t)k] = k * (int64_t)DMB_VECTOR_SIZE;
    vd[(size_t)k].data_off = (uint64_t)k * DMB_VECTOR_SIZE * sizeof(dmb_string_t);
    vd[(size_t)k].val_off = k * DMB_VALIDITY_WORDS;
  }
  ro[(size_t)nck] = n;
  src->counts = (const uint32_t *)upload_job(sc, cc.data(), cc.size() * sizeof(uint32_t));
  src->row_off = (const int64_t *)upload_job(sc, ro.data(), ro.size() * sizeof(int64_t));
  src->vecs = (const dmb_vec_desc *)upload_job(sc, vd.data(), vd.size() * sizeof(dmb_vec_desc));
  if (!src->counts || !src->row_off || !src->vecs) return -1;
  src->in = d_str;
  src->heap = d_heap;
  src->heap_host_base = 1ull << 42;
  src->heap_len = total * 4;
  src->validity = d_masks;
  src->nchunks = nck;
  return 0;
}

// ------------------------------------------------------------------ DuckDB type -> Arrow
struct ArrowMap {
  int32_t op = -1;      // fixed-width conversion, or -1 for strings
  bool is_string = false;
  bool is_list = false;    // LIST of one fixed-width leaf: pipelined (run_list)
  bool is_nested = false;  // STRUCT / MAP / every other LIST: converted synchronously (nested_to_arrow)
  std::string format, child_format;
  int32_t child_op = -1;
};

// the scalar and string types; the caller maps ENUM, STRUCT, MAP and LIST, which need more than the type
bool type_arrow_map(const ColType &col, ArrowMap *m) {
  char buf[48];
  auto same = [&](const char *fmt) { m->op = DMB_OP(col.phys, DMB_DST_SAME); m->format = fmt; return true; };
  switch (col.type_id) {
    case DMB_TYPE_BOOLEAN: m->op = DMB_OP(DMB_PHYS_BOOL, DMB_DST_BOOL_BITS); m->format = "b"; return true;
    case DMB_TYPE_TINYINT: return same("c");
    case DMB_TYPE_SMALLINT: return same("s");
    case DMB_TYPE_INTEGER: return same("i");
    case DMB_TYPE_BIGINT: return same("l");
    case DMB_TYPE_UTINYINT: return same("C");
    case DMB_TYPE_USMALLINT: return same("S");
    case DMB_TYPE_UINTEGER: return same("I");
    case DMB_TYPE_UBIGINT: return same("L");
    case DMB_TYPE_FLOAT: return same("f");
    case DMB_TYPE_DOUBLE: return same("g");
    case DMB_TYPE_DATE: return same("tdD");
    case DMB_TYPE_TIME: return same("ttu");
    case DMB_TYPE_TIME_NS: return same("ttn");
    case DMB_TYPE_TIME_TZ: return same("L");  // packed micros|offset bits, as stored
    case DMB_TYPE_TIMESTAMP: return same("tsu:");
    case DMB_TYPE_TIMESTAMP_TZ: return same("tsu:UTC");
    case DMB_TYPE_TIMESTAMP_S: return same("tss:");
    case DMB_TYPE_TIMESTAMP_MS: return same("tsm:");
    case DMB_TYPE_TIMESTAMP_NS: return same("tsn:");
    case DMB_TYPE_INTERVAL: m->op = DMB_OP(DMB_PHYS_INTERVAL, DMB_DST_MONTH_DAY_NANO); m->format = "tin"; return true;
    case DMB_TYPE_HUGEINT: m->op = DMB_OP(DMB_PHYS_I128, DMB_DST_I128); m->format = "d:38,0"; return true;
    case DMB_TYPE_UHUGEINT:
    case DMB_TYPE_UUID: m->op = DMB_OP(DMB_PHYS_U128, DMB_DST_SAME); m->format = "w:16"; return true;
    case DMB_TYPE_DECIMAL:
      m->op = DMB_OP(col.phys, DMB_DST_I128);
      snprintf(buf, sizeof(buf), "d:%d,%d", col.dec_width > 0 ? col.dec_width : 38, col.dec_scale);
      m->format = buf;
      return true;
    case DMB_TYPE_VARCHAR: m->is_string = true; m->format = "u"; return true;
    case DMB_TYPE_BLOB: m->is_string = true; m->format = "z"; return true;
    default: set_error("column type %d has no Arrow mapping", col.type_id); return false;
  }
}

// Arrow keeps these as DuckDB stores them: a gathered LIST child needs no second pass
bool stored_as_arrow(const ColType &t, int32_t op) { return op == DMB_OP(t.phys, DMB_DST_SAME) || t.type_id == DMB_TYPE_HUGEINT; }

bool arrow_map(const Col &col, ArrowMap *m) {
  switch (col.type_id) {
    case DMB_TYPE_ENUM:  // dictionary-encoded: the indices as stored, the labels as the dictionary (export_column)
      if (!col.dict) { set_error("ENUM column without a dictionary"); return false; }
      m->op = DMB_OP(col.phys, DMB_DST_SAME);
      m->format = col.phys == DMB_PHYS_U8 ? "C" : col.phys == DMB_PHYS_U16 ? "S" : "I";
      return true;
    case DMB_TYPE_STRUCT:
      if (!col.is_struct) { set_error("STRUCT column without field vectors"); return false; }
      m->is_nested = true;
      m->format = "+s";
      return true;
    case DMB_TYPE_MAP:
      if (!col.node || col.node->kind != ListNode::kStruct || col.node->leaves.size() != 2) { set_error("MAP column: the child must be STRUCT<key, value>"); return false; }
      m->is_nested = true;
      m->format = "+m";
      return true;
    case DMB_TYPE_LIST: {  // (fill_column gives every LIST column its node)
      m->format = "+l";
      const ListNode &node = *col.node;
      if (node.kind != ListNode::kLeaf || node.leaves[0].phys == DMB_PHYS_STRING) { m->is_nested = true; return true; }
      // one fixed-width leaf: a flat child may have any fixed-width type, and one without an Arrow mapping fails here,
      // at export, so that the result's other columns still serve
      const Leaf &leaf = node.leaves[0];
      ArrowMap cm;
      if (!type_arrow_map(leaf, &cm) || cm.is_string) { set_error("LIST child type %d has no Arrow mapping here", leaf.type_id); return false; }
      m->is_list = true;
      m->child_op = cm.op;
      m->child_format = cm.format;
      return true;
    }
    default: return type_arrow_map(col, m);
  }
}


// ------------------------------------------------------------------ nested types: STRUCT, MAP, LIST
// (SURVEY.md 8f item 3; the reference rejects them on its chunk path, src/duckdb_native.c:271-303, and has no Arrow
// mapping: the contract is the Arrow format, checked with pyarrow in tests/test_gpu_nested.py.)
//   STRUCT          the fields are columns of their own (hidden behind the visible ones): each is converted like a
//                   top-level column; the parent contributes its validity bitmap
//   LIST<x>         a ListNode, whether dmb_host_list gave the child in its flat fixed-width fields or as child_col.
//                   Level by level on DENSE arrays: list_emit_kernel gathers every leaf vector family of the child
//                   level through the entries (one launch per leaf: offsets are recomputed, the entries are tiny next
//                   to the children); a gathered leaf is a dense column, so
//                     fixed width     -> its Arrow form (second pass of fixed_batch_kernel when it is not stored that way)
//                     VARCHAR / BLOB  -> the string kernels over the gathered string_t as 2048-element pseudo chunks,
//                                        the child vectors' heaps gathered into one arena by the stager
//                     STRUCT          -> every field gathered with the same entries (+ the struct's own validity)
//                     LIST            -> the gathered inner entries (rebased onto the grandchild slab by the stager) are
//                                        the entries of the next level: the same kernel again, over pseudo chunks
//   MAP             LIST<STRUCT<key, value>> exported as Arrow map<key, value>
// A top-level LIST of one fixed-width leaf runs in materialise_arrow's pipeline (run_list: its copy-in, kernels and
// copy-out overlap the neighbouring columns').  Every other nested column is converted synchronously inside
// launch_arrow_col (nested_to_arrow: no copy-in / copy-out overlap).
void copy_bits(uint64_t *dst, uint64_t dst_bit, const uint64_t *src, uint64_t nbits) {  // src bits [0, nbits) -> dst bits [dst_bit, ...); dst pre-zeroed
  for (uint64_t i = 0; i < nbits;) {
    const uint64_t d = dst_bit + i;
    const unsigned take = (unsigned)std::min<uint64_t>(std::min<uint64_t>(64 - (d & 63), 64 - (i & 63)), nbits - i);
    uint64_t bits = src ? (src[i >> 6] >> (i & 63)) : ~0ull;
    if (take < 64) bits &= (1ull << take) - 1ull;
    dst[d >> 6] |= bits << (d & 63);
    i += take;
  }
}

bool leaf_from_column(const dmb_host_column &hc, int64_t nch, Leaf *leaf) {
  leaf->name = hc.name ? hc.name : "";
  leaf->type_id = hc.type_id;
  leaf->phys = hc.phys;
  leaf->dec_width = hc.dec_width;
  leaf->dec_scale = hc.dec_scale;
  leaf->width = dmb_phys_width(hc.phys);
  if (leaf->width <= 0) { set_error("nested column '%s': bad physical type %d", leaf->name.c_str(), hc.phys); return false; }
  if (nch > 0 && !hc.data) { set_error("nested column '%s': no data pointers", leaf->name.c_str()); return false; }
  leaf->data.assign(hc.data, hc.data + nch);
  if (hc.validity) {
    leaf->validity.assign((const void *const *)hc.validity, (const void *const *)hc.validity + nch);
    bool any = false;
    for (const void *p : leaf->validity) any |= p != nullptr;
    if (!any) leaf->validity.clear();
  }
  return true;
}

// the flat form of a list's child (child_type_id ... child_validity) as a column of its own
dmb_host_column flat_child(const dmb_host_list &l) {
  dmb_host_column f;
  memset(&f, 0, sizeof(f));
  f.name = "item";
  f.type_id = l.child_type_id;
  f.phys = l.child_phys;
  f.dec_width = l.child_dec_width;
  f.dec_scale = l.child_dec_scale;
  f.data = l.child_data;
  f.validity = l.child_validity;
  return f;
}

// a node's per-chunk child sizes and their running sum
std::shared_ptr<ListNode> sized_node(const uint64_t *sizes, int64_t nch) {
  auto node = std::make_shared<ListNode>();
  node->sizes.assign(sizes, sizes + nch);
  node->base.assign((size_t)nch + 1, 0);
  for (int64_t k = 0; k < nch; ++k) node->base[(size_t)k + 1] = node->base[(size_t)k] + node->sizes[(size_t)k];
  return node;
}

// the child level of a LIST / MAP from its host description (dmb_host_list with child_col)
std::shared_ptr<ListNode> build_node(const dmb_host_list *l, int64_t nch, int depth) {
  if (depth > 4) { set_error("LIST nesting deeper than 4 levels"); return nullptr; }
  const dmb_host_column *cc = l->child_col;
  if (!cc || (nch > 0 && !l->child_sizes)) { set_error("LIST column: child_col / child_sizes missing"); return nullptr; }
  auto node = sized_node(l->child_sizes, nch);
  auto add_leaf = [&](const dmb_host_column &hc) {
    if (hc.type_id == DMB_TYPE_ENUM) { set_error("nested column '%s': ENUM inside LIST / MAP is not supported", hc.name ? hc.name : ""); return false; }
    node->leaves.emplace_back();
    return leaf_from_column(hc, nch, &node->leaves.back());
  };
  if (cc->type_id == DMB_TYPE_STRUCT) {
    if (!cc->struct_ || cc->struct_->nfields <= 0 || !cc->struct_->fields) { set_error("LIST<STRUCT>: no fields"); return nullptr; }
    node->kind = ListNode::kStruct;
    for (int32_t f = 0; f < cc->struct_->nfields; ++f) {
      const dmb_host_column &fc = cc->struct_->fields[f];
      if (fc.type_id == DMB_TYPE_STRUCT || fc.type_id == DMB_TYPE_LIST || fc.type_id == DMB_TYPE_MAP) { set_error("LIST<STRUCT>: field '%s' is itself nested (not supported)", fc.name ? fc.name : ""); return nullptr; }
      if (!add_leaf(fc)) return nullptr;
    }
    if (cc->validity) {
      node->struct_validity.validity.assign((const void *const *)cc->validity, (const void *const *)cc->validity + nch);
      for (const void *p : node->struct_validity.validity) node->has_struct_validity |= p != nullptr;
    }
    node->struct_validity.width = 1;
    node->struct_validity.phys = DMB_PHYS_U8;
    node->struct_validity.type_id = DMB_TYPE_UTINYINT;
  } else if (cc->type_id == DMB_TYPE_LIST) {
    if (!cc->list) { set_error("LIST<LIST>: the inner list's child vectors are missing"); return nullptr; }
    node->kind = ListNode::kList;
    dmb_host_column entries = *cc;
    entries.phys = DMB_PHYS_U128;
    if (!add_leaf(entries)) return nullptr;
    dmb_host_list inner = *cc->list;
    const dmb_host_column flat = flat_child(inner);
    if (!inner.child_col) inner.child_col = &flat;
    node->inner = build_node(&inner, nch, depth + 1);
    if (!node->inner) return nullptr;
  } else {
    node->kind = ListNode::kLeaf;
    if (!add_leaf(*cc)) return nullptr;
  }
  return node;
}

// chunks [c0, c1) of a node (slice_result)
std::shared_ptr<ListNode> slice_node(const ListNode &p, int64_t c0, int64_t c1) {
  auto n = sized_node(p.sizes.data() + c0, c1 - c0);
  n->kind = p.kind;
  auto slice_leaf = [&](const Leaf &pl) {
    Leaf l;
    static_cast<ColType &>(l) = pl;
    if (!pl.data.empty()) l.data.assign(pl.data.begin() + c0, pl.data.begin() + c1);
    if (!pl.validity.empty()) l.validity.assign(pl.validity.begin() + c0, pl.validity.begin() + c1);
    return l;
  };
  for (const Leaf &pl : p.leaves) n->leaves.push_back(slice_leaf(pl));
  n->struct_validity = slice_leaf(p.struct_validity);
  n->has_struct_validity = p.has_struct_validity;
  if (p.inner) n->inner = slice_node(*p.inner, c0, c1);
  return n;
}

// host -> device: every leaf of the node as one flat slab.  dense_bits: the validity as ONE bitmap over the slab (levels
// below the first: their entries were rebased onto the slab), else one padded mask per chunk.
int32_t stage_node(Result *r, ListNode &node, bool dense_bits) {
  if (node.staged) return 0;
  CtxCore &c = *r->core;
  const int64_t nch = r->nchunks;
  const uint64_t total = node.base[(size_t)nch];
  uint64_t *h_base = (uint64_t *)keep_pin(r, (size_t)(nch + 1) * 8), *h_sizes = (uint64_t *)keep_pin(r, (size_t)(nch + 1) * 8);
  node.d_base = (uint64_t *)keep_dev(r, (size_t)(nch + 1) * 8);
  node.d_sizes = (uint64_t *)keep_dev(r, (size_t)(nch + 1) * 8);
  if (!h_base || !h_sizes || !node.d_base || !node.d_sizes) return -1;
  memcpy(h_base, node.base.data(), (size_t)(nch + 1) * 8);
  if (nch) memcpy(h_sizes, node.sizes.data(), (size_t)nch * 8);
  if (check_cuda(cudaMemcpyAsync(node.d_base, h_base, (size_t)(nch + 1) * 8, cudaMemcpyHostToDevice, c.s_in), "list child base H2D")) return -1;
  if (nch && check_cuda(cudaMemcpyAsync(node.d_sizes, h_sizes, (size_t)nch * 8, cudaMemcpyHostToDevice, c.s_in), "list child sizes H2D")) return -1;
  auto stage_leaf = [&](Leaf &leaf, bool zero_payload, const ListNode *rebase_onto) -> int32_t {
    const size_t W = (size_t)leaf.width;
    uint8_t *arena = (uint8_t *)keep_pin(r, (size_t)total * W + 64);
    leaf.d_data = (uint8_t *)keep_dev(r, (size_t)total * W + 64);
    if (!arena || !leaf.d_data) return -1;
    if (zero_payload) memset(arena, 0, (size_t)total * W);
    // validity
    std::vector<int64_t> voff((size_t)(nch > 0 ? nch : 1), -1);
    uint64_t words = 0;
    const bool any_mask = !leaf.validity.empty();
    if (dense_bits) words = any_mask ? (total + 63) / 64 + 2 : 0;
    else
      for (int64_t k = 0; k < nch; ++k)
        if (any_mask && leaf.validity[(size_t)k]) { voff[(size_t)k] = (int64_t)words; words += (node.sizes[(size_t)k] + 63) / 64 + 1; }
    uint64_t *warena = words ? (uint64_t *)keep_pin(r, (size_t)(words + 2) * 8) : nullptr;
    if (words) {
      leaf.d_validity = (uint64_t *)keep_dev(r, (size_t)(words + 2) * 8);
      if (!warena || !leaf.d_validity) return -1;
      memset(warena, 0, (size_t)(words + 2) * 8);
    }
    // strings: where chunk k's heap bytes go in the arena (size pass), then gather + pointer rewrite
    const bool is_string = leaf.phys == DMB_PHYS_STRING;
    std::vector<uint64_t> hstart;
    uint8_t *harena = nullptr;
    const uint64_t fake_base = 1ull << 43;
    if (is_string) {
      hstart.assign((size_t)nch + 1, 0);
      parallel_for(c, nch, [&](int64_t k) {
        const dmb_string_t *e = reinterpret_cast<const dmb_string_t *>(leaf.data[(size_t)k]);
        const void *mask = any_mask ? leaf.validity[(size_t)k] : nullptr;
        uint64_t sum = 0;
        for (uint64_t i = 0; e && i < node.sizes[(size_t)k]; ++i)
          if (host_row_valid(mask, (uint32_t)i) && e[i].length > 12) sum += e[i].length;
        hstart[(size_t)k + 1] = sum;
      });
      for (int64_t k = 0; k < nch; ++k) hstart[(size_t)k + 1] += hstart[(size_t)k];
      leaf.heap_len = hstart[(size_t)nch];
      harena = (uint8_t *)keep_pin(r, (size_t)leaf.heap_len + 32);
      leaf.d_heap = (uint8_t *)keep_dev(r, (size_t)leaf.heap_len + 32);
      if (!harena || !leaf.d_heap) return -1;
    }
    parallel_for(c, nch, [&](int64_t k) {
      const uint64_t sz = node.sizes[(size_t)k];
      uint8_t *dst = arena + (size_t)node.base[(size_t)k] * W;
      if (sz && !zero_payload) memcpy(dst, leaf.data[(size_t)k], (size_t)sz * W);
      const void *mask = any_mask ? leaf.validity[(size_t)k] : nullptr;
      if (rebase_onto) {  // inner list entries: offsets become positions in the grandchild slab
        uint64_t *e = reinterpret_cast<uint64_t *>(dst);
        const uint64_t add = rebase_onto->base[(size_t)k];
        for (uint64_t i = 0; i < sz; ++i) e[2 * i] += add;
      }
      if (is_string) {
        dmb_string_t *e = reinterpret_cast<dmb_string_t *>(dst);
        uint64_t pos = hstart[(size_t)k];
        for (uint64_t i = 0; i < sz; ++i) {
          if (!host_row_valid(mask, (uint32_t)i) || e[i].length <= 12) continue;
          memcpy(harena + pos, reinterpret_cast<const void *>((uintptr_t)e[i].tail.ptr), e[i].length);
          e[i].tail.ptr = fake_base + pos;
          pos += e[i].length;
        }
      }
      if (words && !dense_bits && voff[(size_t)k] >= 0) memcpy(warena + voff[(size_t)k], mask, (size_t)((sz + 63) / 64) * 8);
    });
    if (words && dense_bits)  // (serial: neighbouring chunks share words)
      for (int64_t k = 0; k < nch; ++k)
        copy_bits(warena, node.base[(size_t)k], reinterpret_cast<const uint64_t *>(leaf.validity[(size_t)k]), node.sizes[(size_t)k]);
    if (total && check_cuda(cudaMemcpyAsync(leaf.d_data, arena, (size_t)total * W, cudaMemcpyHostToDevice, c.s_in), "nested child H2D")) return -1;
    if (words && check_cuda(cudaMemcpyAsync(leaf.d_validity, warena, (size_t)words * 8, cudaMemcpyHostToDevice, c.s_in), "nested child masks H2D")) return -1;
    if (!dense_bits) {
      int64_t *h_voff = (int64_t *)keep_pin(r, (size_t)(nch + 1) * 8);
      leaf.d_val_off = (int64_t *)keep_dev(r, (size_t)(nch + 1) * 8);
      if (!h_voff || !leaf.d_val_off) return -1;
      if (nch) memcpy(h_voff, voff.data(), (size_t)nch * 8);
      if (nch && check_cuda(cudaMemcpyAsync(leaf.d_val_off, h_voff, (size_t)nch * 8, cudaMemcpyHostToDevice, c.s_in), "nested child mask offsets H2D")) return -1;
    }
    if (is_string && leaf.heap_len && check_cuda(cudaMemcpyAsync(leaf.d_heap, harena, (size_t)leaf.heap_len, cudaMemcpyHostToDevice, c.s_in), "nested child heap H2D")) return -1;
    r->bytes_h2d += total * W + words * 8 + leaf.heap_len;
    return 0;
  };
  for (Leaf &leaf : node.leaves)
    if (stage_leaf(leaf, false, node.kind == ListNode::kList ? node.inner.get() : nullptr)) return -1;
  if (node.kind == ListNode::kStruct && node.has_struct_validity && stage_leaf(node.struct_validity, true, nullptr)) return -1;
  if (node.inner && stage_node(r, *node.inner, true)) return -1;
  node.staged = true;
  return 0;
}

// the entries a gather reads: the LIST column's own vectors, or (levels below) the dense inner entries as pseudo chunks
struct EntrySrc {
  const void *d_entries = nullptr;
  const uint64_t *d_validity = nullptr;
  const dmb_vec_desc *d_vecs = nullptr;
  const uint32_t *d_counts = nullptr;
  const int64_t *d_row_off = nullptr;
  int64_t nchunks = 0, nrows = 0;
  const uint64_t *d_child_base = nullptr, *d_child_sizes = nullptr;
  uint64_t cap = 0;  // elements the gather produces (host pass)
  bool dense_bits = false;
};
struct GatherOut {
  void *d_offsets = nullptr;
  uint8_t *d_child = nullptr;
  uint64_t *d_bitmap = nullptr;  // whole 32-word masks: the next pass reads it as chunk masks
  unsigned long long *h_ctr = nullptr;  // pinned: [0] elements [1] nulls [2] flags [3] the parent's null count (run_list)
  cudaEvent_t done = nullptr;
};

// the entries of a LIST / MAP column itself, over its node's child slab
EntrySrc column_entries(const Result *r, const Col &col, uint64_t cap) {
  EntrySrc es;
  es.d_entries = col.d_data;
  es.d_validity = col.d_validity;
  es.d_vecs = col.d_vecs;
  es.d_counts = r->d_counts;
  es.d_row_off = r->d_row_off;
  es.nchunks = r->nchunks;
  es.nrows = r->nrows;
  es.d_child_base = col.node->d_base;
  es.d_child_sizes = col.node->d_sizes;
  es.cap = cap;
  return es;
}

// metadata of a dense array of n elements cut into 2048-element pseudo chunks (masks: words [32 k, 32 k + 32) of a bitmap)
struct Pseudo {
  const uint32_t *d_counts = nullptr;
  const int64_t *d_row_off = nullptr;
  const dmb_vec_desc *d_vecs = nullptr;
  int64_t nchunks = 0;
};
int32_t make_pseudo(Scope &sc, uint64_t n, size_t elem_bytes, Pseudo *out) {
  const int64_t nck = (int64_t)((n + DMB_VECTOR_SIZE - 1) / DMB_VECTOR_SIZE);
  std::vector<uint32_t> cc((size_t)(nck > 0 ? nck : 1), DMB_VECTOR_SIZE);
  std::vector<int64_t> ro((size_t)nck + 1);
  std::vector<dmb_vec_desc> vd((size_t)(nck > 0 ? nck : 1));
  if (nck) cc[(size_t)nck - 1] = (uint32_t)(n - (uint64_t)(nck - 1) * DMB_VECTOR_SIZE);
  for (int64_t k = 0; k < nck; ++k) {
    ro[(size_t)k] = k * (int64_t)DMB_VECTOR_SIZE;
    vd[(size_t)k].data_off = (uint64_t)k * DMB_VECTOR_SIZE * elem_bytes;
    vd[(size_t)k].val_off = k * DMB_VALIDITY_WORDS;
  }
  ro[(size_t)nck] = (int64_t)n;
  out->d_counts = (const uint32_t *)upload_job(sc, cc.data(), cc.size() * sizeof(uint32_t));
  out->d_row_off = (const int64_t *)upload_job(sc, ro.data(), ro.size() * sizeof(int64_t));
  out->d_vecs = (const dmb_vec_desc *)upload_job(sc, vd.data(), vd.size() * sizeof(dmb_vec_desc));
  out->nchunks = nck;
  return (out->d_counts && out->d_row_off && out->d_vecs) ? 0 : -1;
}

int32_t gather_leaf(Result *r, Scope &sc, const EntrySrc &es, const Leaf &leaf, GatherOut *out) {
  CtxCore &c = *r->core;
  const uint64_t cap = es.cap;
  if (cap > 0x7fffffffull) { set_error("nested column: %llu child elements exceed int32 offsets; use smaller batches", (unsigned long long)cap); return -1; }
  out->d_offsets = sc.dalloc((size_t)(es.nrows + 1) * 4 + 64);
  out->d_child = (uint8_t *)sc.dalloc((size_t)cap * (size_t)leaf.width + 64);
  const size_t bm_words = (size_t)((cap + DMB_VECTOR_SIZE - 1) / DMB_VECTOR_SIZE * DMB_VALIDITY_WORDS + 2);
  out->d_bitmap = (uint64_t *)sc.dalloc(bm_words * 8 + 256);
  unsigned long long *d_ctr = (unsigned long long *)sc.dalloc(16);
  void *d_scratch = sc.dalloc(dmb_dev_list_scratch_bytes(es.nchunks) + 16);
  out->h_ctr = (unsigned long long *)sc.palloc(32);
  out->done = sc.event(false);
  if (!out->d_offsets || !out->d_child || !out->d_bitmap || !d_ctr || !d_scratch || !out->h_ctr || !out->done) return -1;
  memset(out->h_ctr, 0, 32);
  if (check_cuda(cudaMemsetAsync(out->d_bitmap, 0, bm_words * 8 + 256, c.s_compute), "nested bitmap memset")) return -1;
  if (es.nrows == 0) {
    if (check_cuda(cudaMemsetAsync(out->d_offsets, 0, 4, c.s_compute), "nested offsets memset")) return -1;
    cudaEventRecord(out->done, c.s_compute);
    return 0;
  }
  if (check_cuda(cudaMemsetAsync(d_ctr, 0, 16, c.s_compute), "nested counters memset")) return -1;
  dmb_list_job job;
  memset(&job, 0, sizeof(job));
  job.in_entries = es.d_entries;
  job.in_validity = es.d_validity;
  job.vecs = es.d_vecs;
  job.child_base = es.d_child_base;
  job.child_data = leaf.d_data;
  job.child_validity = leaf.d_validity;
  job.child_val_off = leaf.d_val_off;
  job.out_offsets = out->d_offsets;
  job.out_child = out->d_child;
  job.out_child_validity = out->d_bitmap;
  job.total = d_ctr;
  job.child_null_count = d_ctr + 1;
  job.child_width = leaf.width;
  job.large = es.dense_bits ? DMB_LIST_DENSE_CHILD_BITS : 0;
  job.child_sizes = es.d_child_sizes;
  cudaEvent_t k0 = sc.event(true), k1 = sc.event(true);
  if (!k0 || !k1) return -1;
  cudaEventRecord(k0, c.s_compute);
  if (dmb_dev_list_batch(&job, es.d_counts, es.d_row_off, es.nchunks, es.nrows, (int64_t)cap, d_scratch, c.s_compute)) return -1;
  cudaEventRecord(k1, c.s_compute);
  sc.kernel_spans.emplace_back(k0, k1);
  if (check_cuda(cudaMemcpyAsync(out->h_ctr, d_ctr, 16, cudaMemcpyDeviceToHost, c.s_compute), "nested counters D2H")) return -1;
  if (check_cuda(cudaMemcpyAsync(out->h_ctr + 2, d_scratch, 8, cudaMemcpyDeviceToHost, c.s_compute), "nested flags D2H")) return -1;
  cudaEventRecord(out->done, c.s_compute);
  return 0;
}

// waits for a gather and decodes list_emit_kernel's error flags (every LIST path)
int32_t check_gather(const GatherOut &g, uint64_t cap) {
  if (check_cuda(cudaEventSynchronize(g.done), "list gather wait")) return -1;
  const unsigned long long f = g.h_ctr[2];
  if (f & 8ull) { set_error("a LIST entry reaches outside its chunk's child vector (offset + length > duckdb_list_vector_get_size)"); return -1; }
  if (f & 4ull) { set_error("a LIST chunk's look-back gave up waiting for its predecessors (GPU preempted or oversubscribed?); run the call again"); return -1; }
  if (f & 2ull) { set_error("a LIST chunk holds more than 4 G child elements"); return -1; }
  if (f & 1ull) { set_error("LIST child elements exceed int32 offsets; use smaller batches"); return -1; }
  if (g.h_ctr[0] != cap) { set_error("LIST column: the device gathered %llu child elements, the host counted %llu", g.h_ctr[0], (unsigned long long)cap); return -1; }
  return 0;
}

// a gathered fixed-width leaf that Arrow stores differently (BOOLEAN -> bits, DECIMAL -> decimal128, INTERVAL ->
// month_day_nano; `cap` > 0 elements): fixed_batch_kernel over the dense child as 2048-element pseudo chunks, the gathered
// bitmap as their masks.  Returns the converted values (*bytes of them) on the compute stream.
uint8_t *convert_gathered(Scope &sc, const Leaf &leaf, const GatherOut &g, uint64_t cap, int32_t op, size_t *bytes) {
  const int32_t ow = dmb_op_out_width(op);
  if (ow < 0) { set_error("LIST child '%s': unsupported conversion 0x%x", leaf.name.c_str(), op); return nullptr; }
  Pseudo ps;
  if (make_pseudo(sc, cap, (size_t)leaf.width, &ps)) return nullptr;
  *bytes = ow == 0 ? (size_t)((cap + 7) / 8) : (size_t)cap * (size_t)ow;
  uint8_t *d_out = (uint8_t *)sc.dalloc(*bytes + 64);
  if (!d_out) return nullptr;
  dmb_fixed_job fj;
  memset(&fj, 0, sizeof(fj));
  fj.in_data = g.d_child;
  fj.in_validity = g.d_bitmap;
  fj.vecs = ps.d_vecs;
  fj.out_values = d_out;
  fj.op = op;
  void *fjd = upload_job(sc, &fj, sizeof(fj));
  cudaEvent_t k0 = sc.event(true), k1 = sc.event(true);
  if (!fjd || !k0 || !k1) return nullptr;
  cudaEventRecord(k0, sc.c.s_compute);
  if (dmb_dev_fixed_batch((const dmb_fixed_job *)fjd, &fj, 1, ps.d_counts, ps.d_row_off, ps.nchunks, (int64_t)cap, sc.c.s_compute)) return nullptr;
  cudaEventRecord(k1, sc.c.s_compute);
  sc.kernel_spans.emplace_back(k0, k1);
  return d_out;
}

// a gathered leaf (dense, `cap` elements) -> its Arrow array in pinned memory.  Synchronous.
std::shared_ptr<ArrowColOut> leaf_to_arrow(Result *r, Scope &sc, const Leaf &leaf, const GatherOut &g, uint64_t cap);

std::shared_ptr<ArrowColOut> pinned_copy(Result *r, const std::shared_ptr<ArrowColOut> &o, const void *d_values, size_t values_bytes,
                                         const void *d_validity, size_t validity_bytes, const void *d_data, size_t data_bytes) {
  CtxCore &c = *r->core;
  o->values_bytes = values_bytes;
  o->validity_bytes = validity_bytes;
  o->data_bytes = data_bytes;
  o->values = c.pin.alloc(values_bytes + 64);
  o->validity = c.pin.alloc(validity_bytes + 64);
  if (d_data || data_bytes) o->data = c.pin.alloc(data_bytes + 64);
  if (!o->values || !o->validity || ((d_data || data_bytes) && !o->data)) return nullptr;
  memset(o->values, 0, values_bytes < 64 ? values_bytes + 8 : 64);  // (an empty offsets buffer still reads as [0])
  if (values_bytes && d_values && check_cuda(cudaMemcpyAsync(o->values, d_values, values_bytes, cudaMemcpyDeviceToHost, c.s_compute), "nested values D2H")) return nullptr;
  if (validity_bytes && d_validity && check_cuda(cudaMemcpyAsync(o->validity, d_validity, validity_bytes, cudaMemcpyDeviceToHost, c.s_compute), "nested bitmap D2H")) return nullptr;
  if (data_bytes && d_data && check_cuda(cudaMemcpyAsync(o->data, d_data, data_bytes, cudaMemcpyDeviceToHost, c.s_compute), "nested data D2H")) return nullptr;
  r->bytes_d2h += values_bytes + validity_bytes + data_bytes;
  return o;
}

// one level: gather every leaf of `node` through `es`, convert, recurse.  Returns the Arrow child array of that level
// (kLeaf: the leaf; kStruct: struct<fields>; kList: list<...>) and, through *offsets_owner, the gather whose offsets /
// counters describe the level (the caller turns them into its own offsets buffer).
std::shared_ptr<ArrowColOut> node_to_arrow(Result *r, Scope &sc, const EntrySrc &es, ListNode &node, uint64_t inner_cap, GatherOut *first);

std::shared_ptr<ArrowColOut> leaf_to_arrow(Result *r, Scope &sc, const Leaf &leaf, const GatherOut &g, uint64_t cap) {
  CtxCore &c = *r->core;
  auto o = std::make_shared<ArrowColOut>();
  o->core = r->core;
  o->name = leaf.name;
  o->length = (int64_t)cap;
  o->null_count = (int64_t)g.h_ctr[1];
  const size_t bm_bytes = (size_t)((cap + 7) / 8);
  ArrowMap m;
  if (!type_arrow_map(leaf, &m)) { set_error("nested column '%s': child type %d has no Arrow mapping here", leaf.name.c_str(), leaf.type_id); return nullptr; }
  o->format = m.format;
  if (m.is_string) {
    // the gathered string_t are a dense column: 2048-element pseudo chunks, the gathered bitmap as their masks, the
    // arena the stager gathered as the heap
    Pseudo ps;
    if (make_pseudo(sc, cap, sizeof(dmb_string_t), &ps)) return nullptr;
    const size_t data_cap = 12 * (size_t)cap + (size_t)leaf.heap_len;
    void *d_off = sc.dalloc((size_t)(cap + 1) * 4 + 64);
    uint8_t *d_data = (uint8_t *)sc.dalloc(data_cap + 64);
    void *d_scratch = sc.dalloc(dmb_dev_string_scratch_bytes(ps.nchunks > 0 ? ps.nchunks : 1));
    unsigned long long *d_total = (unsigned long long *)sc.dalloc(8), *h = (unsigned long long *)sc.palloc(16);
    if (!d_off || !d_data || !d_scratch || !d_total || !h) return nullptr;
    h[0] = h[1] = 0;
    if (check_cuda(cudaMemsetAsync(d_off, 0, 4, c.s_compute), "nested offsets memset") || check_cuda(cudaMemsetAsync(d_total, 0, 8, c.s_compute), "nested total memset")) return nullptr;
    if (cap) {
      dmb_string_job job;
      memset(&job, 0, sizeof(job));
      job.in = reinterpret_cast<const dmb_string_t *>(g.d_child);
      job.in_validity = g.d_bitmap;
      job.vecs = ps.d_vecs;
      job.heap_dev = leaf.d_heap;
      job.heap_host_base = 1ull << 43;
      job.heap_len = leaf.heap_len;
      job.out_offsets = d_off;
      job.out_data = d_data;
      job.total_bytes = d_total;
      job.mode = DMB_STR_ARROW_UTF8;
      job.out_data_cap = data_cap;
      if (dmb_dev_string_batch(&job, ps.d_counts, ps.d_row_off, ps.nchunks, (int64_t)cap, d_scratch, c.s_compute)) return nullptr;
      if (check_cuda(cudaMemcpyAsync(h, d_total, 8, cudaMemcpyDeviceToHost, c.s_compute), "nested total D2H")) return nullptr;
      if (check_cuda(cudaMemcpyAsync(h + 1, (unsigned long long *)d_scratch + 1, 8, cudaMemcpyDeviceToHost, c.s_compute), "nested flags D2H")) return nullptr;
      if (check_cuda(cudaStreamSynchronize(c.s_compute), "nested string sync")) return nullptr;
      if (h[1] & kStrFlagOverflow) { set_error("nested column '%s': more than 2^31 string bytes; use smaller batches (record-batch stream)", leaf.name.c_str()); return nullptr; }
      if (string_flags_error(h[1])) return nullptr;
    }
    return pinned_copy(r, o, d_off, (size_t)(cap + 1) * 4, g.d_bitmap, bm_bytes, d_data, (size_t)h[0]);
  }
  if (stored_as_arrow(leaf, m.op) || cap == 0) {
    const int ow = dmb_op_out_width(m.op);
    return pinned_copy(r, o, g.d_child, cap == 0 ? 0 : (size_t)cap * (size_t)(ow > 0 ? ow : leaf.width), g.d_bitmap, bm_bytes, nullptr, 0);
  }
  size_t out_bytes = 0;
  uint8_t *d_out = convert_gathered(sc, leaf, g, cap, m.op, &out_bytes);
  if (!d_out) return nullptr;
  return pinned_copy(r, o, d_out, out_bytes, g.d_bitmap, bm_bytes, nullptr, 0);
}

std::shared_ptr<ArrowColOut> node_to_arrow(Result *r, Scope &sc, const EntrySrc &es, ListNode &node, uint64_t inner_cap, GatherOut *first) {
  const uint64_t cap = es.cap;
  const size_t bm_bytes = (size_t)((cap + 7) / 8);
  if (node.kind == ListNode::kLeaf) {
    if (gather_leaf(r, sc, es, node.leaves[0], first) || check_gather(*first, cap)) return nullptr;
    return leaf_to_arrow(r, sc, node.leaves[0], *first, cap);
  }
  if (node.kind == ListNode::kStruct) {
    auto o = std::make_shared<ArrowColOut>();
    o->core = r->core;
    o->name = "item";
    o->format = "+s";
    o->length = (int64_t)cap;
    o->no_values = true;
    for (size_t f = 0; f < node.leaves.size(); ++f) {
      GatherOut g;
      if (gather_leaf(r, sc, es, node.leaves[f], &g) || check_gather(g, cap)) return nullptr;
      if (f == 0) *first = g;
      auto ch = leaf_to_arrow(r, sc, node.leaves[f], g, cap);
      if (!ch) return nullptr;
      o->children.push_back(ch);
    }
    if (node.has_struct_validity) {
      GatherOut gv;
      if (gather_leaf(r, sc, es, node.struct_validity, &gv) || check_gather(gv, cap)) return nullptr;
      o->null_count = (int64_t)gv.h_ctr[1];
      return pinned_copy(r, o, nullptr, 0, gv.d_bitmap, bm_bytes, nullptr, 0);
    }
    o->validity = nullptr;  // no NULL structs: no validity buffer (null_count 0)
    o->validity_bytes = 0;
    return o;
  }
  // LIST<LIST<...>>: the gathered inner entries (already rebased onto the grandchild slab) are the next level's entries
  GatherOut g;
  if (gather_leaf(r, sc, es, node.leaves[0], &g) || check_gather(g, cap)) return nullptr;
  *first = g;
  CtxCore &c = *r->core;
  Pseudo ps;
  if (make_pseudo(sc, cap, 16, &ps)) return nullptr;
  ListNode &in = *node.inner;
  const uint64_t inner_total = in.base.back();
  std::vector<uint64_t> zeros((size_t)ps.nchunks + 1, 0), sizes((size_t)(ps.nchunks > 0 ? ps.nchunks : 1), inner_total);
  EntrySrc es2;
  es2.d_entries = g.d_child;
  es2.d_validity = g.d_bitmap;
  es2.d_vecs = ps.d_vecs;
  es2.d_counts = ps.d_counts;
  es2.d_row_off = ps.d_row_off;
  es2.nchunks = ps.nchunks;
  es2.nrows = (int64_t)cap;
  es2.d_child_base = (const uint64_t *)upload_job(sc, zeros.data(), zeros.size() * 8);
  es2.d_child_sizes = (const uint64_t *)upload_job(sc, sizes.data(), sizes.size() * 8);
  es2.cap = inner_cap;
  es2.dense_bits = true;
  if (!es2.d_child_base || !es2.d_child_sizes) return nullptr;
  GatherOut g2;
  auto child = node_to_arrow(r, sc, es2, in, 0, &g2);
  if (!child) return nullptr;
  if (child->name.empty()) child->name = "item";
  auto o = std::make_shared<ArrowColOut>();
  o->core = r->core;
  o->name = "item";
  o->format = "+l";
  o->length = (int64_t)cap;
  o->null_count = (int64_t)g.h_ctr[1];
  o->children.push_back(child);
  (void)c;
  return pinned_copy(r, o, g2.d_offsets, (size_t)(cap + 1) * 4, g.d_bitmap, bm_bytes, nullptr, 0);
}

// host passes over the entries: how many elements each level's gather produces (sizes the outputs exactly and refuses
// entries that reach outside their child vector before anything is launched)
int32_t nested_caps(Result *r, const Col &col, uint64_t *cap1, uint64_t *cap2) {
  CtxCore &c = *r->core;
  const int64_t nch = r->nchunks;
  const ListNode &node = *col.node;
  std::vector<uint64_t> p1((size_t)(nch > 0 ? nch : 1), 0), p2((size_t)(nch > 0 ? nch : 1), 0);
  std::atomic<bool> outside{false};
  const bool nested = node.kind == ListNode::kList;
  if (nested && node.inner->kind == ListNode::kList) { set_error("LIST nesting deeper than two levels is not supported"); return -1; }
  parallel_for(c, nch, [&](int64_t k) {
    const uint64_t *e = reinterpret_cast<const uint64_t *>(col.data[(size_t)k]);
    const void *mask = col.validity.empty() ? nullptr : col.validity[(size_t)k];
    const uint64_t csize = node.sizes[(size_t)k];
    const uint64_t *ie = nested ? reinterpret_cast<const uint64_t *>(node.leaves[0].data[(size_t)k]) : nullptr;
    const void *imask = (nested && !node.leaves[0].validity.empty()) ? node.leaves[0].validity[(size_t)k] : nullptr;
    const uint64_t isize = nested ? node.inner->sizes[(size_t)k] : 0;
    uint64_t s1 = 0, s2 = 0;
    for (uint32_t i = 0; e && i < r->counts[(size_t)k]; ++i) {
      if (!host_row_valid(mask, i)) continue;
      const uint64_t off = e[2 * i], len = e[2 * i + 1];
      if (off > csize || len > csize - off) { outside.store(true); continue; }
      s1 += len;
      for (uint64_t q = off; nested && q < off + len; ++q) {
        if (imask && !((reinterpret_cast<const uint64_t *>(imask)[q >> 6] >> (q & 63)) & 1ull)) continue;
        const uint64_t io = ie[2 * q], il = ie[2 * q + 1];
        if (io > isize || il > isize - io) { outside.store(true); continue; }
        s2 += il;
      }
    }
    p1[(size_t)k] = s1;
    p2[(size_t)k] = s2;
  });
  if (outside.load()) { set_error("nested column '%s': a list entry reaches outside its chunk's child vector", col.name.c_str()); return -1; }
  *cap1 = *cap2 = 0;
  for (int64_t k = 0; k < nch; ++k) { *cap1 += p1[(size_t)k]; *cap2 += p2[(size_t)k]; }
  return 0;
}

// A top-level LIST of one fixed-width leaf, launched in materialise_arrow's pipeline and copied out by drain_arrow_col
struct ListRun {
  FixedRun validity;  // the LIST column's own bitmap / null count
  GatherOut g;        // done: after the conversion pass and the parent's null count as well
  uint64_t cap = 0;
  uint8_t *d_child_out = nullptr;  // the child in its Arrow form (== g.d_child when it is exported as stored)
  size_t child_out_bytes = 0;
};

int32_t run_list(Result *r, Scope &sc, int j, int32_t child_op, ListRun *out) {
  Col &col = r->cols[(size_t)j];
  CtxCore &c = *r->core;
  const Leaf &leaf = col.node->leaves[0];
  // the child slab first: the entries' staging and the host pass below overlap its copy-in
  if (stage_node(r, *col.node, false)) return -1;
  // the column's own validity bitmap + null count (also stages the entries)
  if (run_fixed(r, sc, j, DMB_OP_VALIDITY_ONLY, 0, true, false, &out->validity)) return -1;
  cudaEvent_t e = sc.event(false);  // the child slab was copied on the copy-in stream
  if (!e) return -1;
  cudaEventRecord(e, c.s_in);
  if (check_cuda(cudaStreamWaitEvent(c.s_compute, e, 0), "wait list child")) return -1;
  uint64_t cap2 = 0;
  if (nested_caps(r, col, &out->cap, &cap2)) return -1;
  if (gather_leaf(r, sc, column_entries(r, col, out->cap), leaf, &out->g)) return -1;
  out->d_child_out = out->g.d_child;
  out->child_out_bytes = (size_t)out->cap * (size_t)leaf.width;
  if (!stored_as_arrow(leaf, child_op) && out->cap > 0) {
    out->d_child_out = convert_gathered(sc, leaf, out->g, out->cap, child_op, &out->child_out_bytes);
    if (!out->d_child_out) return -1;
  }
  if (check_cuda(cudaMemcpyAsync(out->g.h_ctr + 3, out->validity.d_null_count, 8, cudaMemcpyDeviceToHost, c.s_compute), "null count D2H")) return -1;
  cudaEventRecord(out->g.done, c.s_compute);
  return 0;
}

struct Pending;
int32_t launch_arrow_col(Result *r, Scope &sc, int j, int string_mode, Pending *p, size_t exact_cap);
std::shared_ptr<ArrowColOut> convert_column_sync(Result *r, Scope &sc, int j);

// STRUCT / MAP / LIST with a described child -> the finished Arrow array (synchronous)
std::shared_ptr<ArrowColOut> nested_to_arrow(Result *r, Scope &sc, int j) {
  NvtxRange nvtx("dmb::nested_to_arrow");
  CtxCore &c = *r->core;
  const int64_t n = r->nrows;
  // the parent's own validity bitmap + null count
  FixedRun fr;
  if (run_fixed(r, sc, j, DMB_OP_VALIDITY_ONLY, 0, true, false, &fr)) return nullptr;
  unsigned long long *h_null = (unsigned long long *)sc.palloc(8);
  if (!h_null) return nullptr;
  *h_null = 0;
  if (n && check_cuda(cudaMemcpyAsync(h_null, fr.d_null_count, 8, cudaMemcpyDeviceToHost, c.s_compute), "null count D2H")) return nullptr;
  auto o = std::make_shared<ArrowColOut>();
  o->core = r->core;
  o->name = r->cols[(size_t)j].name;
  o->length = n;
  if (r->cols[(size_t)j].is_struct) {
    o->format = "+s";
    o->no_values = true;
    const std::vector<int> kids = r->cols[(size_t)j].kids;  // (copy: converting a kid may touch r->cols)
    for (int kid : kids) {
      auto ch = convert_column_sync(r, sc, kid);
      if (!ch) return nullptr;
      o->children.push_back(ch);
    }
    if (!pinned_copy(r, o, nullptr, 0, fr.d_bitmap, n ? fr.bitmap_bytes : 0, nullptr, 0)) return nullptr;
  } else {
    Col &col = r->cols[(size_t)j];
    ListNode &node = *col.node;
    uint64_t cap1 = 0, cap2 = 0;
    if (nested_caps(r, col, &cap1, &cap2)) return nullptr;
    if (stage_node(r, node, false)) return nullptr;
    cudaEvent_t e = sc.event(false);  // the child slabs were copied on the copy-in stream
    if (!e) return nullptr;
    cudaEventRecord(e, c.s_in);
    if (check_cuda(cudaStreamWaitEvent(c.s_compute, e, 0), "wait nested children")) return nullptr;
    GatherOut g1;
    auto child = node_to_arrow(r, sc, column_entries(r, col, cap1), node, cap2, &g1);
    if (!child) return nullptr;
    const bool is_map = col.type_id == DMB_TYPE_MAP;
    o->format = is_map ? "+m" : "+l";
    if (is_map) {  // Arrow map<key, value>: entries struct and keys are non-nullable
      child->name = "entries";
      child->flags = 0;
      if (child->children.size() == 2) {
        if (child->children[0]->null_count != 0) { set_error("MAP column '%s': NULL keys", col.name.c_str()); return nullptr; }
        child->children[0]->flags = 0;
        if (child->children[0]->name.empty()) child->children[0]->name = "key";
        if (child->children[1]->name.empty()) child->children[1]->name = "value";
      }
    } else if (child->name.empty()) {
      child->name = "item";
    }
    o->children.push_back(child);
    if (!pinned_copy(r, o, g1.d_offsets, (size_t)(n + 1) * 4, fr.d_bitmap, n ? fr.bitmap_bytes : 0, nullptr, 0)) return nullptr;
  }
  if (check_cuda(cudaStreamSynchronize(c.s_compute), "nested sync")) return nullptr;
  o->null_count = (int64_t)*h_null;
  return o;
}

struct Pending {  // one column between its kernel launch and its device->host copies
  ArrowMap map;
  FixedRun fr;
  StringRun sr;
  ListRun lr;
  std::shared_ptr<ArrowColOut> out;
  unsigned long long *h_null = nullptr;
};

int32_t launch_arrow_col(Result *r, Scope &sc, int j, int string_mode, Pending *p, size_t exact_cap = 0) {
  Col &col = r->cols[(size_t)j];
  if (!arrow_map(col, &p->map)) return -1;
  if (p->map.is_nested) {
    p->out = nested_to_arrow(r, sc, j);
    return p->out ? 0 : -1;
  }
  p->out = std::make_shared<ArrowColOut>();
  p->out->core = r->core;
  p->out->name = col.name;
  p->out->length = r->nrows;
  if (col.type_id == DMB_TYPE_ENUM) p->out->dict = col.dict;
  if (p->map.is_list) {
    p->lr = ListRun();
    if (run_list(r, sc, j, p->map.child_op, &p->lr)) return -1;
    p->out->format = p->map.format;
    auto ch = std::make_shared<ArrowColOut>();
    ch->core = r->core;
    ch->name = col.node->leaves[0].name.empty() ? "item" : col.node->leaves[0].name;
    ch->format = p->map.child_format;
    p->out->children.push_back(ch);
    return 0;
  }
  if (p->map.is_string) {
    p->sr = StringRun();
    if (run_string(r, sc, j, string_mode, true, false, &p->sr, exact_cap, /*as_text=*/false)) return -1;
    p->out->format = string_mode == DMB_STR_ARROW_LARGE ? (col.type_id == DMB_TYPE_BLOB ? "Z" : "U") : p->map.format;
  } else {
    p->fr = FixedRun();
    if (run_fixed(r, sc, j, p->map.op, 0, true, false, &p->fr)) return -1;
    p->out->format = p->map.format;
  }
  return 0;
}

// enqueue the device->host copies of a launched column on the copy-out stream.
// Returns 1 when a utf8 column overflowed int32 offsets and must be relaunched with large offsets.
int32_t drain_arrow_col(Result *r, Scope &sc, Pending *p) {
  CtxCore &c = *r->core;
  if (p->map.is_nested) return 0;  // converted (and copied out) at launch
  ArrowColOut &o = *p->out;
  const int64_t n = r->nrows;
  if (p->map.is_list) {
    ListRun &l = p->lr;
    ArrowColOut &ch = *o.children[0];
    if (check_gather(l.g, l.cap)) return -1;
    o.values_bytes = (size_t)(n + 1) * 4;
    o.validity_bytes = l.validity.bitmap_bytes;
    o.null_count = (int64_t)l.g.h_ctr[3];
    ch.length = (int64_t)l.cap;
    ch.null_count = (int64_t)l.g.h_ctr[1];
    ch.values_bytes = l.child_out_bytes;
    ch.validity_bytes = (size_t)((l.cap + 7) / 8);
    o.values = c.pin.alloc(o.values_bytes + 64);
    o.validity = c.pin.alloc(o.validity_bytes + 64);
    ch.values = c.pin.alloc(ch.values_bytes + 64);
    ch.validity = c.pin.alloc(ch.validity_bytes + 64);
    if (!o.values || !o.validity || !ch.values || !ch.validity) return -1;
    if (check_cuda(cudaStreamWaitEvent(c.s_out, l.g.done, 0), "wait kernel")) return -1;
    if (check_cuda(cudaMemcpyAsync(o.values, l.g.d_offsets, o.values_bytes, cudaMemcpyDeviceToHost, c.s_out), "list offsets D2H")) return -1;
    if (o.validity_bytes && check_cuda(cudaMemcpyAsync(o.validity, l.validity.d_bitmap, o.validity_bytes, cudaMemcpyDeviceToHost, c.s_out), "bitmap D2H")) return -1;
    if (ch.values_bytes && check_cuda(cudaMemcpyAsync(ch.values, l.d_child_out, ch.values_bytes, cudaMemcpyDeviceToHost, c.s_out), "list child D2H")) return -1;
    if (ch.validity_bytes && check_cuda(cudaMemcpyAsync(ch.validity, l.g.d_bitmap, ch.validity_bytes, cudaMemcpyDeviceToHost, c.s_out), "list child bitmap D2H")) return -1;
    r->bytes_d2h += o.values_bytes + o.validity_bytes + ch.values_bytes + ch.validity_bytes;
    return 0;
  }
  if (p->map.is_string) {
    StringRun &s = p->sr;
    if (check_cuda(cudaEventSynchronize(s.done), "string kernel wait")) return -1;
    if (!(s.h_ctr[1] & ~(kStrFlagDataCap | kStrFlagOverflow)) && !s.h_ctr[3]) {
      if ((s.h_ctr[1] & kStrFlagOverflow) && s.mode == DMB_STR_ARROW_UTF8) return 1;  // redo with 64-bit offsets
      if ((s.h_ctr[1] & kStrFlagDataCap) && !s.exact) return 2;                        // redo, sized exactly
    }
    if (string_flags_error(s.h_ctr[1] | (s.h_ctr[3] ? (1ull << 63) : 0ull))) return -1;
    const size_t total = (size_t)s.h_ctr[0];
    o.values_bytes = s.offsets_bytes;
    o.validity_bytes = s.validity.bitmap_bytes;
    o.data_bytes = total;
    o.values = c.pin.alloc(o.values_bytes + 64);
    o.validity = c.pin.alloc(o.validity_bytes + 64);
    o.data = c.pin.alloc(total + 64);
    if (!o.values || !o.validity || !o.data) return -1;
    o.null_count = (int64_t)s.h_ctr[2];
    if (n == 0) {
      memset(o.values, 0, o.values_bytes);
      return 0;
    }
    if (check_cuda(cudaStreamWaitEvent(c.s_out, s.done, 0), "wait kernel")) return -1;
    if (check_cuda(cudaMemcpyAsync(o.values, s.d_offsets, o.values_bytes, cudaMemcpyDeviceToHost, c.s_out), "offsets D2H")) return -1;
    if (total && check_cuda(cudaMemcpyAsync(o.data, s.d_data, total, cudaMemcpyDeviceToHost, c.s_out), "utf8 data D2H")) return -1;
    if (o.validity_bytes && check_cuda(cudaMemcpyAsync(o.validity, s.validity.d_bitmap, o.validity_bytes, cudaMemcpyDeviceToHost, c.s_out), "bitmap D2H")) return -1;
    r->bytes_d2h += o.values_bytes + total + o.validity_bytes;
    return 0;
  }
  FixedRun &f = p->fr;
  o.values_bytes = f.values_bytes;
  o.validity_bytes = f.bitmap_bytes;
  o.values = c.pin.alloc(o.values_bytes + 64);
  o.validity = c.pin.alloc(o.validity_bytes + 64);
  p->h_null = (unsigned long long *)sc.palloc(8);
  if (!o.values || !o.validity || !p->h_null) return -1;
  *p->h_null = 0;
  if (n == 0) return 0;
  if (check_cuda(cudaStreamWaitEvent(c.s_out, f.done, 0), "wait kernel")) return -1;
  if (o.values_bytes && check_cuda(cudaMemcpyAsync(o.values, f.d_values, o.values_bytes, cudaMemcpyDeviceToHost, c.s_out), "values D2H")) return -1;
  if (o.validity_bytes && check_cuda(cudaMemcpyAsync(o.validity, f.d_bitmap, o.validity_bytes, cudaMemcpyDeviceToHost, c.s_out), "bitmap D2H")) return -1;
  if (check_cuda(cudaMemcpyAsync(p->h_null, f.d_null_count, 8, cudaMemcpyDeviceToHost, c.s_out), "null count D2H")) return -1;
  r->bytes_d2h += o.values_bytes + o.validity_bytes + 8;
  return 0;
}

// drain + the two relaunch cases of a string column (1: utf8 offsets overflowed -> 64-bit offsets; 2: aliased string_t
// pointers overflowed the first-guess data buffer -> sized exactly from the total the first launch reported)
int32_t drain_with_redo(Result *r, Scope &sc, Pending *p, int j) {
  int32_t rc = drain_arrow_col(r, sc, p);
  for (int redo = 0; redo < 2 && (rc == 1 || rc == 2); ++redo) {
    const int mode = rc == 1 ? DMB_STR_ARROW_LARGE : p->sr.mode;
    const size_t exact = (size_t)p->sr.h_ctr[0];
    *p = Pending();
    if (launch_arrow_col(r, sc, j, mode, p, exact)) return -1;
    rc = drain_arrow_col(r, sc, p);
  }
  return rc > 0 ? -1 : rc;
}

// one column, start to finish (STRUCT fields)
std::shared_ptr<ArrowColOut> convert_column_sync(Result *r, Scope &sc, int j) {
  CtxCore &c = *r->core;
  Pending p;
  const Col &col = r->cols[(size_t)j];
  const bool surely_large = col.phys == DMB_PHYS_STRING && (col.heap_len > 0x7fffffffull || col.force_large);
  if (launch_arrow_col(r, sc, j, surely_large ? DMB_STR_ARROW_LARGE : DMB_STR_ARROW_UTF8, &p)) return nullptr;
  if (drain_with_redo(r, sc, &p, j)) return nullptr;
  if (check_cuda(cudaStreamSynchronize(c.s_compute), "sync compute") || check_cuda(cudaStreamSynchronize(c.s_out), "sync copy-out")) return nullptr;
  if (!p.map.is_string && !p.map.is_list && !p.map.is_nested && p.h_null) p.out->null_count = (int64_t)*p.h_null;
  r->cols[(size_t)j].arrow = p.out;
  return p.out;
}

int32_t materialise_arrow(Result *r) {
  if (r->arrow_ready) return 0;
  NvtxRange nvtx("dmb::materialise_arrow");
  CtxCore &c = *r->core;
  if (!c.bind()) return -1;
  const double t0 = now_ms();
  const int ncols = r->column_count;  // (STRUCT fields live behind the visible columns and are converted by their parent)
  {
    std::vector<Pending> pend((size_t)ncols);  // declared first: the Scope drains the streams before these die
    Scope sc(c);
    cudaEvent_t in0 = sc.event(true), in1 = sc.event(true), out0 = sc.event(true), out1 = sc.event(true);
    if (!in0 || !in1 || !out0 || !out1) return -1;
    r->bytes_h2d = 0;
    r->bytes_d2h = 0;
    const bool restage = !r->meta_staged;
    cudaEventRecord(in0, c.s_in);
    cudaEventRecord(out0, c.s_out);
    auto drain = [&](int j) -> int32_t {
      const double t_d0 = wall_ms();
      const int32_t rc = drain_with_redo(r, sc, &pend[(size_t)j], j);
      c.t_drain_wait += wall_ms() - t_d0;
      return rc;
    };
    c.t_gather = c.t_ring_wait = c.t_drain_wait = c.t_stage = c.t_launch = 0;
    // Processing order.  Copy-in and copy-out are two machines every column passes through in that order (the kernel in
    // between is ~2 % of either): a two-machine flow shop, whose makespan Johnson's rule minimises -- columns that grow on
    // the way (copy-in shorter than copy-out: DECIMAL -> decimal128) first, by increasing copy-in; the rest (VARCHAR: 16-byte
    // string_t in, 4-byte offsets out) after them, by decreasing copy-out.  The copy-out stream then never waits for a long
    // copy-in behind a short one, and the two ends that cannot overlap are the smallest transfers.  (Round 1's order --
    // small columns at both ends, large ones in the middle -- left the copy-out stream idle behind the 2.5 GB copy-ins of the
    // text columns: 266 vs 237 ms for the C2 table in the bytes / link-rate model, lower bound 231.)
    std::vector<int> order((size_t)ncols);
    {
      std::vector<uint64_t> w_in((size_t)ncols), w_out((size_t)ncols);
      const uint64_t n = (uint64_t)r->nrows;
      for (int j = 0; j < ncols; ++j) {
        const Col &col = r->cols[(size_t)j];
        ArrowMap m;
        const bool mapped = arrow_map(col, &m);
        const uint64_t list_bytes = mapped && m.is_list ? col.node->base.back() * (uint64_t)col.node->leaves[0].width : 0;
        w_in[(size_t)j] = (uint64_t)col.width * n + col.heap_len + list_bytes;
        uint64_t out = w_in[(size_t)j];
        if (mapped && !m.is_nested && !m.is_list) {
          if (m.is_string) out = 4 * n + (col.heap_len ? col.heap_len : 4 * n);  // (inlined bytes are not known before the kernel: a guess)
          else { const int32_t ow = dmb_op_out_width(m.op); out = ow > 0 ? (uint64_t)ow * n : n / 8; }
        }
        w_out[(size_t)j] = out;
        order[(size_t)j] = j;
      }
      std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
        const bool ga = w_in[(size_t)a] < w_out[(size_t)a], gb = w_in[(size_t)b] < w_out[(size_t)b];
        if (ga != gb) return ga;                                       // the growing columns first ...
        if (ga) return w_in[(size_t)a] < w_in[(size_t)b];              // ... by increasing copy-in
        return w_out[(size_t)a] > w_out[(size_t)b];                    // the others by decreasing copy-out
      });
    }
    for (int k = 0; k < ncols; ++k) {
      const int j = order[(size_t)k];
      const Col &col = r->cols[(size_t)j];
      const bool surely_large = col.phys == DMB_PHYS_STRING && (col.heap_len > 0x7fffffffull || col.force_large);
      const double t_l0 = wall_ms();
      if (launch_arrow_col(r, sc, j, surely_large ? DMB_STR_ARROW_LARGE : DMB_STR_ARROW_UTF8, &pend[(size_t)j])) return -1;
      c.t_launch += wall_ms() - t_l0;
      if (k > 0 && drain(order[(size_t)k - 1])) return -1;
    }
    cudaEventRecord(in1, c.s_in);
    if (ncols > 0 && drain(order[(size_t)ncols - 1])) return -1;
    cudaEventRecord(out1, c.s_out);
    if (check_cuda(cudaStreamSynchronize(c.s_in), "sync copy-in") || check_cuda(cudaStreamSynchronize(c.s_compute), "sync compute") ||
        check_cuda(cudaStreamSynchronize(c.s_out), "sync copy-out"))
      return -1;
    for (int j = 0; j < ncols; ++j) {
      Pending &p = pend[(size_t)j];
      if (!p.map.is_string && !p.map.is_list && !p.map.is_nested && p.h_null) p.out->null_count = (int64_t)*p.h_null;
      r->cols[(size_t)j].arrow = p.out;
    }
    float f = 0;
    r->t_h2d = (restage && cudaEventElapsedTime(&f, in0, in1) == cudaSuccess) ? f : 0;
    r->t_d2h = cudaEventElapsedTime(&f, out0, out1) == cudaSuccess ? f : 0;
    r->t_kernels = sc.kernel_ms();
  }
  r->t_total = now_ms() - t0;
  static const bool trace = getenv("DMB_TRACE_STAGE") != nullptr;
  if (trace)
    fprintf(stderr, "[dmb] materialise_arrow %.1f ms: gather + string compaction %.1f (of which waiting for a ring buffer %.1f), drain (kernel waits + D2H enqueue) %.1f, stage_column %.1f, launch_arrow_col (staging included) %.1f, h2d stream %.1f, d2h stream %.1f\n",
            r->t_total, c.t_gather, c.t_ring_wait, c.t_drain_wait, c.t_stage, c.t_launch, r->t_h2d, r->t_d2h);
  r->arrow_ready = true;
  return 0;
}

// ------------------------------------------------------------------ Arrow C Data export
struct ExportPriv {
  std::vector<std::shared_ptr<ArrowColOut>> cols;
  const void *buffers[3] = {nullptr, nullptr, nullptr};
  std::vector<ArrowArray *> child_arrays;
  std::vector<ArrowSchema *> child_schemas;
  std::shared_ptr<EnumDict> dict;  // a dictionary array's buffers
  std::string format, name;
};

void release_array(ArrowArray *a) {
  if (!a || !a->release) return;
  ExportPriv *p = reinterpret_cast<ExportPriv *>(a->private_data);
  for (ArrowArray *ch : p->child_arrays) {
    if (ch->release) ch->release(ch);
    free(ch);
  }
  if (a->dictionary) {
    if (a->dictionary->release) a->dictionary->release(a->dictionary);
    free(a->dictionary);
    a->dictionary = nullptr;
  }
  delete p;
  a->release = nullptr;
}

void release_schema(ArrowSchema *s) {
  if (!s || !s->release) return;
  ExportPriv *p = reinterpret_cast<ExportPriv *>(s->private_data);
  for (ArrowSchema *ch : p->child_schemas) {
    if (ch->release) ch->release(ch);
    free(ch);
  }
  if (s->dictionary) {
    if (s->dictionary->release) s->dictionary->release(s->dictionary);
    free(s->dictionary);
    s->dictionary = nullptr;
  }
  delete p;
  s->release = nullptr;
}

void export_column(const std::shared_ptr<ArrowColOut> &o, ArrowArray *a, ArrowSchema *s) {
  if (a) {
    ExportPriv *p = new ExportPriv();
    p->cols.push_back(o);
    memset(a, 0, sizeof(*a));
    a->length = o->length;
    a->null_count = o->null_count;
    a->offset = 0;
    p->buffers[0] = o->validity;
    p->buffers[1] = o->values;
    p->buffers[2] = o->data;
    a->n_buffers = o->data ? 3 : 2;
    a->buffers = p->buffers;
    a->release = release_array;
    a->private_data = p;
    if (!o->children.empty()) {  // LIST / MAP: one child array; STRUCT: one per field
      a->n_buffers = o->no_values ? 1 : 2;
      for (const auto &chd : o->children) {
        ArrowArray *ca = (ArrowArray *)calloc(1, sizeof(ArrowArray));
        export_column(chd, ca, nullptr);
        p->child_arrays.push_back(ca);
      }
      a->n_children = (int64_t)p->child_arrays.size();
      a->children = p->child_arrays.data();
    }
    if (o->dict) {  // ENUM: the labels as a utf8 dictionary array (no nulls), buffers shared with the result
      static const char kNoBytes[1] = {0};
      ArrowArray *da = (ArrowArray *)calloc(1, sizeof(ArrowArray));
      ExportPriv *dp = new ExportPriv();
      dp->dict = o->dict;
      da->length = (int64_t)o->dict->size();
      dp->buffers[0] = nullptr;
      dp->buffers[1] = o->dict->offsets.data();
      dp->buffers[2] = o->dict->data.empty() ? kNoBytes : o->dict->data.data();
      da->n_buffers = 3;
      da->buffers = dp->buffers;
      da->release = release_array;
      da->private_data = dp;
      a->dictionary = da;
    }
  }
  if (s) {
    ExportPriv *p = new ExportPriv();
    p->format = o->format;
    p->name = o->name;
    memset(s, 0, sizeof(*s));
    s->format = p->format.c_str();
    s->name = p->name.c_str();
    s->flags = o->flags;  // ARROW_FLAG_NULLABLE
    s->release = release_schema;
    s->private_data = p;
    if (!o->children.empty()) {
      for (const auto &chd : o->children) {
        ArrowSchema *cs = (ArrowSchema *)calloc(1, sizeof(ArrowSchema));
        export_column(chd, nullptr, cs);
        p->child_schemas.push_back(cs);
      }
      s->n_children = (int64_t)p->child_schemas.size();
      s->children = p->child_schemas.data();
    }
    if (o->dict) {
      ArrowSchema *ds = (ArrowSchema *)calloc(1, sizeof(ArrowSchema));
      ExportPriv *dp = new ExportPriv();
      dp->format = "u";
      ds->format = dp->format.c_str();
      ds->name = dp->name.c_str();
      ds->release = release_schema;
      ds->private_data = dp;
      s->dictionary = ds;
    }
  }
}

// ------------------------------------------------------------------ typed columns
struct TypedMap {
  int32_t tag, op, width;
};

bool typed_map(const Col &col, TypedMap *m) {
  auto set = [&](int32_t tag, int32_t dst, int32_t width) { m->tag = tag; m->op = DMB_OP(col.phys, dst); m->width = width; return true; };
  switch (col.type_id) {
    case DMB_TYPE_BOOLEAN: return set(DMB_VALUE_BOOL, DMB_DST_BOOL_BYTE, 1);
    case DMB_TYPE_TINYINT: case DMB_TYPE_SMALLINT: case DMB_TYPE_INTEGER: case DMB_TYPE_BIGINT:
    case DMB_TYPE_UTINYINT: case DMB_TYPE_USMALLINT: case DMB_TYPE_UINTEGER: case DMB_TYPE_UBIGINT:
      return set(DMB_VALUE_INT, DMB_DST_I32_SAT, 4);  // src/duckdb_parsing.mbt:88-99 -> parse_int :203-237
    case DMB_TYPE_FLOAT: case DMB_TYPE_DOUBLE: return set(DMB_VALUE_DOUBLE, DMB_DST_F64, 8);
    case DMB_TYPE_DATE: return set(DMB_VALUE_DATE, DMB_DST_DATE_REF, 4);
    // parse_timestamp semantics (src/duckdb_parsing.mbt:375-398), including the day-number quirk
    case DMB_TYPE_TIMESTAMP: case DMB_TYPE_TIMESTAMP_TZ: return set(DMB_VALUE_TIMESTAMP, DMB_DST_TS_REF, 8);
    case DMB_TYPE_TIMESTAMP_S: return set(DMB_VALUE_TIMESTAMP, DMB_DST_TS_REF_FROM_S, 8);
    case DMB_TYPE_TIMESTAMP_MS: return set(DMB_VALUE_TIMESTAMP, DMB_DST_TS_REF_FROM_MS, 8);
    case DMB_TYPE_TIMESTAMP_NS: return set(DMB_VALUE_TIMESTAMP, DMB_DST_TS_REF_FROM_NS, 8);
    case DMB_TYPE_VARCHAR: m->tag = DMB_VALUE_STRING; m->op = -1; m->width = 0; return true;
    default:
      // DECIMAL, HUGEINT, UHUGEINT, INTERVAL, TIME*, BLOB, UUID stay Value::String (libduckdb's
      // text rendering) in the reference, src/duckdb_parsing.mbt:120-141
      if (text_supported(col)) { m->tag = DMB_VALUE_STRING; m->op = -1; m->width = 0; return true; }
      set_error("column type %d is a text-rendered Value::String in the reference; its rendering is not reproduced on the device", col.type_id);
      return false;
  }
}

// utf8 offsets + data + byte validity of column j's text form (the VARCHAR column itself, or the
// device rendering of a fixed-width column), copied into pinned buffers owned by the result
int32_t text_column_out(Result *r, Scope &sc, int j, TypedOut &t) {
  CtxCore &c = *r->core;
  const int64_t n = r->nrows;
  StringRun s;
  if (run_string_sync(r, sc, j, DMB_STR_ARROW_UTF8, false, true, &s)) return -1;
  const size_t total = (size_t)s.h_ctr[0];
  t.offsets = keep_pin(r, s.offsets_bytes);
  t.data = keep_pin(r, total);
  if (!t.offsets || !t.data) return -1;
  if (n == 0) memset(t.offsets, 0, s.offsets_bytes);
  if (n && check_cuda(cudaMemcpyAsync(t.offsets, s.d_offsets, s.offsets_bytes, cudaMemcpyDeviceToHost, c.s_compute), "offsets D2H")) return -1;
  if (total && check_cuda(cudaMemcpyAsync(t.data, s.d_data, total, cudaMemcpyDeviceToHost, c.s_compute), "data D2H")) return -1;
  if (n && check_cuda(cudaMemcpyAsync(t.valid, s.validity.d_valid_bytes, (size_t)n, cudaMemcpyDeviceToHost, c.s_compute), "valid D2H")) return -1;
  if (check_cuda(cudaStreamSynchronize(c.s_compute), "typed sync")) return -1;
  t.null_count = (int64_t)s.h_ctr[2];
  return 0;
}

int32_t typed_column(Result *r, int j, dmb_typed_column *out) {
  Col &col = r->cols[(size_t)j];
  CtxCore &c = *r->core;
  if (!c.bind()) return -1;
  const int64_t n = r->nrows;
  if (!col.typed.ready) {
    TypedMap m;
    if (!typed_map(col, &m)) return -1;
    Scope sc(c);
    TypedOut &t = col.typed;
    t.tag = m.tag;
    t.width = m.width;
    t.valid = keep_pin(r, (size_t)n);
    if (!t.valid) return -1;
    if (m.op < 0) {
      if (text_column_out(r, sc, j, t)) return -1;
    } else {
      FixedRun f;
      if (run_fixed(r, sc, j, m.op, 0, false, true, &f)) return -1;
      t.values = keep_pin(r, f.values_bytes);
      unsigned long long *h_null = (unsigned long long *)sc.palloc(8);
      if (!t.values || !h_null) return -1;
      *h_null = 0;
      if (n && check_cuda(cudaMemcpyAsync(t.values, f.d_values, f.values_bytes, cudaMemcpyDeviceToHost, c.s_compute), "values D2H")) return -1;
      if (n && check_cuda(cudaMemcpyAsync(t.valid, f.d_valid_bytes, (size_t)n, cudaMemcpyDeviceToHost, c.s_compute), "valid D2H")) return -1;
      if (n && check_cuda(cudaMemcpyAsync(h_null, f.d_null_count, 8, cudaMemcpyDeviceToHost, c.s_compute), "null count D2H")) return -1;
      if (check_cuda(cudaStreamSynchronize(c.s_compute), "typed sync")) return -1;
      t.null_count = (int64_t)*h_null;
    }
    t.ready = true;
  }
  const TypedOut &t = col.typed;
  out->tag = t.tag;
  out->width = t.width;
  out->length = n;
  out->null_count = t.null_count;
  out->values = t.values;
  out->valid = (const uint8_t *)t.valid;
  out->offsets = (const int32_t *)t.offsets;
  out->data = (const uint8_t *)t.data;
  return 0;
}

// the string form of any column: what Connection::query collects cell by cell through
// duckdb_mb_result_is_null / duckdb_mb_result_value (src/duckdb_native.c:215-238)
int32_t text_column(Result *r, int j, dmb_typed_column *out) {
  Col &col = r->cols[(size_t)j];
  CtxCore &c = *r->core;
  if (!c.bind()) return -1;
  const int64_t n = r->nrows;
  if (!text_supported(col)) {
    set_error("column %d (type %d): libduckdb's text rendering of this type is not reproduced on the device", j, col.type_id);
    return -1;
  }
  if (col.typed.ready && col.typed.tag == DMB_VALUE_STRING && !col.text.ready) col.text = col.typed;
  if (!col.text.ready) {
    Scope sc(c);
    TypedOut &t = col.text;
    t.tag = DMB_VALUE_STRING;
    t.width = 0;
    t.valid = keep_pin(r, (size_t)n);
    if (!t.valid) return -1;
    if (text_column_out(r, sc, j, t)) return -1;
    t.ready = true;
  }
  const TypedOut &t = col.text;
  out->tag = t.tag;
  out->width = 0;
  out->length = n;
  out->null_count = t.null_count;
  out->values = nullptr;
  out->valid = (const uint8_t *)t.valid;
  out->offsets = (const int32_t *)t.offsets;
  out->data = (const uint8_t *)t.data;
  return 0;
}

// ------------------------------------------------------------------ reference packed getters
moonbit_bytes_t empty_bytes() { return moonbit_make_bytes_raw(0); }  // duckdb_mb_make_bytes("", 0)

enum GetterKind { kGetInt32, kGetInt64, kGetDouble, kGetBool };

// The reference reads a cell with duckdb_value_int64 / _double / _boolean (src/duckdb_native.c:2384,2417,2449,2541),
// and libduckdb casts by the column's LOGICAL type: integers, floats, HUGEINT and UHUGEINT by TryCast (failure -> 0),
// DECIMAL by its scale (TryCastFromDecimal), and DATE / TIME* / TIMESTAMP* / INTERVAL / UUID / ENUM have no cast to a
// number, so the cell reads as 0.  VARCHAR -> number (libduckdb parses the text) is not reproduced: 0 as well.
// Only the same-family casts are pinned by reference tests (SURVEY.md 8c); the rest is UNPINNED.
struct GetterOp {
  int32_t op, param;
};
GetterOp getter_op(const Col &col, GetterKind kind) {
  static const int32_t kDst[] = {DMB_DST_I32_TRUNC, DMB_DST_I64, DMB_DST_F64, DMB_DST_BOOL_BYTE};
  static const int32_t kDecDst[] = {DMB_DST_DEC_I32_TRUNC, DMB_DST_DEC_I64, DMB_DST_DEC_F64, DMB_DST_DEC_BOOL_BYTE};
  switch (col.type_id) {
    case DMB_TYPE_BOOLEAN: case DMB_TYPE_TINYINT: case DMB_TYPE_SMALLINT: case DMB_TYPE_INTEGER: case DMB_TYPE_BIGINT:
    case DMB_TYPE_UTINYINT: case DMB_TYPE_USMALLINT: case DMB_TYPE_UINTEGER: case DMB_TYPE_UBIGINT:
    case DMB_TYPE_FLOAT: case DMB_TYPE_DOUBLE: case DMB_TYPE_HUGEINT: case DMB_TYPE_UHUGEINT:
      return GetterOp{DMB_OP(col.phys, kDst[kind]), 0};
    case DMB_TYPE_DECIMAL:
      return GetterOp{DMB_OP(col.phys, kDecDst[kind]), col.dec_scale};
    default:
      return GetterOp{DMB_OP_VALIDITY_ONLY, 0};
  }
}

// ---- device -> a pageable host buffer (a MoonBit Bytes payload) through the pinned ring: DMA of piece i+1 runs while the
// host threads copy piece i out of the ring.  (cudaMemcpyAsync straight into pageable memory is staged by the driver in
// small serialised pieces, ~5x slower.)
int32_t d2h_pageable(CtxCore &c, cudaStream_t st, uint8_t *dst, const uint8_t *src_dev, size_t bytes) {
  struct Piece { int b; size_t off, len; };
  std::vector<Piece> inflight;
  auto drain_one = [&]() -> int32_t {
    const Piece p = inflight.front();
    inflight.erase(inflight.begin());
    if (check_cuda(cudaEventSynchronize(c.ring_free[p.b]), "getter D2H wait")) return -1;
    const size_t sub = 2u << 20;
    const int64_t nsub = (int64_t)((p.len + sub - 1) / sub);
    const uint8_t *from = c.ring[p.b];
    parallel_for(c, nsub, [&](int64_t i) {
      const size_t o = (size_t)i * sub;
      memcpy(dst + p.off + o, from + o, p.len - o < sub ? p.len - o : sub);
    });
    return 0;
  };
  for (size_t off = 0; off < bytes; off += kStageBytes) {
    if ((int)inflight.size() >= kStageBuffers - 1 && drain_one()) return -1;
    const size_t len = bytes - off < kStageBytes ? bytes - off : kStageBytes;
    const int b = c.ring_acquire();
    if (b < 0) return -1;
    if (check_cuda(cudaMemcpyAsync(c.ring[b], src_dev + off, len, cudaMemcpyDeviceToHost, st), "getter D2H")) return -1;
    if (check_cuda(cudaEventRecord(c.ring_free[b], st), "getter D2H record")) return -1;
    inflight.push_back(Piece{b, off, len});
  }
  while (!inflight.empty())
    if (drain_one()) return -1;
  return 0;
}

void copy_out(CtxCore &c, uint8_t *dst, const uint8_t *src, size_t bytes) {  // pinned cache -> Bytes, on the host threads when large
  const size_t sub = 2u << 20;
  if (bytes <= 2 * sub) { memcpy(dst, src, bytes); return; }
  parallel_for(c, (int64_t)((bytes + sub - 1) / sub), [&](int64_t i) {
    const size_t o = (size_t)i * sub;
    memcpy(dst + o, src + o, bytes - o < sub ? bytes - o : sub);
  });
}

constexpr int kGetString = 4;
// the getter the reference's schema picks for a column (src/duckdb_native.c:2314-2339): what a MoonBit caller will ask for
int schema_getter_kind(const Col &col) {
  switch (col.type_id) {
    case DMB_TYPE_BOOLEAN: return kGetBool;
    case DMB_TYPE_TINYINT: case DMB_TYPE_SMALLINT: case DMB_TYPE_INTEGER: return kGetInt32;
    case DMB_TYPE_BIGINT: return kGetInt64;
    case DMB_TYPE_FLOAT: case DMB_TYPE_DOUBLE: return kGetDouble;
    default: return kGetString;
  }
}

// The reference's callers read a result column by column, one blocking FFI call each.  On the first getter call of a
// result that fits, EVERY column is converted in one pipelined pass -- copy-in of column j+1, kernel of column j and
// copy-out of column j-1 overlap on the three streams, like materialise_arrow -- into complete blobs in pinned memory,
// each for the getter its schema type selects (and the nullable flavour of the first call); the calls that follow are a
// memcpy into the Bytes.  A call the prediction missed (another getter kind / flavour) takes the on-demand path below.
constexpr uint64_t kGetterPrefetchCap = 1ull << 30;  // blob bytes held in pinned memory per result

int32_t prefetch_getters(Result *r, bool nullable) {
  r->getters_prefetched = true;  // one attempt
  NvtxRange nvtx("dmb::prefetch_getters");
  CtxCore &c = *r->core;
  const int ncols = r->column_count;
  const int64_t n = r->nrows;
  static const int kWidth[] = {4, 8, 8, 1};
  uint64_t estimate = 0;
  for (int jj = 0; jj < ncols; ++jj) {
    const Col &col = r->cols[(size_t)jj];
    const int kind = schema_getter_kind(col);
    if (kind == kGetString) {
      if (!text_supported(col)) return 0;  // (the on-demand path reports the error for that column)
      estimate += col.phys == DMB_PHYS_STRING ? col.heap_len + 14ull * (uint64_t)n : 50ull * (uint64_t)n;
      if (col.phys == DMB_PHYS_STRING && col.heap_len == 0 && col.heap_base != (const uint8_t *)DMB_HEAP_INLINE_ONLY) estimate += 32ull * (uint64_t)n;  // scattered heap: unknown yet
    } else {
      estimate += 4 + (uint64_t)n * (uint64_t)(kWidth[kind] + 1);
    }
  }
  if (ncols < 2 || estimate > kGetterPrefetchCap) return 0;
  std::vector<FixedRun> fr((size_t)ncols);
  std::vector<StringRun> sr((size_t)ncols);
  std::vector<int> kinds((size_t)ncols, -1);
  Scope sc(c);
  const int32_t row_count = r->row_count;
  for (int j = 0; j < ncols; ++j) {  // pass 1: stage + launch every column
    const Col &col = r->cols[(size_t)j];
    const int kind = schema_getter_kind(col);
    if (kind == kGetString) {
      if (run_string(r, sc, j, DMB_STR_REF_BLOB, false, nullable, &sr[(size_t)j])) return -1;
    } else {
      const GetterOp gop = getter_op(col, (GetterKind)kind);
      if (run_fixed(r, sc, j, gop.op, kWidth[kind], false, nullable, &fr[(size_t)j], gop.param)) return -1;
    }
    kinds[(size_t)j] = kind;
  }
  for (int j = 0; j < ncols; ++j) {  // pass 2: the blobs, assembled in pinned memory by the copy engine
    Col &col = r->cols[(size_t)j];
    const int kind = kinds[(size_t)j];
    if (kind == kGetString) {
      StringRun &s = sr[(size_t)j];
      if (check_cuda(cudaEventSynchronize(s.done), "string kernel wait")) return -1;
      if (s.h_ctr[1] || s.h_ctr[3]) continue;  // flagged (error, or aliased pointers that need an exact-size relaunch): on demand
      const uint64_t total_data_len = s.h_ctr[0] - s.h_ctr[2];
      const int64_t total64 = 8 + (int64_t)total_data_len + (nullable ? row_count : 0);
      if (total64 > 0x7fffffffll) continue;
      uint8_t *blob = (uint8_t *)keep_pin(r, (size_t)total64);
      if (!blob) return -1;
      const int32_t tdl = (int32_t)total_data_len;
      memcpy(blob, &row_count, 4);
      memcpy(blob + 4, &tdl, 4);
      if (check_cuda(cudaStreamWaitEvent(c.s_out, s.done, 0), "wait kernel")) return -1;
      if (total_data_len && check_cuda(cudaMemcpyAsync(blob + 8, s.d_data, (size_t)total_data_len, cudaMemcpyDeviceToHost, c.s_out), "string data D2H")) return -1;
      if (nullable && check_cuda(cudaMemcpyAsync(blob + 8 + total_data_len, s.validity.d_valid_bytes, (size_t)row_count, cudaMemcpyDeviceToHost, c.s_out), "validity D2H")) return -1;
      r->bytes_d2h += total_data_len + (nullable ? (size_t)row_count : 0);
      col.gc_blob = blob;
      col.gc_bytes = (size_t)total64;
    } else {
      const int w = kWidth[kind];
      const int64_t total64 = 4 + (int64_t)row_count * w + (nullable ? row_count : 0);
      if (total64 > 0x7fffffffll) continue;
      uint8_t *blob = (uint8_t *)keep_pin(r, (size_t)total64);
      if (!blob) return -1;
      FixedRun &f = fr[(size_t)j];
      memcpy(blob, &row_count, 4);
      const size_t vbytes = (size_t)row_count * (size_t)w;
      if (check_cuda(cudaStreamWaitEvent(c.s_out, f.done, 0), "wait kernel")) return -1;
      if (check_cuda(cudaMemcpyAsync(blob + 4, f.d_values, vbytes, cudaMemcpyDeviceToHost, c.s_out), "values D2H")) return -1;
      if (nullable && check_cuda(cudaMemcpyAsync(blob + 4 + vbytes, f.d_valid_bytes, (size_t)row_count, cudaMemcpyDeviceToHost, c.s_out), "validity D2H")) return -1;
      r->bytes_d2h += vbytes + (nullable ? (size_t)row_count : 0);
      col.gc_blob = blob;
      col.gc_bytes = (size_t)total64;
    }
    col.gc_kind = kind;
    col.gc_nullable = nullable;
  }
  if (check_cuda(cudaStreamSynchronize(c.s_out), "getter prefetch sync")) {
    for (Col &col : r->cols) col.gc_kind = -1;
    return -1;
  }
  return 0;
}

// a prefetched blob that matches the call, copied into a fresh Bytes; NULL when there is none
moonbit_bytes_t cached_blob(Result *r, int32_t col_idx, int kind, bool nullable) {
  if (!r->getters_prefetched && r->row_count > 0) {
    char saved[512];
    snprintf(saved, sizeof(saved), "%s", duckdb_mb_gpu_last_error());
    if (prefetch_getters(r, nullable)) set_error("%s", saved);  // a failed prefetch is not the caller's error: the on-demand path decides
  }
  const Col &col = r->cols[(size_t)col_idx];
  if (col.gc_kind != kind || col.gc_nullable != nullable || !col.gc_blob) return nullptr;
  moonbit_bytes_t blob = moonbit_make_bytes_raw((int32_t)col.gc_bytes);
  if (!blob) return nullptr;
  copy_out(*r->core, blob, col.gc_blob, col.gc_bytes);
  return blob;
}

// [n:i32][values][validity bytes]  (src/duckdb_native.c:2359-2454, 2516-2546, 2572-2685, 2761-2797)
moonbit_bytes_t getter_fixed(Result *r, int32_t col_idx, GetterKind kind, bool nullable) {
  if (!r) return empty_bytes();
  const int32_t row_count = r->row_count;
  if (col_idx < 0 || col_idx >= r->column_count || row_count <= 0) return empty_bytes();
  CtxCore &c = *r->core;
  std::lock_guard<std::mutex> g(c.mu);
  if (!c.bind()) return empty_bytes();
  static const int kWidth[] = {4, 8, 8, 1};
  const int w = kWidth[kind];
  const int64_t total64 = 4 + (int64_t)row_count * w + (nullable ? row_count : 0);
  if (total64 > 0x7fffffffll) {  // the reference's int32 total_size overflows here (:2371,2404)
    set_error("result blob of %lld bytes exceeds the int32 length of MoonBit Bytes", (long long)total64);
    return empty_bytes();
  }
  if (moonbit_bytes_t hit = cached_blob(r, col_idx, (int)kind, nullable)) return hit;
  const Col &col = r->cols[(size_t)col_idx];
  Scope sc(c);
  FixedRun f;
  // a type libduckdb cannot cast to a number yields zero values (getter_op)
  const GetterOp gop = getter_op(col, kind);
  if (run_fixed(r, sc, col_idx, gop.op, w, false, nullable, &f, gop.param)) return empty_bytes();
  moonbit_bytes_t blob = moonbit_make_bytes_raw((int32_t)total64);
  if (!blob) { set_error("out of memory"); return empty_bytes(); }
  memcpy(blob, &row_count, 4);
  const size_t vbytes = (size_t)row_count * (size_t)w;
  bool ok = d2h_pageable(c, c.s_compute, blob + 4, f.d_values, vbytes) == 0;
  if (ok && nullable) ok = d2h_pageable(c, c.s_compute, blob + 4 + vbytes, f.d_valid_bytes, (size_t)row_count) == 0;
  r->bytes_d2h += vbytes + (nullable ? (size_t)row_count : 0);
  if (!ok) { memset(blob, 0, (size_t)total64); }
  return blob;
}

// [n:i32][total:i32][s0\0 s1\0 ...][validity bytes]  (src/duckdb_native.c:2456-2514, 2687-2759).
// The reference counts no terminator for a NULL row in `total` but still writes one, so the
// stream it keeps is the first `total` bytes of the full NUL-terminated stream.
moonbit_bytes_t getter_string(Result *r, int32_t col_idx, bool nullable) {
  if (!r) return empty_bytes();
  const int32_t row_count = r->row_count;
  if (col_idx < 0 || col_idx >= r->column_count || row_count <= 0) return empty_bytes();
  CtxCore &c = *r->core;
  std::lock_guard<std::mutex> g(c.mu);
  if (!c.bind()) return empty_bytes();
  const Col &col = r->cols[(size_t)col_idx];
  if (!text_supported(col)) {
    // (every scalar type of the reference's stream whitelist is rendered by K7; what is left is LIST and friends)
    set_error("get_column_string: libduckdb's text rendering of column type %d is not reproduced on the device", col.type_id);
    return empty_bytes();
  }
  if (moonbit_bytes_t hit = cached_blob(r, col_idx, kGetString, nullable)) return hit;
  Scope sc(c);
  StringRun s;
  if (run_string_sync(r, sc, col_idx, DMB_STR_REF_BLOB, false, nullable, &s)) return empty_bytes();
  const uint64_t stream_total = s.h_ctr[0], nulls = s.h_ctr[2];
  const uint64_t total_data_len = stream_total - nulls;
  const int64_t total64 = 8 + (int64_t)total_data_len + (nullable ? row_count : 0);
  if (total64 > 0x7fffffffll) {  // int32 total_size overflow in the reference (:2488)
    set_error("result blob of %lld bytes exceeds the int32 length of MoonBit Bytes", (long long)total64);
    return empty_bytes();
  }
  moonbit_bytes_t blob = moonbit_make_bytes_raw((int32_t)total64);
  if (!blob) { set_error("out of memory"); return empty_bytes(); }
  const int32_t tdl = (int32_t)total_data_len;
  memcpy(blob, &row_count, 4);
  memcpy(blob + 4, &tdl, 4);
  bool ok = true;
  if (total_data_len) ok = d2h_pageable(c, c.s_compute, blob + 8, s.d_data, (size_t)total_data_len) == 0;
  if (ok && nullable) ok = d2h_pageable(c, c.s_compute, blob + 8 + total_data_len, s.validity.d_valid_bytes, (size_t)row_count) == 0;
  r->bytes_d2h += total_data_len + (nullable ? (size_t)row_count : 0);
  if (!ok) memset(blob + 8, 0, (size_t)total64 - 8);
  return blob;
}

}  // namespace
}  // namespace dmb


namespace dmb {
namespace {

// One column of the batch -> r->cols[j] (already allocated).  STRUCT fields become columns of their own appended behind
// the visible ones (Col::kids); a LIST / MAP gets a ListNode, whichever form its child came in.
bool fill_column(Result *r, int j, const dmb_host_column &hc, int64_t nch, const uint32_t *counts, int depth) {
  if (depth > 4) { set_error("column '%s': STRUCT nesting deeper than 4 levels", hc.name ? hc.name : ""); return false; }
  if (hc.type_id == DMB_TYPE_STRUCT) {
    if (!hc.struct_ || hc.struct_->nfields <= 0 || !hc.struct_->fields) { set_error("column %d: STRUCT column without fields", j); return false; }
    {
      Col &col = r->cols[(size_t)j];
      col.name = hc.name ? hc.name : "";
      col.type_id = DMB_TYPE_STRUCT;
      col.phys = DMB_PHYS_U8;  // no payload of its own: validity + descriptors only
      col.width = 1;
      col.is_struct = true;
      col.data.assign((size_t)nch, nullptr);
      if (hc.validity) {
        col.validity.assign((const void *const *)hc.validity, (const void *const *)hc.validity + nch);
        for (const void *p : col.validity) col.any_validity |= p != nullptr;
        if (!col.any_validity) col.validity.clear();
      }
    }
    for (int32_t f = 0; f < hc.struct_->nfields; ++f) {
      const int kid = (int)r->cols.size();
      r->cols.emplace_back();
      r->cols[(size_t)j].kids.push_back(kid);
      if (!fill_column(r, kid, hc.struct_->fields[f], nch, counts, depth + 1)) return false;
    }
    return true;
  }
  Col &col = r->cols[(size_t)j];
    col.name = hc.name ? hc.name : "";
    col.type_id = hc.type_id;
    col.phys = hc.phys;
    col.dec_width = hc.dec_width;
    col.dec_scale = hc.dec_scale;
    col.width = dmb_phys_width(hc.phys);
    if (col.width <= 0) { set_error("column %d: bad physical type %d", j, hc.phys); return false; }
    if (nch > 0 && !hc.data) { set_error("column %d: no data pointers", j); return false; }
    col.data.assign(hc.data, hc.data + nch);
    for (int64_t k = 0; k < nch; ++k)
      if (counts[k] && !col.data[(size_t)k]) { set_error("column %d: chunk %lld has rows but a null data pointer", j, (long long)k); return false; }
    if (hc.validity) {
      col.validity.assign((const void *const *)hc.validity, (const void *const *)hc.validity + nch);
      for (const void *p : col.validity) col.any_validity |= p != nullptr;
      if (!col.any_validity) col.validity.clear();
    }
    col.heap_base = (const uint8_t *)hc.heap_base;
    col.heap_len = hc.heap_len;
    if (hc.type_id == DMB_TYPE_ENUM) {
      if (hc.phys != DMB_PHYS_U8 && hc.phys != DMB_PHYS_U16 && hc.phys != DMB_PHYS_U32) { set_error("column %d: ENUM indices are uint8/uint16/uint32", j); return false; }
      const dmb_enum_dict *d = hc.dict;
      if (!d || !d->offsets || (d->size && d->offsets[d->size] && !d->data)) { set_error("column %d: ENUM column without a dictionary", j); return false; }
      auto dict = std::make_shared<EnumDict>();
      dict->offsets.assign(d->offsets, d->offsets + (size_t)d->size + 1);
      if (dict->offsets[0] != 0 || dict->offsets[d->size] > 0x7fffffffu) { set_error("column %d: ENUM dictionary offsets must start at 0 and stay below 2 GiB", j); return false; }
      for (uint32_t i = 0; i < d->size; ++i) {
        if (dict->offsets[i + 1] < dict->offsets[i]) { set_error("column %d: ENUM dictionary offsets are not monotonic", j); return false; }
        const uint32_t len = dict->offsets[i + 1] - dict->offsets[i];
        if (len > dict->max_len) dict->max_len = len;
      }
      if (d->offsets[d->size]) dict->data.assign(d->data, d->data + d->offsets[d->size]);
      col.dict = dict;
    }
    if (hc.type_id == DMB_TYPE_LIST || hc.type_id == DMB_TYPE_MAP) {
      const dmb_host_list *l = hc.list;
      if (col.width != 16) { set_error("column %d: LIST / MAP vectors hold 16-byte list entries (phys DMB_PHYS_U128)", j); return false; }
      if (l && l->child_col) {
        col.node = build_node(l, nch, 0);
        if (!col.node) return false;
        col.is_map = hc.type_id == DMB_TYPE_MAP;
      } else if (hc.type_id == DMB_TYPE_MAP) {
        set_error("column %d: MAP column without its STRUCT<key, value> child (dmb_host_list.child_col)", j);
        return false;
      } else {
        // the flat form: one leaf of any fixed-width type (build_node's refusals are for described children; a type without
        // an Arrow mapping fails at export, and the result's other columns still serve)
        if (!l || (nch > 0 && (!l->child_data || !l->child_sizes))) { set_error("column %d: LIST column without child vectors", j); return false; }
        if (dmb_phys_width(l->child_phys) <= 0 || l->child_phys == DMB_PHYS_STRING) { set_error("column %d: LIST child must be a fixed-width type (physical type %d)", j, l->child_phys); return false; }
        for (int64_t k = 0; k < nch; ++k)
          if (l->child_sizes[k] && !l->child_data[k]) { set_error("column %d: chunk %lld has child elements but a null child pointer", j, (long long)k); return false; }
        col.node = sized_node(l->child_sizes, nch);
        col.node->leaves.emplace_back();
        if (!leaf_from_column(flat_child(*l), nch, &col.node->leaves.back())) return false;
      }
    }
  return true;
}

}  // namespace
}  // namespace dmb

// =====================================================================================  L1
extern "C" duckdb_mb_arrow_result *duckdb_mb_gpu_result_from_chunks(duckdb_mb_gpu_ctx *ctx, const dmb_host_batch *batch) {
  if (!ctx || !ctx->core) { set_error("duckdb_mb_gpu_result_from_chunks: null context"); return nullptr; }
  if (!batch || batch->ncols < 0 || batch->nchunks < 0 || (batch->ncols > 0 && !batch->cols) || (batch->nchunks > 0 && !batch->counts)) {
    set_error("duckdb_mb_gpu_result_from_chunks: malformed batch");
    return nullptr;
  }
  std::unique_ptr<Result> r(new Result());
  r->core = ctx->core;
  r->nchunks = batch->nchunks;
  r->pinned_input = (batch->flags & DMB_BATCH_PINNED) != 0;
  r->counts.assign(batch->counts, batch->counts + batch->nchunks);
  r->row_off.assign((size_t)batch->nchunks + 1, 0);
  for (int64_t k = 0; k < batch->nchunks; ++k) {
    if (batch->counts[k] > DMB_VECTOR_SIZE) { set_error("chunk %lld has %u rows (> %d)", (long long)k, batch->counts[k], DMB_VECTOR_SIZE); return nullptr; }
    r->row_off[(size_t)k + 1] = r->row_off[(size_t)k] + batch->counts[k];
  }
  r->nrows = r->row_off[(size_t)batch->nchunks];
  r->column_count = batch->ncols;
  r->row_count = (int32_t)r->nrows;  // idx_t -> int32_t, src/duckdb_native.c:2265
  r->cols.resize((size_t)batch->ncols);
  for (int32_t j = 0; j < batch->ncols; ++j)
    if (!fill_column(r.get(), j, batch->cols[j], batch->nchunks, batch->counts, 0)) return nullptr;
  return r.release();
}

extern "C" int32_t duckdb_mb_gpu_result_materialise_arrow(duckdb_mb_arrow_result *r) {
  if (!r) { set_error("null result"); return 0; }
  std::lock_guard<std::mutex> g(r->core->mu);
  return materialise_arrow(r) == 0 ? 1 : 0;
}

extern "C" int32_t duckdb_mb_gpu_result_export_arrow(duckdb_mb_arrow_result *r, int32_t col, struct ArrowArray *out_array,
                                                     struct ArrowSchema *out_schema) {
  if (!r) { set_error("null result"); return 0; }
  if (col < -1 || col >= r->column_count) { set_error("column %d out of range", col); return 0; }
  std::lock_guard<std::mutex> g(r->core->mu);
  if (materialise_arrow(r)) return 0;
  if (col >= 0) {
    export_column(r->cols[(size_t)col].arrow, out_array, out_schema);
    return 1;
  }
  // whole batch: struct array, one child per (visible) column
  const size_t nc = (size_t)r->column_count;
  if (out_array) {
    ExportPriv *p = new ExportPriv();
    memset(out_array, 0, sizeof(*out_array));
    for (size_t j = 0; j < nc; ++j) {
      ArrowArray *ch = (ArrowArray *)calloc(1, sizeof(ArrowArray));
      export_column(r->cols[j].arrow, ch, nullptr);
      p->child_arrays.push_back(ch);
    }
    out_array->length = r->nrows;
    out_array->null_count = 0;
    out_array->n_buffers = 1;
    out_array->buffers = p->buffers;  // validity = NULL
    out_array->n_children = (int64_t)nc;
    out_array->children = p->child_arrays.data();
    out_array->release = release_array;
    out_array->private_data = p;
  }
  if (out_schema) {
    ExportPriv *p = new ExportPriv();
    memset(out_schema, 0, sizeof(*out_schema));
    for (size_t j = 0; j < nc; ++j) {
      ArrowSchema *ch = (ArrowSchema *)calloc(1, sizeof(ArrowSchema));
      export_column(r->cols[j].arrow, nullptr, ch);
      p->child_schemas.push_back(ch);
    }
    p->format = "+s";
    out_schema->format = p->format.c_str();
    out_schema->name = p->name.c_str();
    out_schema->n_children = (int64_t)nc;
    out_schema->children = p->child_schemas.data();
    out_schema->release = release_schema;
    out_schema->private_data = p;
  }
  return 1;
}

extern "C" int32_t duckdb_mb_gpu_result_typed_column(duckdb_mb_arrow_result *r, int32_t col, dmb_typed_column *out) {
  if (!r || !out) { set_error("null argument"); return 0; }
  if (col < 0 || col >= r->column_count) { set_error("column %d out of range", col); return 0; }
  std::lock_guard<std::mutex> g(r->core->mu);
  return typed_column(r, col, out) == 0 ? 1 : 0;
}

extern "C" int32_t duckdb_mb_gpu_result_text_column(duckdb_mb_arrow_result *r, int32_t col, dmb_typed_column *out) {
  if (!r || !out) { set_error("null argument"); return 0; }
  if (col < 0 || col >= r->column_count) { set_error("column %d out of range", col); return 0; }
  std::lock_guard<std::mutex> g(r->core->mu);
  return text_column(r, col, out) == 0 ? 1 : 0;
}

extern "C" int32_t duckdb_mb_gpu_result_timings(duckdb_mb_arrow_result *r, double *out4) {
  if (!r || !out4) return 0;
  out4[0] = r->t_h2d;
  out4[1] = r->t_kernels;
  out4[2] = r->t_d2h;
  out4[3] = r->t_total;
  return 1;
}

extern "C" int32_t duckdb_mb_gpu_result_link_bytes(duckdb_mb_arrow_result *r, uint64_t *out2) {
  if (!r || !out2) return 0;
  out2[0] = r->bytes_h2d;
  out2[1] = r->bytes_d2h;
  return 1;
}

// =====================================================================================  L2
extern "C" int32_t duckdb_mb_arrow_column_count(duckdb_mb_arrow_result *r) { return r ? r->column_count : 0; }
extern "C" int32_t duckdb_mb_arrow_row_count(duckdb_mb_arrow_result *r) { return r ? r->row_count : 0; }

// JSON [{"name":..,"nullable":true,"type_id":..}], type map of src/duckdb_native.c:2314-2339;
// names are not escaped and nullable is always true, like the reference (:2342-2346)
extern "C" moonbit_bytes_t duckdb_mb_arrow_schema(duckdb_mb_arrow_result *r) {
  std::string json = "[";
  if (r) {
    for (int32_t i = 0; i < r->column_count; ++i) {
      const Col &col = r->cols[(size_t)i];
      const char *type_id = "string";
      switch (col.type_id) {
        case DMB_TYPE_BOOLEAN: type_id = "bool"; break;
        case DMB_TYPE_TINYINT: case DMB_TYPE_SMALLINT: case DMB_TYPE_INTEGER: type_id = "int32"; break;
        case DMB_TYPE_BIGINT: type_id = "int64"; break;
        case DMB_TYPE_FLOAT: case DMB_TYPE_DOUBLE: type_id = "double"; break;
        default: break;
      }
      if (i) json += ",";
      json += "{\"name\":\"" + col.name + "\",\"nullable\":true,\"type_id\":\"" + type_id + "\"}";
    }
  }
  json += "]";
  moonbit_bytes_t b = moonbit_make_bytes_raw((int32_t)json.size());
  if (b) memcpy(b, json.data(), json.size());
  return b;
}

extern "C" moonbit_bytes_t duckdb_mb_arrow_get_column_int32(duckdb_mb_arrow_result *r, int32_t col) { return getter_fixed(r, col, kGetInt32, false); }
extern "C" moonbit_bytes_t duckdb_mb_arrow_get_column_int64(duckdb_mb_arrow_result *r, int32_t col) { return getter_fixed(r, col, kGetInt64, false); }
extern "C" moonbit_bytes_t duckdb_mb_arrow_get_column_double(duckdb_mb_arrow_result *r, int32_t col) { return getter_fixed(r, col, kGetDouble, false); }
extern "C" moonbit_bytes_t duckdb_mb_arrow_get_column_bool(duckdb_mb_arrow_result *r, int32_t col) { return getter_fixed(r, col, kGetBool, false); }
extern "C" moonbit_bytes_t duckdb_mb_arrow_get_column_string(duckdb_mb_arrow_result *r, int32_t col) { return getter_string(r, col, false); }
extern "C" moonbit_bytes_t duckdb_mb_arrow_get_column_int32_nullable(duckdb_mb_arrow_result *r, int32_t col) { return getter_fixed(r, col, kGetInt32, true); }
extern "C" moonbit_bytes_t duckdb_mb_arrow_get_column_int64_nullable(duckdb_mb_arrow_result *r, int32_t col) { return getter_fixed(r, col, kGetInt64, true); }
extern "C" moonbit_bytes_t duckdb_mb_arrow_get_column_double_nullable(duckdb_mb_arrow_result *r, int32_t col) { return getter_fixed(r, col, kGetDouble, true); }
extern "C" moonbit_bytes_t duckdb_mb_arrow_get_column_bool_nullable(duckdb_mb_arrow_result *r, int32_t col) { return getter_fixed(r, col, kGetBool, true); }
extern "C" moonbit_bytes_t duckdb_mb_arrow_get_column_string_nullable(duckdb_mb_arrow_result *r, int32_t col) { return getter_string(r, col, true); }

extern "C" void duckdb_mb_arrow_destroy(duckdb_mb_arrow_result *r) { free_result(r); }
extern "C" int32_t duckdb_mb_is_null_arrow_result(duckdb_mb_arrow_result *r) { return r == nullptr ? 1 : 0; }

// ------------------------------------------------------------------ per-cell drop-ins
// The reference's materialised-result and streaming-chunk accessors hand MoonBit one cell per FFI
// call (Connection::query, src/duckdb_native.mbt:477-497; ResultStream::next, :557-577).  Here the
// column's text form is produced once on the GPU (K7 + K5, cached in pinned memory by
// text_column) and a cell is a slice of it.
namespace dmb {
namespace {

// the VARCHAR rendering of cell (col, row) of the whole result, strlen-truncated like the
// reference's `strlen(value)` copy; empty Bytes for NULL, bad indices and types with no renderer
moonbit_bytes_t cell_text(Result *r, int32_t col, int64_t row) {
  if (!r || col < 0 || col >= r->column_count || row < 0 || row >= r->nrows) return empty_bytes();
  Col &c = r->cols[(size_t)col];
  dmb_typed_column t;
  {
    std::lock_guard<std::mutex> g(r->core->mu);
    if (text_column(r, col, &t)) return empty_bytes();
  }
  if (!t.valid[row]) return empty_bytes();
  const uint8_t *s = t.data + t.offsets[row];
  int32_t len = t.offsets[row + 1] - t.offsets[row];
  const void *nul = len > 0 ? memchr(s, 0, (size_t)len) : nullptr;
  if (nul) len = (int32_t)((const uint8_t *)nul - s);
  moonbit_bytes_t b = moonbit_make_bytes_raw(len);
  if (len > 0) memcpy(b, s, (size_t)len);
  return b;
}

// duckdb_validity_row_is_valid on the chunk's own mask (src/duckdb_native.c:529-534)
int32_t cell_is_null(Result *r, int32_t col, int64_t chunk, int32_t row) {
  if (!r || col < 0 || col >= r->column_count || row < 0 || row >= DMB_VECTOR_SIZE || chunk < 0 || chunk >= r->nchunks) return 1;
  const Col &c = r->cols[(size_t)col];
  const uint64_t *mask = c.validity.empty() ? nullptr : (const uint64_t *)c.validity[(size_t)chunk];
  if (!mask) return 0;
  return ((mask[row >> 6] >> (row & 63)) & 1ull) ? 0 : 1;
}

}  // namespace
}  // namespace dmb

// ---- materialised result: src/duckdb_native.c:174-254 (the handle is the same result object)
extern "C" void duckdb_mb_result_destroy(duckdb_mb_arrow_result *r) { free_result(r); }
extern "C" int32_t duckdb_mb_is_null_result(duckdb_mb_arrow_result *r) { return r == nullptr ? 1 : 0; }
extern "C" int32_t duckdb_mb_result_column_count(duckdb_mb_arrow_result *r) { return r ? r->column_count : 0; }
extern "C" int32_t duckdb_mb_result_row_count(duckdb_mb_arrow_result *r) { return r ? r->row_count : 0; }
extern "C" moonbit_bytes_t duckdb_mb_result_column_name(duckdb_mb_arrow_result *r, int32_t col) {
  if (!r || col < 0 || col >= r->column_count) return empty_bytes();
  const std::string &n = r->cols[(size_t)col].name;
  moonbit_bytes_t b = moonbit_make_bytes_raw((int32_t)n.size());
  memcpy(b, n.data(), n.size());
  return b;
}
extern "C" int32_t duckdb_mb_result_column_type(duckdb_mb_arrow_result *r, int32_t col) {
  if (!r || col < 0 || col >= r->column_count) return DMB_TYPE_INVALID;
  return r->cols[(size_t)col].type_id;
}
extern "C" int32_t duckdb_mb_result_is_null(duckdb_mb_arrow_result *r, int32_t col, int32_t row) {
  if (!r) return 1;
  if (col < 0 || col >= r->column_count || row < 0 || row >= r->nrows) return 1;  // duckdb_value_is_null: out of range counts as NULL
  // locate the chunk of the row: chunks are at most 2048 rows, so start from the regular guess
  int64_t k = row / DMB_VECTOR_SIZE;
  if (k >= r->nchunks) k = r->nchunks - 1;
  while (k > 0 && r->row_off[(size_t)k] > row) --k;
  while (k + 1 < r->nchunks && r->row_off[(size_t)k + 1] <= row) ++k;
  return cell_is_null(r, col, k, (int32_t)(row - r->row_off[(size_t)k]));
}
extern "C" moonbit_bytes_t duckdb_mb_result_value(duckdb_mb_arrow_result *r, int32_t col, int32_t row) {
  return cell_text(r, col, row);
}

// ---- streaming chunks: src/duckdb_native.c:260-667
struct duckdb_mb_stream {
  duckdb_mb_arrow_result *result;
  int64_t next_chunk;
  bool owns_result = false;
};
struct duckdb_mb_chunk {
  duckdb_mb_stream *stream;
  int64_t index;
};

static bool stream_supported_type(int32_t type_id) {  // whitelist of src/duckdb_native.c:271-303
  switch (type_id) {
    case DMB_TYPE_BOOLEAN: case DMB_TYPE_TINYINT: case DMB_TYPE_SMALLINT: case DMB_TYPE_INTEGER: case DMB_TYPE_BIGINT:
    case DMB_TYPE_UTINYINT: case DMB_TYPE_USMALLINT: case DMB_TYPE_UINTEGER: case DMB_TYPE_UBIGINT: case DMB_TYPE_FLOAT:
    case DMB_TYPE_DOUBLE: case DMB_TYPE_VARCHAR: case DMB_TYPE_BLOB: case DMB_TYPE_DATE: case DMB_TYPE_TIME:
    case DMB_TYPE_TIME_NS: case DMB_TYPE_TIME_TZ: case DMB_TYPE_TIMESTAMP: case DMB_TYPE_TIMESTAMP_TZ:
    case DMB_TYPE_TIMESTAMP_S: case DMB_TYPE_TIMESTAMP_MS: case DMB_TYPE_TIMESTAMP_NS: case DMB_TYPE_INTERVAL:
    case DMB_TYPE_HUGEINT: case DMB_TYPE_UHUGEINT: case DMB_TYPE_UUID:
      return true;
    default: return false;
  }
}

// what duckdb_mb_query_stream does after running the SQL (duckdb_mb_stream_from_result, :319-353);
// the stream does not own the result
extern "C" duckdb_mb_stream *duckdb_mb_gpu_stream_from_result(duckdb_mb_arrow_result *r) {
  if (!r) { set_error("result is null"); return nullptr; }
  for (int32_t c = 0; c < r->column_count; ++c)
    if (!stream_supported_type(r->cols[(size_t)c].type_id)) { set_error("streaming query has unsupported column type"); return nullptr; }
  duckdb_mb_stream *s = new duckdb_mb_stream();
  s->result = r;
  s->next_chunk = 0;
  return s;
}
extern "C" duckdb_mb_stream *duckdb_mb_gpu_stream_from_result_owned(duckdb_mb_arrow_result *r) {
  duckdb_mb_stream *s = duckdb_mb_gpu_stream_from_result(r);
  if (!s) { free_result(r); return nullptr; }
  s->owns_result = true;
  return s;
}
extern "C" void duckdb_mb_gpu_result_set_owner(duckdb_mb_arrow_result *r, void *owner, void (*destroy)(void *)) {
  if (!r) return;
  r->owner = destroy ? std::shared_ptr<void>(owner, destroy) : std::shared_ptr<void>();
}
extern "C" void duckdb_mb_stream_destroy(duckdb_mb_stream *s) {
  if (!s) return;
  if (s->owns_result) free_result(s->result);
  delete s;
}
extern "C" int32_t duckdb_mb_is_null_stream(duckdb_mb_stream *s) { return s == nullptr ? 1 : 0; }
extern "C" int32_t duckdb_mb_stream_column_count(duckdb_mb_stream *s) { return s ? s->result->column_count : 0; }
extern "C" moonbit_bytes_t duckdb_mb_stream_column_name(duckdb_mb_stream *s, int32_t col) {
  return s ? duckdb_mb_result_column_name(s->result, col) : empty_bytes();
}
// NULL with an empty last error at the end of the stream (:472-480)
extern "C" duckdb_mb_chunk *duckdb_mb_stream_fetch_chunk(duckdb_mb_stream *s) {
  if (!s || !s->result) { set_error("stream is null"); return nullptr; }
  if (s->next_chunk >= s->result->nchunks) { set_error("%s", ""); return nullptr; }
  duckdb_mb_chunk *c = new duckdb_mb_chunk();
  c->stream = s;
  c->index = s->next_chunk++;
  return c;
}
extern "C" void duckdb_mb_chunk_destroy(duckdb_mb_chunk *c) { delete c; }
extern "C" int32_t duckdb_mb_is_null_chunk(duckdb_mb_chunk *c) { return c == nullptr ? 1 : 0; }
extern "C" int32_t duckdb_mb_chunk_row_count(duckdb_mb_chunk *c) {
  return (c && c->stream) ? (int32_t)c->stream->result->counts[(size_t)c->index] : 0;
}
extern "C" int32_t duckdb_mb_chunk_column_count(duckdb_mb_chunk *c) { return (c && c->stream) ? c->stream->result->column_count : 0; }
extern "C" int32_t duckdb_mb_chunk_is_null(duckdb_mb_chunk *c, int32_t col, int32_t row) {
  if (!c || !c->stream) return 1;
  return cell_is_null(c->stream->result, col, c->index, row);
}
// UNPINNED format: the reference renders the cell with duckdb_value_to_string (:305-318), which no
// reference test looks at; this returns the VARCHAR cast of the cell like duckdb_mb_result_value
extern "C" moonbit_bytes_t duckdb_mb_chunk_value(duckdb_mb_chunk *c, int32_t col, int32_t row) {
  if (!c || !c->stream || row < 0) return empty_bytes();
  duckdb_mb_arrow_result *r = c->stream->result;
  if (row >= (int32_t)r->counts[(size_t)c->index]) return empty_bytes();
  return cell_text(r, col, r->row_off[(size_t)c->index] + row);
}

extern "C" double duckdb_mb_bytes_to_double(const char *bytes, int32_t offset) {
  double d;
  memcpy(&d, bytes + offset, sizeof(d));
  return d;
}

// =====================================================================================  one table over N GPUs / streams
// SURVEY.md §8e: the chunk list is cut into contiguous ranges of whole chunks; every range is an independent result on
// its own context (own GPU, own host link, own host thread) and exports an independent record batch whose utf8 offsets
// start at 0.  The only cross-GPU datum is one byte total per string column per part; their exclusive scan on the host
// gives the base a part's offsets are shifted by when one logical column is wanted (no NCCL, NVLink unused).
// The same slicing on ONE context is what feeds an ArrowArrayStream: record batches of a bounded number of rows, so a
// column with more than 2^31 string bytes (BASELINE config C3) leaves as several utf8 batches.
namespace dmb {
namespace {

// chunks [c0, c1) of `p` as a result of its own on `core` (pointer tables copied; the host vectors, dictionaries and the
// glue's owner are shared)
Result *slice_result(const Result *p, const std::shared_ptr<CtxCore> &core, int64_t c0, int64_t c1) {
  std::unique_ptr<Result> r(new Result());
  r->core = core;
  r->owner = p->owner;
  r->nchunks = c1 - c0;
  r->pinned_input = p->pinned_input;
  r->counts.assign(p->counts.begin() + c0, p->counts.begin() + c1);
  r->row_off.assign((size_t)r->nchunks + 1, 0);
  for (int64_t k = 0; k < r->nchunks; ++k) r->row_off[(size_t)k + 1] = r->row_off[(size_t)k] + r->counts[(size_t)k];
  r->nrows = r->row_off[(size_t)r->nchunks];
  r->column_count = p->column_count;
  r->row_count = (int32_t)r->nrows;
  r->cols.resize(p->cols.size());
  for (size_t j = 0; j < p->cols.size(); ++j) {
    const Col &pc = p->cols[j];
    Col &col = r->cols[j];
    static_cast<ColType &>(col) = pc;
    col.force_large = pc.force_large;
    col.dict = pc.dict ? std::make_shared<EnumDict>() : nullptr;  // device copies are per result: own dictionary object
    if (pc.dict) {
      col.dict->offsets = pc.dict->offsets;
      col.dict->data = pc.dict->data;
      col.dict->max_len = pc.dict->max_len;
    }
    col.data.assign(pc.data.begin() + c0, pc.data.begin() + c1);
    if (!pc.validity.empty()) {
      col.validity.assign(pc.validity.begin() + c0, pc.validity.begin() + c1);
      for (const void *q : col.validity) col.any_validity |= q != nullptr;
      if (!col.any_validity) col.validity.clear();
    }
    col.heap_base = pc.heap_base;
    col.heap_len = pc.heap_len;
    if (pc.phys == DMB_PHYS_STRING && pc.heap_len > 0 && pc.heap_base && pc.heap_base != (const uint8_t *)DMB_HEAP_INLINE_ONLY) {
      // a registered contiguous heap: this part stages only the span its own pointers reach
      std::vector<uint64_t> lo((size_t)(r->nchunks > 0 ? r->nchunks : 1), ~0ull), hi((size_t)(r->nchunks > 0 ? r->nchunks : 1), 0ull);
      parallel_for(*core, r->nchunks, [&](int64_t k) {
        const dmb_string_t *e = reinterpret_cast<const dmb_string_t *>(col.data[(size_t)k]);
        const void *mask = col.validity.empty() ? nullptr : col.validity[(size_t)k];
        uint64_t l = ~0ull, h = 0;
        for (uint32_t i = 0; e && i < r->counts[(size_t)k]; ++i) {
          if (!host_row_valid(mask, i) || e[i].length <= 12) continue;
          l = e[i].tail.ptr < l ? e[i].tail.ptr : l;
          h = e[i].tail.ptr + e[i].length > h ? e[i].tail.ptr + e[i].length : h;
        }
        lo[(size_t)k] = l;
        hi[(size_t)k] = h;
      });
      uint64_t l = ~0ull, h = 0;
      for (int64_t k = 0; k < r->nchunks; ++k) { l = lo[(size_t)k] < l ? lo[(size_t)k] : l; h = hi[(size_t)k] > h ? hi[(size_t)k] : h; }
      const uint64_t b0 = (uint64_t)(uintptr_t)pc.heap_base, b1 = b0 + pc.heap_len;
      if (h > l && l >= b0 && h <= b1) {  // (pointers outside the registered heap: keep the whole heap, the kernel reports them)
        const uint64_t a = l & ~15ull;  // keep the staged copy 16-byte phase-aligned with the host heap
        col.heap_base = (const uint8_t *)(uintptr_t)(a < b0 ? b0 : a);
        col.heap_len = h - (uint64_t)(uintptr_t)col.heap_base;
      } else if (h <= l) {
        col.heap_base = (const uint8_t *)DMB_HEAP_INLINE_ONLY;  // no pointer string in this part
        col.heap_len = 0;
      }
    }
    col.is_struct = pc.is_struct;
    col.kids = pc.kids;  // (the hidden field columns are sliced like every other column, at the same indices)
    col.is_map = pc.is_map;
    if (pc.node) col.node = slice_node(*pc.node, c0, c1);
  }
  return r.release();
}

}  // namespace
}  // namespace dmb

struct duckdb_mb_gpu_sharded {
  std::vector<duckdb_mb_arrow_result *> parts;
  std::vector<int64_t> first_row;  // [nparts + 1]
  std::string error;
  // stream state
  size_t next = 0;
  std::thread ahead;        // materialises part `next` while the consumer works on the one before
  int32_t ahead_rc = 0;
  std::string ahead_error;
  bool ahead_running = false;
};

namespace dmb {
namespace {

typedef duckdb_mb_gpu_sharded Sharded;

int32_t materialise_locked(Result *r, std::string *err) {
  std::lock_guard<std::mutex> g(r->core->mu);
  const int32_t rc = materialise_arrow(r);
  if (rc && err) *err = duckdb_mb_gpu_last_error();  // (thread-local: read it on the thread that failed)
  return rc;
}

// ---- ArrowArrayStream over the parts (Arrow C stream interface): one record batch per part, materialised one ahead
int stream_get_schema(struct ArrowArrayStream *st, struct ArrowSchema *out) {
  Sharded *s = reinterpret_cast<Sharded *>(st->private_data);
  if (s->parts.empty()) { s->error = "empty stream"; return 22; }
  // the schema is that of part 0 (every part agrees: same columns; string columns either all utf8 or all large_utf8)
  Result *r = s->parts[0];
  if (s->ahead_running) { s->ahead.join(); s->ahead_running = false; }
  std::string err;
  if (materialise_locked(r, &err)) { s->error = err; return 5; }
  if (!duckdb_mb_gpu_result_export_arrow(r, -1, nullptr, out)) { s->error = duckdb_mb_gpu_last_error(); return 5; }
  return 0;
}

int stream_get_next(struct ArrowArrayStream *st, struct ArrowArray *out) {
  Sharded *s = reinterpret_cast<Sharded *>(st->private_data);
  if (s->ahead_running) {
    s->ahead.join();
    s->ahead_running = false;
    if (s->ahead_rc) { s->error = s->ahead_error; return 5; }
  }
  if (s->next >= s->parts.size()) {  // end of stream: a released array
    memset(out, 0, sizeof(*out));
    return 0;
  }
  Result *r = s->parts[s->next];
  std::string err;
  if (materialise_locked(r, &err)) { s->error = err; return 5; }
  if (s->next > 0) {  // every batch must have the schema handed out by get_schema
    Result *r0 = s->parts[0];
    for (size_t j = 0; j < r->cols.size() && r0->arrow_ready; ++j)
      if (r->cols[j].arrow->format != r0->cols[j].arrow->format) {
        char buf[160];
        snprintf(buf, sizeof(buf), "record batch %zu: column %zu is '%s' but the stream's schema says '%s'", s->next, j,
                 r->cols[j].arrow->format.c_str(), r0->cols[j].arrow->format.c_str());
        s->error = buf;
        return 22;
      }
  }
  if (!duckdb_mb_gpu_result_export_arrow(r, -1, out, nullptr)) { s->error = duckdb_mb_gpu_last_error(); return 5; }
  // the exported array owns its pinned buffers: the part's device copies and pointer tables can go (part 0 stays: schema)
  if (s->next > 0) { free_result(r); s->parts[s->next] = nullptr; }
  ++s->next;
  if (s->next < s->parts.size()) {  // start on the next part while the consumer reads this one
    Result *nx = s->parts[s->next];
    s->ahead_rc = 0;
    s->ahead_running = true;
    s->ahead = std::thread([s, nx] {
      s->ahead_rc = materialise_locked(nx, &s->ahead_error);
    });
  }
  return 0;
}

const char *stream_last_error(struct ArrowArrayStream *st) {
  Sharded *s = reinterpret_cast<Sharded *>(st->private_data);
  return s->error.empty() ? nullptr : s->error.c_str();
}

void stream_release(struct ArrowArrayStream *st) {
  if (!st || !st->release) return;
  Sharded *s = reinterpret_cast<Sharded *>(st->private_data);
  if (s->ahead_running) { s->ahead.join(); s->ahead_running = false; }
  for (Result *&p : s->parts) { if (p) free_result(p); p = nullptr; }
  delete s;
  st->release = nullptr;
  st->private_data = nullptr;
}

}  // namespace
}  // namespace dmb

extern "C" duckdb_mb_gpu_sharded *duckdb_mb_gpu_result_shard(duckdb_mb_arrow_result *r, duckdb_mb_gpu_ctx *const *ctxs, int32_t nctx,
                                                            int64_t max_rows_per_part) {
  if (!r) { set_error("duckdb_mb_gpu_result_shard: null result"); return nullptr; }
  std::vector<std::shared_ptr<CtxCore>> cores;
  if (!ctxs || nctx <= 0) cores.push_back(r->core);
  else
    for (int32_t g = 0; g < nctx; ++g) {
      if (!ctxs[g] || !ctxs[g]->core) { set_error("duckdb_mb_gpu_result_shard: context %d is null", g); return nullptr; }
      cores.push_back(ctxs[g]->core);
    }
  const int64_t G = (int64_t)cores.size(), C = r->nchunks;
  std::unique_ptr<Sharded> s(new Sharded());
  // a string column that cannot be one utf8 batch in SOME part is large in every part (one schema for the table)
  const int64_t per_gpu = C > 0 ? (C + G - 1) / G : 0;  // GPU g gets chunks [g * ceil(C / G), ...)
  int64_t chunks_per_part = per_gpu;
  if (max_rows_per_part > 0) {
    const int64_t m = max_rows_per_part / DMB_VECTOR_SIZE;
    chunks_per_part = m < 1 ? 1 : (m < per_gpu ? m : per_gpu);
  }
  s->first_row.push_back(0);
  for (int64_t g = 0; g < G; ++g) {
    const int64_t g0 = g * per_gpu < C ? g * per_gpu : C, g1 = g0 + per_gpu < C ? g0 + per_gpu : C;
    if (g0 >= g1) {  // fewer chunks than contexts: this context's part is an empty record batch
      if (max_rows_per_part <= 0 || s->parts.empty()) {
        Result *part = slice_result(r, cores[(size_t)g], g0, g0);
        s->parts.push_back(part);
        s->first_row.push_back(s->first_row.back());
      }
      continue;
    }
    for (int64_t c0 = g0; c0 < g1; c0 += chunks_per_part) {
      const int64_t c1 = c0 + chunks_per_part < g1 ? c0 + chunks_per_part : g1;
      Result *part = slice_result(r, cores[(size_t)g], c0, c1);
      s->parts.push_back(part);
      s->first_row.push_back(s->first_row.back() + part->nrows);
    }
  }
  for (size_t j = 0; j < r->cols.size(); ++j) {
    bool large = false;
    for (Result *p : s->parts) {
      const Col &c = p->cols[j];
      large |= c.phys == DMB_PHYS_STRING && (c.heap_len > 0x7fffffffull || c.force_large);
    }
    if (large) for (Result *p : s->parts) p->cols[j].force_large = true;
  }
  return s.release();
}

extern "C" duckdb_mb_gpu_sharded *duckdb_mb_gpu_result_from_chunks_sharded(duckdb_mb_gpu_ctx *const *ctxs, int32_t nctx, const dmb_host_batch *batch) {
  if (!ctxs || nctx <= 0 || !ctxs[0]) { set_error("duckdb_mb_gpu_result_from_chunks_sharded: no contexts"); return nullptr; }
  duckdb_mb_arrow_result *whole = duckdb_mb_gpu_result_from_chunks(ctxs[0], batch);  // pointer tables only: nothing is staged
  if (!whole) return nullptr;
  duckdb_mb_gpu_sharded *s = duckdb_mb_gpu_result_shard(whole, ctxs, nctx, 0);
  free_result(whole);
  return s;
}

extern "C" void duckdb_mb_gpu_sharded_destroy(duckdb_mb_gpu_sharded *s) {
  if (!s) return;
  if (s->ahead_running) s->ahead.join();
  for (Result *p : s->parts) if (p) free_result(p);
  delete s;
}

extern "C" int32_t duckdb_mb_gpu_sharded_part_count(duckdb_mb_gpu_sharded *s) { return s ? (int32_t)s->parts.size() : 0; }
extern "C" duckdb_mb_arrow_result *duckdb_mb_gpu_sharded_part(duckdb_mb_gpu_sharded *s, int32_t i) {
  return (s && i >= 0 && (size_t)i < s->parts.size()) ? s->parts[(size_t)i] : nullptr;
}
extern "C" int64_t duckdb_mb_gpu_sharded_first_row(duckdb_mb_gpu_sharded *s, int32_t i) {
  return (s && i >= 0 && (size_t)i < s->first_row.size()) ? s->first_row[(size_t)i] : -1;
}

// every part on its own host thread (parts that share a context take turns: one blocking call at a time per context)
extern "C" int32_t duckdb_mb_gpu_sharded_materialise_arrow(duckdb_mb_gpu_sharded *s) {
  if (!s) { set_error("null sharded result"); return 0; }
  const size_t n = s->parts.size();
  std::vector<int32_t> rc(n, 0);
  std::vector<std::string> errs(n);
  std::vector<std::thread> th;
  for (size_t i = 0; i < n; ++i) th.emplace_back([&, i] { rc[i] = materialise_locked(s->parts[i], &errs[i]); });
  for (auto &t : th) t.join();
  for (size_t i = 0; i < n; ++i)
    if (rc[i]) { set_error("part %zu: %s", i, errs[i].c_str()); return 0; }
  // one schema for the table: if a utf8 column overflowed int32 offsets in some part only, the other parts follow
  if (n > 1)
    for (size_t j = 0; j < s->parts[0]->cols.size(); ++j) {
      bool any_large = false, any_small = false;
      for (Result *p : s->parts) {
        const std::string &f = p->cols[j].arrow->format;
        any_large |= f == "U" || f == "Z";
        any_small |= f == "u" || f == "z";
      }
      if (any_large && any_small) {
        for (Result *p : s->parts) { p->cols[j].force_large = true; p->arrow_ready = false; }
        return duckdb_mb_gpu_sharded_materialise_arrow(s);
      }
    }
  return 1;
}

// host exclusive scan of the per-part utf8 byte totals of string column `col`: out[i] = base of part i, out[nparts] = total
extern "C" int32_t duckdb_mb_gpu_sharded_string_bases(duckdb_mb_gpu_sharded *s, int32_t col, uint64_t *out) {
  if (!s || !out) { set_error("null argument"); return 0; }
  uint64_t acc = 0;
  for (size_t i = 0; i < s->parts.size(); ++i) {
    Result *p = s->parts[i];
    if (!p || !p->arrow_ready || col < 0 || col >= p->column_count) { set_error("string_bases: part %zu is not materialised / bad column", i); return 0; }
    const ArrowColOut &o = *p->cols[(size_t)col].arrow;
    if (!o.data && o.data_bytes == 0 && o.format != "u" && o.format != "U" && o.format != "z" && o.format != "Z") { set_error("string_bases: column %d is not a string column", col); return 0; }
    out[i] = acc;
    acc += o.data_bytes;
  }
  out[s->parts.size()] = acc;
  return 1;
}

// the parts as an ArrowArrayStream (one record batch each, in row order); the stream takes the handle over
extern "C" int32_t duckdb_mb_gpu_sharded_export_stream(duckdb_mb_gpu_sharded *s, struct ArrowArrayStream *out) {
  if (!s || !out) { set_error("null argument"); return 0; }
  memset(out, 0, sizeof(*out));
  out->get_schema = stream_get_schema;
  out->get_next = stream_get_next;
  out->get_last_error = stream_last_error;
  out->release = stream_release;
  out->private_data = s;
  return 1;
}

// a result as a stream of record batches of at most max_batch_rows rows (<= 0: 16 M), converted one batch ahead of the
// consumer.  Replaces the silent large_utf8 switch for columns with more than 2^31 string bytes: every batch is plain utf8.
extern "C" int32_t duckdb_mb_gpu_result_export_stream(duckdb_mb_arrow_result *r, int64_t max_batch_rows, struct ArrowArrayStream *out) {
  if (!r || !out) { set_error("null argument"); return 0; }
  duckdb_mb_gpu_sharded *s = duckdb_mb_gpu_result_shard(r, nullptr, 0, max_batch_rows > 0 ? max_batch_rows : (16ll << 20));
  if (!s) return 0;
  return duckdb_mb_gpu_sharded_export_stream(s, out);
}
