// Reverse path: Arrow record batches (or rows buffered column-wise) -> DuckDB DataChunk vectors,
// gated by the appender protocol of the reference (src/duckdb_appender_state_machine.mbt:54-239).
//
// The reference appends one cell per FFI call (src/duckdb_native.mbt:974-1058 ->
// src/duckdb_native.c:1100-1235).  Here a whole record batch is converted by kernels_reverse.cu in
// sub-batches of a few million rows: copy-in of sub-batch b+1, the kernels of b and copy-out of
// b-1 overlap on the context's three streams, and every finished 2048-row chunk is handed to the
// sink in the layout duckdb_append_data_chunk takes (src/duckdb_native.c:2109-2132).
//
// The row-at-a-time calls of the reference (begin_row / append_* / end_row) are kept as a
// column-wise host buffer that is converted by the same kernels on flush, so the state machine
// is the reference's own.

#include <chrono>
#include <math.h>
#include <stdarg.h>
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

enum { kNotCreated = 0, kReady = 1, kRowInProgress = 2, kFlushed = 3, kClosed = 4, kError = 5 };

struct RowBuf {  // one column of buffered rows (row API)
  int width = 0;               // bytes per value; 0: string
  // DECIMAL: the table column's width / scale (duckdb_mb_gpu_appender_set_decimal; 0: not declared yet, the first
  // DECIMAL cell or Arrow batch declares it); values buffered as int128.  Arrow batches narrow to this width too.
  int32_t dec_prec = 0, dec_scale = 0;
  std::vector<uint8_t> values, valid;
  std::vector<int32_t> offsets;  // strings: n+1 entries
  std::vector<uint8_t> data;
};

// one column of a conversion request (host pointers, whole batch)
struct ColInput {
  int rev_op = 0, w_in = 0, w_out = 0;
  bool is_string = false, large = false, is_bits = false, is_list = false;
  const uint8_t *values = nullptr;       // fixed: first value of the slice; bits: bitmap base
  const uint8_t *validity = nullptr;     // Arrow bitmap base or NULL
  int64_t bit_offset = 0;                // array offset in bits (validity and bool values)
  const uint8_t *valid_bytes = nullptr;  // row API: one byte per row instead of a bitmap
  const uint8_t *offsets = nullptr;      // strings, lists: first offset of the slice
  const uint8_t *data = nullptr;         // strings: Arrow data buffer base
  const ColInput *child = nullptr;       // lists: the child array, its rows are the list elements
  int64_t child_len = 0;                 // lists: elements in the child array
};

// the table's child type of a LIST column (duckdb_mb_gpu_appender_set_list); type_id 0: not declared
struct ListDecl {
  int32_t type_id = 0, dec_width = 0, dec_scale = 0;
};

// what duckdb_mb_gpu_appender_list_child hands out during a sink call, per LIST column
struct SinkList {
  const uint8_t *values = nullptr;  // the sub-batch's child values, dense
  const uint64_t *words = nullptr;  // the sub-batch's child masks, chunk k at cword[k]
  const int64_t *bounds = nullptr;  // Arrow offsets at the sub-batch's chunk boundaries
  const int64_t *cword = nullptr;
  int w = 0;                        // bytes per child value
};

}  // namespace
}  // namespace dmb

using namespace dmb;

struct duckdb_mb_gpu_appender {
  std::shared_ptr<CtxCore> core;
  int32_t ncols = 0;
  std::vector<int32_t> type_ids;
  dmb_chunk_sink sink = nullptr;
  void *user = nullptr;
  dmb_appender_flush_hook on_flush = nullptr;      // glue: duckdb_appender_flush after the chunks have been handed over
  dmb_appender_destroy_hook on_destroy = nullptr;  // glue: duckdb_appender_destroy + free of `user`
  int state = kNotCreated;
  int cur_col = 0;
  int64_t row_count = 0, flushed_row_count = 0, buffered_rows = 0;
  char error[256] = {0};
  std::vector<RowBuf> rows;
  std::vector<ListDecl> lists;
  std::vector<SinkList> sink_lists;  // valid while sink_chunk >= 0: chunk sink_chunk of the sub-batch being handed over
  int64_t sink_chunk = -1;
  int64_t sub_rows = 4 << 20;
  int64_t list_child_cap = 0;  // kListChildCap unless DMB_REV_LIST_CHILD_CAP says otherwise
  double t[4] = {0, 0, 0, 0};
  uint64_t bytes_h2d = 0, bytes_d2h = 0;
};

namespace dmb {
namespace {

typedef duckdb_mb_gpu_appender App;

int32_t fail(App *a, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(a->error, sizeof(a->error), fmt, ap);
  va_end(ap);
  set_error("%s", a->error);
  return 0;
}

// any command the model does not allow in the current state moves it to Error
// (src/duckdb_appender_state_machine.mbt:228-238); Closed and Error are sticky (:218-227)
int32_t illegal(App *a, const char *cmd) {
  if (a->state == kClosed) return fail(a, "%s: appender is closed", cmd);
  if (a->state == kError) return fail(a, "%s: appender is in the error state", cmd);
  static const char *names[] = {"NotCreated", "Ready", "RowInProgress", "Flushed", "Closed", "Error"};
  fail(a, "%s is not allowed in state %s", cmd, names[a->state]);
  a->state = kError;
  return 0;
}

int row_width(int32_t type_id) {
  switch (type_id) {
    case DMB_TYPE_BOOLEAN: case DMB_TYPE_TINYINT: case DMB_TYPE_UTINYINT: return 1;
    case DMB_TYPE_SMALLINT: case DMB_TYPE_USMALLINT: return 2;
    case DMB_TYPE_INTEGER: case DMB_TYPE_UINTEGER: case DMB_TYPE_FLOAT: case DMB_TYPE_DATE: return 4;
    case DMB_TYPE_BIGINT: case DMB_TYPE_UBIGINT: case DMB_TYPE_DOUBLE: case DMB_TYPE_TIMESTAMP:
    case DMB_TYPE_TIMESTAMP_S: case DMB_TYPE_TIMESTAMP_MS: case DMB_TYPE_TIMESTAMP_NS: case DMB_TYPE_TIMESTAMP_TZ:
    case DMB_TYPE_TIME: case DMB_TYPE_TIME_NS: return 8;
    case DMB_TYPE_VARCHAR: case DMB_TYPE_BLOB: return 0;
    case DMB_TYPE_INTERVAL: case DMB_TYPE_DECIMAL: return 16;  // DECIMAL: int128 in the buffer, narrowed on flush
    default: return -1;
  }
}

int copy_op(int w) {
  switch (w) {
    case 1: return DMB_REV_COPY1;
    case 2: return DMB_REV_COPY2;
    case 4: return DMB_REV_COPY4;
    case 8: return DMB_REV_COPY8;
    default: return DMB_REV_COPY16;
  }
}

// An Arrow decimal `fmt` ("d:p,s" or "d:p,s,bits") into a column of DuckDB DECIMAL(*w, *s); HUGEINT is DECIMAL(38, 0).
// The values must be decimal128 with the column's scale and a precision that fits its width; they are narrowed to the
// column's physical width (int16 / int32 / int64 / int128 for w <= 4 / 9 / 18 / 38), which keeps every value within
// the Arrow precision exact.  *w == 0: the column is not declared yet, and this Arrow type declares it.
bool map_decimal(App *a, int c, const char *what, const char *fmt, int32_t type_id, int32_t *w, int32_t *s, ColInput *in) {
  // d:p,s[,bits]: each field one to three decimal digits, nothing else
  long f[3] = {0, 0, 128};
  int nf = 0;
  const char *q = fmt + 2;
  for (; nf < 3; ++nf) {
    int digits = 0;
    for (f[nf] = 0; *q >= '0' && *q <= '9' && digits < 3; ++q, ++digits) f[nf] = 10 * f[nf] + (*q - '0');
    if (!digits || (*q != ',' && *q != '\0')) break;
    if (*q++ == '\0') { ++nf; break; }
  }
  const long p = f[0], sc = f[1], bits = f[2];
  char col[32];
  if (type_id == DMB_TYPE_HUGEINT) snprintf(col, sizeof(col), "HUGEINT");
  else if (*w) snprintf(col, sizeof(col), "DECIMAL(%d,%d)", *w, *s);
  else snprintf(col, sizeof(col), "DECIMAL");
  if (nf < 2 || q[-1] != '\0') {
    fail(a, "column %d: Arrow %s '%s' is not a decimal format", c, what, fmt);
    return false;
  }
  if (bits != 128) {
    fail(a, "column %d: Arrow %s '%s' is a %ld-bit decimal; only decimal128 can be appended to a %s column", c, what, fmt, bits, col);
    return false;
  }
  if (p < 1 || p > 38 || sc > p) {
    fail(a, "column %d: Arrow %s '%s' is not a DECIMAL(width, scale) DuckDB can store", c, what, fmt);
    return false;
  }
  if (*w == 0) { *w = (int32_t)p; *s = (int32_t)sc; }
  if (sc != *s) {
    fail(a, "column %d: Arrow %s '%s' has scale %ld; the column is %s", c, what, fmt, sc, col);
    return false;
  }
  if (p > *w) {
    fail(a, "column %d: Arrow %s '%s' has precision %ld; the column is %s", c, what, fmt, p, col);
    return false;
  }
  in->w_in = 16;
  if (*w <= 4) { in->rev_op = DMB_REV_I128_TO_I16; in->w_out = 2; }
  else if (*w <= 9) { in->rev_op = DMB_REV_I128_TO_I32; in->w_out = 4; }
  else if (*w <= 18) { in->rev_op = DMB_REV_I128_TO_I64; in->w_out = 8; }
  else { in->rev_op = DMB_REV_COPY16; in->w_out = 16; }
  return true;
}

// Arrow format string of a child -> conversion for a DuckDB column of `type_id`; `dec_w` / `dec_s`: the column's
// DECIMAL(w, s) when it is one (w == 0: not declared yet, set from the Arrow type)
bool map_format(App *a, int c, const char *what, const char *fmt, int32_t type_id, int32_t *dec_w, int32_t *dec_s, ColInput *in) {
  auto fixed = [&](int w) { in->rev_op = copy_op(w); in->w_in = w; in->w_out = w; return true; };
  auto is = [&](const char *f) { return strcmp(fmt, f) == 0; };
  auto starts = [&](const char *f) { return strncmp(fmt, f, strlen(f)) == 0; };
  switch (type_id) {
    case DMB_TYPE_BOOLEAN:
      if (is("b")) { in->rev_op = DMB_REV_BITS_TO_BOOL; in->is_bits = true; in->w_in = 0; in->w_out = 1; return true; }
      break;
    case DMB_TYPE_TINYINT: if (is("c")) return fixed(1); break;
    case DMB_TYPE_UTINYINT: if (is("C")) return fixed(1); break;
    case DMB_TYPE_SMALLINT: if (is("s")) return fixed(2); break;
    case DMB_TYPE_USMALLINT: if (is("S")) return fixed(2); break;
    case DMB_TYPE_INTEGER: if (is("i")) return fixed(4); break;
    case DMB_TYPE_UINTEGER: if (is("I")) return fixed(4); break;
    case DMB_TYPE_FLOAT: if (is("f")) return fixed(4); break;
    case DMB_TYPE_DATE: if (is("tdD")) return fixed(4); break;
    case DMB_TYPE_BIGINT: if (is("l")) return fixed(8); break;
    case DMB_TYPE_UBIGINT: if (is("L")) return fixed(8); break;
    case DMB_TYPE_DOUBLE: if (is("g")) return fixed(8); break;
    case DMB_TYPE_TIME: if (is("ttu")) return fixed(8); break;
    case DMB_TYPE_TIME_NS: if (is("ttn")) return fixed(8); break;
    case DMB_TYPE_TIME_TZ: if (is("L")) return fixed(8); break;
    case DMB_TYPE_TIMESTAMP: case DMB_TYPE_TIMESTAMP_TZ: if (starts("tsu:")) return fixed(8); break;
    case DMB_TYPE_TIMESTAMP_S: if (starts("tss:")) return fixed(8); break;
    case DMB_TYPE_TIMESTAMP_MS: if (starts("tsm:")) return fixed(8); break;
    case DMB_TYPE_TIMESTAMP_NS: if (starts("tsn:")) return fixed(8); break;
    case DMB_TYPE_HUGEINT:
      if (starts("d:")) {  // the unscaled integer of a decimal128 with scale 0
        int32_t w = 38, s = 0;
        return map_decimal(a, c, what, fmt, type_id, &w, &s, in);
      }
      break;
    case DMB_TYPE_UHUGEINT: case DMB_TYPE_UUID: if (is("w:16")) return fixed(16); break;
    case DMB_TYPE_DECIMAL: if (starts("d:")) return map_decimal(a, c, what, fmt, type_id, dec_w, dec_s, in); break;
    case DMB_TYPE_VARCHAR:
      if (is("u") || is("U")) { in->is_string = true; in->large = is("U"); in->w_out = 16; return true; }
      break;
    case DMB_TYPE_BLOB:
      if (is("z") || is("Z")) { in->is_string = true; in->large = is("Z"); in->w_out = 16; return true; }
      break;
    default: break;
  }
  fail(a, "column %d: Arrow %s '%s' cannot be appended to a column of DuckDB type %d", c, what, fmt, type_id);
  return false;
}

// The child elements a sub-batch may hold per LIST column: a sub-batch ends at the 2048-row boundary before the chunk
// that would take a LIST column past this many elements, but always holds at least one chunk, so one chunk's child
// range is never split.  It bounds a slot's child buffers: 16 M elements are 256 MB of string_t or HUGEINT values.
// DMB_REV_LIST_CHILD_CAP overrides it (tests force several sub-batches with it).
constexpr int64_t kListChildCap = 16 << 20;

bool grow(Scope &sc, uint8_t *&p, size_t &cap, size_t need, bool pinned = false) {
  if (p && need <= cap) return true;  // the old block returns to the pool with the scope
  cap = need + need / 8 + 64;
  p = (uint8_t *)(pinned ? sc.palloc(cap) : sc.dalloc(cap));
  return p != nullptr;
}

struct ListOut {  // one LIST column of a slot: the child vectors of the sub-batch and where each chunk's mask starts
  uint8_t *d_child = nullptr, *h_child = nullptr;
  uint8_t *d_words = nullptr, *h_words = nullptr;
  size_t child_cap = 0, h_child_cap = 0, words_cap = 0, h_words_cap = 0;
  int64_t *d_cword = nullptr, *h_cword = nullptr;
  int64_t child_bytes = 0, words = 0;
};

struct Slot {  // device + pinned buffers of one in-flight sub-batch
  std::vector<uint8_t *> d_out, h_out;
  std::vector<uint64_t *> d_val, h_val;
  std::vector<ListOut> lists;                     // [ncols], used by LIST columns
  unsigned int *d_err = nullptr, *h_err = nullptr;  // [ncols]: rev_list_kernel error flags
  cudaEvent_t ev_out = nullptr;
  int64_t r0 = 0, r1 = 0;
  bool busy = false;
};

int32_t sink_slot(App *a, Slot &s, const std::vector<ColInput> &cols, const std::vector<std::vector<int64_t>> &bounds) {
  if (!s.busy) return 1;
  if (check_cuda(cudaEventSynchronize(s.ev_out), "appender copy-out wait")) return fail(a, "%s", duckdb_mb_gpu_last_error());
  s.busy = false;
  const int nc = (int)cols.size();
  for (int c = 0; c < nc; ++c)  // a malformed sub-batch reaches no sink
    if (cols[(size_t)c].is_list && s.h_err[c])
      return fail(a, "column %d: Arrow list offsets decrease within rows [%lld, %lld)", c, (long long)s.r0, (long long)s.r1);
  if (!a->sink) return 1;
  std::vector<const void *> vd((size_t)nc);
  std::vector<const uint64_t *> vv((size_t)nc);
  a->sink_lists.assign((size_t)nc, SinkList());
  for (int c = 0; c < nc; ++c)
    if (cols[(size_t)c].is_list) {
      const ListOut &lo = s.lists[(size_t)c];
      a->sink_lists[(size_t)c] = SinkList{lo.h_child, (const uint64_t *)lo.h_words, bounds[(size_t)c].data() + s.r0 / DMB_VECTOR_SIZE,
                                          lo.h_cword, cols[(size_t)c].child->w_out};
    }
  for (int64_t r = s.r0, k = 0; r < s.r1; r += DMB_VECTOR_SIZE, ++k) {
    const uint32_t count = (uint32_t)(s.r1 - r < DMB_VECTOR_SIZE ? s.r1 - r : DMB_VECTOR_SIZE);
    for (int c = 0; c < nc; ++c) {
      vd[(size_t)c] = s.h_out[(size_t)c] + (size_t)k * DMB_VECTOR_SIZE * (size_t)cols[(size_t)c].w_out;
      vv[(size_t)c] = s.h_val[(size_t)c] + (size_t)k * DMB_VALIDITY_WORDS;
    }
    a->sink_chunk = k;
    const int32_t ok = a->sink(a->user, nc, count, vd.data(), vv.data());
    a->sink_chunk = -1;
    if (!ok) return fail(a, "chunk sink aborted at row %lld", (long long)r);
  }
  return 1;
}

struct InBuf {  // device inputs of one column in one slot
  uint8_t *values = nullptr, *validity = nullptr, *offsets = nullptr, *data = nullptr;
  uint8_t *masks = nullptr;  // row API: the masks built from the validity bytes
  size_t values_cap = 0, validity_cap = 0, offsets_cap = 0, data_cap = 0;
};

// bits [p0, p1) of an Arrow bitmap -> `dst` (grown as needed); returns the bit offset of p0 there, -1 on failure
int64_t stage_bits(App *a, Scope &sc, uint8_t *&dst, size_t &cap, const uint8_t *bm, int64_t p0, int64_t p1) {
  CtxCore &c = *a->core;
  const int64_t byte0 = p0 >> 3, byte1 = (p1 + 7) >> 3;
  if (!grow(sc, dst, cap, (size_t)(byte1 - byte0) + 16) ||
      stage_contiguous(c, c.s_in, dst, bm + byte0, (size_t)(byte1 - byte0), -1, &a->bytes_h2d)) return -1;
  return p0 & 7;
}

// Arrow offset of `row` (strings, lists), read on the host
int64_t offset_at(const ColInput &ci, int64_t row) {
  if (ci.large) { int64_t v; memcpy(&v, ci.offsets + 8 * row, 8); return v; }
  int32_t v; memcpy(&v, ci.offsets + 4 * row, 4); return v;
}

// Stage Arrow rows [r0, r1) of a column that is not a LIST and describe its conversion: `*fj` for a fixed-width
// column, `*sj` for strings (the one that applies is filled).  `*d_validity` / `*bit_off`: the staged bitmap.
int32_t stage_rows(App *a, Scope &sc, const ColInput &ci, InBuf &ib, int col, int64_t r0, int64_t r1, void *out, uint64_t *out_validity,
                   dmb_rev_fixed_job *fj, dmb_rev_string_job *sj, const uint8_t **d_validity, int64_t *bit_off) {
  CtxCore &c = *a->core;
  const int64_t n = r1 - r0;
  *d_validity = nullptr;
  *bit_off = 0;
  if (ci.validity) {
    *bit_off = stage_bits(a, sc, ib.validity, ib.validity_cap, ci.validity, ci.bit_offset + r0, ci.bit_offset + r1);
    if (*bit_off < 0) return fail(a, "%s", duckdb_mb_gpu_last_error());
    *d_validity = ib.validity;
  } else if (ci.valid_bytes) {  // row API: bytes here, masks built from them by dmb_dev_valid_bytes_to_masks
    if (stage_contiguous(c, c.s_in, ib.validity, ci.valid_bytes + r0, (size_t)n, -1, &a->bytes_h2d)) return fail(a, "%s", duckdb_mb_gpu_last_error());
    *d_validity = ib.masks;
  }
  if (ci.is_string) {
    const int ow = ci.large ? 8 : 4;
    if (!grow(sc, ib.offsets, ib.offsets_cap, (size_t)(n + 1) * (size_t)ow + 16) ||
        stage_contiguous(c, c.s_in, ib.offsets, ci.offsets + (size_t)r0 * (size_t)ow, (size_t)(n + 1) * (size_t)ow, -1, &a->bytes_h2d))
      return fail(a, "%s", duckdb_mb_gpu_last_error());
    const int64_t o_first = offset_at(ci, r0), o_last = offset_at(ci, r1);
    if (o_last < o_first || o_first < 0) return fail(a, "column %d: utf8 offsets are not monotonic", col);
    const size_t dbytes = (size_t)(o_last - o_first);
    if (!grow(sc, ib.data, ib.data_cap, dbytes + 64)) return fail(a, "%s", duckdb_mb_gpu_last_error());
    if (dbytes && stage_contiguous(c, c.s_in, ib.data, ci.data + o_first, dbytes, -1, &a->bytes_h2d)) return fail(a, "%s", duckdb_mb_gpu_last_error());
    memset(sj, 0, sizeof(*sj));
    sj->in_offsets = ib.offsets;
    sj->in_data = ib.data - o_first;  // indexed by absolute Arrow offsets
    sj->in_validity = *d_validity;
    sj->in_bit_offset = *bit_off;
    sj->data_host_base = (uint64_t)(uintptr_t)ci.data;
    sj->out = (dmb_string_t *)out;
    sj->out_validity = out_validity;
    sj->large_offsets = ci.large ? 1 : 0;
    return 1;
  }
  memset(fj, 0, sizeof(*fj));
  int64_t values_bit_off = *bit_off;
  if (ci.is_bits) {
    values_bit_off = stage_bits(a, sc, ib.values, ib.values_cap, ci.values, ci.bit_offset + r0, ci.bit_offset + r1);  // same array offset as the validity bitmap
    if (values_bit_off < 0) return fail(a, "%s", duckdb_mb_gpu_last_error());
  } else {
    if (!grow(sc, ib.values, ib.values_cap, (size_t)n * (size_t)ci.w_in + 16) ||
        stage_contiguous(c, c.s_in, ib.values, ci.values + (size_t)r0 * (size_t)ci.w_in, (size_t)n * (size_t)ci.w_in, -1, &a->bytes_h2d))
      return fail(a, "%s", duckdb_mb_gpu_last_error());
  }
  fj->in_values = ib.values;
  fj->in_validity = *d_validity;
  fj->in_bit_offset = values_bit_off;
  fj->out_data = out;
  fj->out_validity = out_validity;
  fj->op = ci.rev_op;
  return 1;
}

}  // namespace
}  // namespace dmb

// end chunk (exclusive) of the sub-batch that starts at chunk k0: at most max_chunks chunks, and no LIST column holds
// more than child_cap elements unless the sub-batch is that one chunk
extern "C" int64_t dmb_rev_list_cut(const int64_t *const *bounds, int32_t nlists, int64_t nchunks, int64_t k0, int64_t max_chunks,
                                    int64_t child_cap) {
  const int64_t last = k0 + max_chunks < nchunks ? k0 + max_chunks : nchunks;
  int64_t k1 = k0 + 1;
  for (; k1 < last; ++k1) {
    bool fits = true;
    for (int32_t l = 0; l < nlists && fits; ++l) fits = bounds[l][k1 + 1] - bounds[l][k0] <= child_cap;
    if (!fits) break;
  }
  return k1;
}

namespace dmb {
namespace {

// convert `nrows` rows described by `cols` and hand the chunks to the sink
int32_t convert_rows(App *a, const std::vector<ColInput> &cols, int64_t nrows) {
  if (nrows <= 0) return 1;
  CtxCore &c = *a->core;
  std::lock_guard<std::mutex> g(c.mu);
  if (!c.bind()) return fail(a, "%s", duckdb_mb_gpu_last_error());
  const double t0 = now_ms();
  const int nc = (int)cols.size();
  int64_t sub = a->sub_rows < nrows ? a->sub_rows : ((nrows + DMB_VECTOR_SIZE - 1) / DMB_VECTOR_SIZE) * DMB_VECTOR_SIZE;
  const int64_t sub_chunks = sub / DMB_VECTOR_SIZE;
  // LIST columns: the Arrow offsets at every chunk boundary, read once; they cut the sub-batches and locate each
  // chunk's child range
  const int64_t nchunks = (nrows + DMB_VECTOR_SIZE - 1) / DMB_VECTOR_SIZE;
  std::vector<std::vector<int64_t>> bounds((size_t)nc);
  std::vector<const int64_t *> list_bounds;
  for (int j = 0; j < nc; ++j) {
    const ColInput &ci = cols[(size_t)j];
    if (!ci.is_list) continue;
    std::vector<int64_t> &b = bounds[(size_t)j];
    b.resize((size_t)nchunks + 1);
    for (int64_t k = 0; k <= nchunks; ++k) b[(size_t)k] = offset_at(ci, k * DMB_VECTOR_SIZE < nrows ? k * DMB_VECTOR_SIZE : nrows);
    for (int64_t k = 0; k < nchunks; ++k)
      if (b[(size_t)k + 1] < b[(size_t)k]) return fail(a, "column %d: Arrow list offsets decrease within rows [%lld, %lld)", j, (long long)(k * DMB_VECTOR_SIZE), (long long)((k + 1) * DMB_VECTOR_SIZE < nrows ? (k + 1) * DMB_VECTOR_SIZE : nrows));
    if (b[0] < 0 || b[(size_t)nchunks] > ci.child_len) return fail(a, "column %d: Arrow list offsets leave the child array (%lld elements)", j, (long long)ci.child_len);
    list_bounds.push_back(b.data());
  }
  std::vector<int64_t> cuts(1, 0);  // sub-batch b: chunks [cuts[b], cuts[b+1])
  while (cuts.back() < nchunks)
    cuts.push_back(dmb_rev_list_cut(list_bounds.data(), (int32_t)list_bounds.size(), nchunks, cuts.back(), sub_chunks, a->list_child_cap));
  Slot slots[2];
  Scope sc(c);
  cudaEvent_t in0 = sc.event(true), in1 = sc.event(true), out0 = sc.event(true), out1 = sc.event(true);
  if (!in0 || !in1 || !out0 || !out1) return fail(a, "%s", duckdb_mb_gpu_last_error());
  const int nslots = cuts.size() > 2 ? 2 : 1;
  for (int s = 0; s < nslots; ++s) {
    slots[s].ev_out = sc.event(false);
    slots[s].lists.resize((size_t)nc);
    slots[s].d_err = (unsigned int *)sc.dalloc(sizeof(unsigned int) * (size_t)nc);
    slots[s].h_err = (unsigned int *)sc.palloc(sizeof(unsigned int) * (size_t)nc);
    if (!slots[s].ev_out || !slots[s].d_err || !slots[s].h_err) return fail(a, "%s", duckdb_mb_gpu_last_error());
    for (int j = 0; j < nc; ++j) {
      const size_t ob = (size_t)sub * (size_t)cols[(size_t)j].w_out, vb = (size_t)sub_chunks * DMB_VALIDITY_WORDS * 8;
      uint8_t *d = (uint8_t *)sc.dalloc(ob), *h = (uint8_t *)sc.palloc(ob);
      uint64_t *dv = (uint64_t *)sc.dalloc(vb), *hv = (uint64_t *)sc.palloc(vb);
      if (!d || !h || !dv || !hv) return fail(a, "%s", duckdb_mb_gpu_last_error());
      slots[s].d_out.push_back(d);
      slots[s].h_out.push_back(h);
      slots[s].d_val.push_back(dv);
      slots[s].h_val.push_back(hv);
      if (cols[(size_t)j].is_list) {
        ListOut &lo = slots[s].lists[(size_t)j];
        lo.d_cword = (int64_t *)sc.dalloc(sizeof(int64_t) * (size_t)(sub_chunks + 1));
        lo.h_cword = (int64_t *)sc.palloc(sizeof(int64_t) * (size_t)(sub_chunks + 1));
        if (!lo.d_cword || !lo.h_cword) return fail(a, "%s", duckdb_mb_gpu_last_error());
      }
    }
  }
  // per-slot device inputs: [slot][column], and the child arrays of LIST columns; sized up front for the columns that
  // are not LISTs, grown on demand for the child ranges
  std::vector<InBuf> inbuf((size_t)nslots * (size_t)nc), childbuf((size_t)nslots * (size_t)nc);
  for (int s = 0; s < nslots; ++s)
    for (int j = 0; j < nc; ++j) {
      const ColInput &ci = cols[(size_t)j];
      InBuf &ib = inbuf[(size_t)s * (size_t)nc + (size_t)j];
      bool ok = true;
      if (ci.is_string || ci.is_list) ok = grow(sc, ib.offsets, ib.offsets_cap, (size_t)(sub + 1) * (ci.large ? 8 : 4) + 64);
      else ok = grow(sc, ib.values, ib.values_cap, ci.is_bits ? (size_t)(sub / 8 + 80) : (size_t)sub * (size_t)ci.w_in + 64);
      if (ci.validity) ok = ok && grow(sc, ib.validity, ib.validity_cap, (size_t)(sub / 8 + 16) + 64);
      else if (ci.valid_bytes) {
        ok = ok && grow(sc, ib.validity, ib.validity_cap, (size_t)sub + 64);
        ib.masks = (uint8_t *)sc.dalloc((size_t)(sub / 8) + 64);
        ok = ok && ib.masks;
      }
      if (!ok) return fail(a, "%s", duckdb_mb_gpu_last_error());
    }
  // per slot: nc jobs of the columns, then one job per LIST column with a fixed-width child (a launch of its own)
  dmb_rev_fixed_job *h_jobs = (dmb_rev_fixed_job *)sc.palloc(sizeof(dmb_rev_fixed_job) * (size_t)nc * 4);
  dmb_rev_fixed_job *d_jobs = (dmb_rev_fixed_job *)sc.dalloc(sizeof(dmb_rev_fixed_job) * (size_t)nc * 4);
  if (!h_jobs || !d_jobs) return fail(a, "%s", duckdb_mb_gpu_last_error());
  cudaEventRecord(in0, c.s_in);
  cudaEventRecord(out0, c.s_out);
  for (size_t b = 0; b + 1 < cuts.size(); ++b) {
    const int64_t r0 = cuts[b] * DMB_VECTOR_SIZE, r1 = cuts[b + 1] * DMB_VECTOR_SIZE < nrows ? cuts[b + 1] * DMB_VECTOR_SIZE : nrows;
    const int64_t n = r1 - r0;
    const int64_t nch = cuts[b + 1] - cuts[b];
    const int si = (int)(b % (size_t)nslots);
    Slot &slot = slots[si];
    if (!sink_slot(a, slot, cols, bounds)) return 0;  // the slot's previous sub-batch leaves first
    // the job array of this slot is reused as well: its previous launch has completed (sink_slot waited)
    dmb_rev_fixed_job *hj = h_jobs + (size_t)si * (size_t)nc * 2, *dj = d_jobs + (size_t)si * (size_t)nc * 2;
    int nfixed = 0, nchild_fixed = 0;
    cudaEvent_t ev_in = sc.event(false), ev_k = sc.event(false), k0 = sc.event(true), k1 = sc.event(true);
    if (!ev_in || !ev_k || !k0 || !k1) return fail(a, "%s", duckdb_mb_gpu_last_error());
    std::vector<dmb_rev_string_job> strs;
    std::vector<dmb_rev_list_job> lists;
    std::vector<int64_t> child_rows;  // element count of each child job: fixed-width ones first, in job order
    std::vector<int64_t> str_rows;
    std::vector<int> masks_from_bytes;  // columns
    for (int j = 0; j < nc; ++j) {
      const ColInput &ci = cols[(size_t)j];
      InBuf &ib = inbuf[(size_t)si * (size_t)nc + (size_t)j];
      const uint8_t *d_validity = nullptr;
      int64_t bit_off = 0;
      if (!ci.is_list) {
        dmb_rev_string_job sj;
        if (!stage_rows(a, sc, ci, ib, j, r0, r1, slot.d_out[(size_t)j], slot.d_val[(size_t)j], &hj[nfixed], &sj, &d_validity, &bit_off)) return 0;
        if (ci.valid_bytes) masks_from_bytes.push_back(j);
        if (ci.is_string) { strs.push_back(sj); str_rows.push_back(n); }
        else ++nfixed;
        continue;
      }
      // LIST: the list offsets and bitmap, then the child range [e0, e1) as a dense column of its own
      const ColInput &cc = *ci.child;
      ListOut &lo = slot.lists[(size_t)j];
      const int64_t *bnd = bounds[(size_t)j].data() + cuts[b];
      const int64_t e0 = bnd[0], e1 = bnd[nch], ne = e1 - e0;
      const int ow = ci.large ? 8 : 4;
      if (ci.validity) {
        bit_off = stage_bits(a, sc, ib.validity, ib.validity_cap, ci.validity, ci.bit_offset + r0, ci.bit_offset + r1);
        if (bit_off < 0) return fail(a, "%s", duckdb_mb_gpu_last_error());
        d_validity = ib.validity;
      }
      if (stage_contiguous(c, c.s_in, ib.offsets, ci.offsets + (size_t)r0 * (size_t)ow, (size_t)(n + 1) * (size_t)ow, -1, &a->bytes_h2d))
        return fail(a, "%s", duckdb_mb_gpu_last_error());
      lo.h_cword[0] = 0;
      for (int64_t k = 0; k < nch; ++k) lo.h_cword[k + 1] = lo.h_cword[k] + (bnd[k + 1] - bnd[k] + 63) / 64;
      lo.words = lo.h_cword[nch];
      if (check_cuda(cudaMemcpyAsync(lo.d_cword, lo.h_cword, sizeof(int64_t) * (size_t)(nch + 1), cudaMemcpyHostToDevice, c.s_in), "child_word H2D"))
        return fail(a, "%s", duckdb_mb_gpu_last_error());
      a->bytes_h2d += sizeof(int64_t) * (uint64_t)(nch + 1);
      const int64_t child_slots = cc.is_string ? ((ne + DMB_VECTOR_SIZE - 1) / DMB_VECTOR_SIZE) * DMB_VECTOR_SIZE : ne;  // rev_string_kernel fills whole vectors
      lo.child_bytes = ne * cc.w_out;
      if (!grow(sc, lo.d_child, lo.child_cap, (size_t)child_slots * (size_t)cc.w_out + 64) ||
          !grow(sc, lo.h_child, lo.h_child_cap, (size_t)lo.child_bytes + 64, true) ||
          !grow(sc, lo.d_words, lo.words_cap, (size_t)lo.words * 8 + 64) || !grow(sc, lo.h_words, lo.h_words_cap, (size_t)lo.words * 8 + 64, true))
        return fail(a, "%s", duckdb_mb_gpu_last_error());
      dmb_rev_list_job lj;
      memset(&lj, 0, sizeof(lj));
      if (ne > 0) {
        dmb_rev_fixed_job *fj = &hj[nc + nchild_fixed];
        dmb_rev_string_job sj;
        const uint8_t *d_cvalidity = nullptr;
        int64_t cbit_off = 0;
        // out_validity NULL: the child masks are the list kernel's, per chunk
        if (!stage_rows(a, sc, cc, childbuf[(size_t)si * (size_t)nc + (size_t)j], j, e0, e1, lo.d_child, nullptr, fj, &sj, &d_cvalidity, &cbit_off)) return 0;
        if (cc.is_string) { strs.push_back(sj); str_rows.push_back(ne); }
        else { ++nchild_fixed; child_rows.push_back(ne); }
        lj.in_child_validity = d_cvalidity;
        lj.child_bit_offset = cbit_off;
      }
      lj.in_offsets = ib.offsets;
      lj.in_validity = d_validity;
      lj.in_bit_offset = bit_off;
      lj.child_word = lo.d_cword;
      lj.out_entries = slot.d_out[(size_t)j];
      lj.out_validity = slot.d_val[(size_t)j];
      lj.out_child_validity = (uint64_t *)lo.d_words;
      lj.error = slot.d_err + j;
      lj.large_offsets = ci.large ? 1 : 0;
      lists.push_back(lj);
    }
    cudaEventRecord(ev_in, c.s_in);
    if (check_cuda(cudaStreamWaitEvent(c.s_compute, ev_in, 0), "wait copy-in")) return fail(a, "%s", duckdb_mb_gpu_last_error());
    cudaEventRecord(k0, c.s_compute);
    for (int j : masks_from_bytes) {
      InBuf &ib = inbuf[(size_t)si * (size_t)nc + (size_t)j];
      if (dmb_dev_valid_bytes_to_masks(ib.validity, (uint64_t *)ib.masks, nullptr, n, c.s_compute)) return fail(a, "%s", duckdb_mb_gpu_last_error());
    }
    if (nfixed || nchild_fixed) {
      const size_t njobs = nchild_fixed ? (size_t)nc + (size_t)nchild_fixed : (size_t)nfixed;
      if (check_cuda(cudaMemcpyAsync(dj, hj, sizeof(dmb_rev_fixed_job) * njobs, cudaMemcpyHostToDevice, c.s_compute), "job H2D")) return fail(a, "%s", duckdb_mb_gpu_last_error());
      if (nfixed && dmb_dev_rev_fixed_batch(dj, hj, nfixed, n, c.s_compute)) return fail(a, "%s", duckdb_mb_gpu_last_error());
      for (int i = 0; i < nchild_fixed; ++i)  // one launch per child: the launch takes one row count for all its jobs
        if (dmb_dev_rev_fixed_batch(dj + nc + i, hj + nc + i, 1, child_rows[(size_t)i], c.s_compute)) return fail(a, "%s", duckdb_mb_gpu_last_error());
    }
    for (size_t i = 0; i < strs.size(); ++i)
      if (dmb_dev_rev_string_batch(&strs[i], str_rows[i], c.s_compute)) return fail(a, "%s", duckdb_mb_gpu_last_error());
    if (!lists.empty() && check_cuda(cudaMemsetAsync(slot.d_err, 0, sizeof(unsigned int) * (size_t)nc, c.s_compute), "error flags reset"))
      return fail(a, "%s", duckdb_mb_gpu_last_error());
    for (auto &lj : lists)
      if (dmb_dev_rev_list_batch(&lj, n, c.s_compute)) return fail(a, "%s", duckdb_mb_gpu_last_error());
    cudaEventRecord(k1, c.s_compute);
    sc.kernel_spans.emplace_back(k0, k1);
    cudaEventRecord(ev_k, c.s_compute);
    if (check_cuda(cudaStreamWaitEvent(c.s_out, ev_k, 0), "wait kernels")) return fail(a, "%s", duckdb_mb_gpu_last_error());
    for (int j = 0; j < nc; ++j) {
      const size_t ob = (size_t)n * (size_t)cols[(size_t)j].w_out, vb = (size_t)nch * DMB_VALIDITY_WORDS * 8;
      if (check_cuda(cudaMemcpyAsync(slot.h_out[(size_t)j], slot.d_out[(size_t)j], ob, cudaMemcpyDeviceToHost, c.s_out), "vectors D2H") ||
          check_cuda(cudaMemcpyAsync(slot.h_val[(size_t)j], slot.d_val[(size_t)j], vb, cudaMemcpyDeviceToHost, c.s_out), "validity D2H"))
        return fail(a, "%s", duckdb_mb_gpu_last_error());
      a->bytes_d2h += ob + vb;
      if (!cols[(size_t)j].is_list) continue;
      const ListOut &lo = slot.lists[(size_t)j];
      if ((lo.child_bytes && check_cuda(cudaMemcpyAsync(lo.h_child, lo.d_child, (size_t)lo.child_bytes, cudaMemcpyDeviceToHost, c.s_out), "child D2H")) ||
          (lo.words && check_cuda(cudaMemcpyAsync(lo.h_words, lo.d_words, (size_t)lo.words * 8, cudaMemcpyDeviceToHost, c.s_out), "child validity D2H")))
        return fail(a, "%s", duckdb_mb_gpu_last_error());
      a->bytes_d2h += (uint64_t)lo.child_bytes + (uint64_t)lo.words * 8;
    }
    if (!lists.empty() && check_cuda(cudaMemcpyAsync(slot.h_err, slot.d_err, sizeof(unsigned int) * (size_t)nc, cudaMemcpyDeviceToHost, c.s_out), "error flags D2H"))
      return fail(a, "%s", duckdb_mb_gpu_last_error());
    cudaEventRecord(slot.ev_out, c.s_out);
    slot.r0 = r0;
    slot.r1 = r1;
    slot.busy = true;
  }
  cudaEventRecord(in1, c.s_in);
  const size_t nsub = cuts.size() - 1;
  for (int k = 0; k < nslots; ++k) {  // oldest first
    Slot &slot = slots[(int)((nsub + (size_t)k) % (size_t)nslots)];
    if (!sink_slot(a, slot, cols, bounds)) return 0;
  }
  cudaEventRecord(out1, c.s_out);
  if (check_cuda(cudaStreamSynchronize(c.s_out), "appender sync") || check_cuda(cudaStreamSynchronize(c.s_in), "appender sync"))
    return fail(a, "%s", duckdb_mb_gpu_last_error());
  float f = 0;
  a->t[0] = cudaEventElapsedTime(&f, in0, in1) == cudaSuccess ? f : 0;
  a->t[1] = sc.kernel_ms();
  a->t[2] = cudaEventElapsedTime(&f, out0, out1) == cudaSuccess ? f : 0;
  a->t[3] = now_ms() - t0;
  return 1;
}

// rows buffered by the row API -> chunks
int32_t flush_rows(App *a) {
  if (a->buffered_rows == 0) return 1;
  std::vector<ColInput> cols((size_t)a->ncols);
  for (int j = 0; j < a->ncols; ++j) {
    RowBuf &rb = a->rows[(size_t)j];
    ColInput &ci = cols[(size_t)j];
    ci.valid_bytes = rb.valid.data();
    if (rb.width == 0) {
      ci.is_string = true;
      ci.w_out = 16;
      ci.offsets = (const uint8_t *)rb.offsets.data();
      if (rb.data.empty()) rb.data.push_back(0);
      ci.data = rb.data.data();
    } else {
      ci.rev_op = copy_op(rb.width);
      ci.w_in = ci.w_out = rb.width;
      ci.values = rb.values.data();
      if (a->type_ids[(size_t)j] == DMB_TYPE_DECIMAL) {  // int128 -> the physical width DuckDB uses for the precision
        if (rb.dec_prec <= 0) {
          fail(a, "flush: DECIMAL column %d has no declared precision (duckdb_mb_gpu_appender_set_decimal)", j);
          return 0;
        }
        if (rb.dec_prec <= 4) { ci.rev_op = DMB_REV_I128_TO_I16; ci.w_out = 2; }
        else if (rb.dec_prec <= 9) { ci.rev_op = DMB_REV_I128_TO_I32; ci.w_out = 4; }
        else if (rb.dec_prec <= 18) { ci.rev_op = DMB_REV_I128_TO_I64; ci.w_out = 8; }
      }
    }
  }
  const int32_t ok = convert_rows(a, cols, a->buffered_rows);
  for (RowBuf &rb : a->rows) {
    rb.values.clear();
    rb.valid.clear();
    rb.data.clear();
    rb.offsets.assign(1, 0);
  }
  a->buffered_rows = 0;
  return ok;
}

RowBuf *cell(App *a, const char *cmd) {
  if (a->state != kRowInProgress) { illegal(a, cmd); return nullptr; }
  if (a->cur_col >= a->ncols) {  // over-filled row (src/duckdb_appender_state_machine.mbt:96-111)
    fail(a, "%s: row already has %d values", cmd, a->ncols);
    a->state = kError;
    return nullptr;
  }
  return &a->rows[(size_t)a->cur_col];
}

template <typename T>
void push_value(RowBuf *rb, T v) {
  const size_t at = rb->values.size();
  rb->values.resize(at + sizeof(T));
  memcpy(rb->values.data() + at, &v, sizeof(T));
}

int32_t type_mismatch(App *a, const char *cmd) {
  fail(a, "%s: column %d has DuckDB type %d", cmd, a->cur_col, a->type_ids[(size_t)a->cur_col]);
  a->state = kError;
  return 0;
}

// numeric cell into a numeric column, C conversion like DuckDB's implicit appender cast
int32_t push_number(App *a, const char *cmd, int64_t iv, double dv, bool is_double) {
  RowBuf *rb = cell(a, cmd);
  if (!rb) return 0;
  const int32_t t = a->type_ids[(size_t)a->cur_col];
  const int64_t as_int = is_double ? (int64_t)nearbyint(dv) : iv;
  const double as_dbl = is_double ? dv : (double)iv;
  switch (t) {
    case DMB_TYPE_TINYINT: case DMB_TYPE_UTINYINT: push_value<int8_t>(rb, (int8_t)as_int); break;
    case DMB_TYPE_SMALLINT: case DMB_TYPE_USMALLINT: push_value<int16_t>(rb, (int16_t)as_int); break;
    case DMB_TYPE_INTEGER: case DMB_TYPE_UINTEGER: case DMB_TYPE_DATE: push_value<int32_t>(rb, (int32_t)as_int); break;
    case DMB_TYPE_BIGINT: case DMB_TYPE_UBIGINT: case DMB_TYPE_TIMESTAMP: case DMB_TYPE_TIMESTAMP_S: case DMB_TYPE_TIMESTAMP_MS:
    case DMB_TYPE_TIMESTAMP_NS: case DMB_TYPE_TIMESTAMP_TZ: case DMB_TYPE_TIME: case DMB_TYPE_TIME_NS:
      push_value<int64_t>(rb, as_int); break;
    case DMB_TYPE_FLOAT: push_value<float>(rb, (float)as_dbl); break;
    case DMB_TYPE_DOUBLE: push_value<double>(rb, as_dbl); break;
    default: return type_mismatch(a, cmd);
  }
  rb->valid.push_back(1);
  a->cur_col++;
  return 1;
}

// the buffers of one Arrow array (already mapped by map_format) at element `off`
void bind_buffers(ColInput &ci, const ArrowArray *arr, int64_t off) {
  static const uint8_t kNoData[16] = {0};
  ci.bit_offset = off;
  ci.validity = (arr->null_count != 0 && arr->n_buffers > 0) ? (const uint8_t *)arr->buffers[0] : nullptr;
  if (ci.is_string || ci.is_list) {
    ci.offsets = arr->n_buffers > 1 && arr->buffers[1] ? (const uint8_t *)arr->buffers[1] + (size_t)off * (ci.large ? 8 : 4) : nullptr;
    if (ci.is_string) ci.data = arr->n_buffers > 2 && arr->buffers[2] ? (const uint8_t *)arr->buffers[2] : kNoData;
  } else if (ci.is_bits) {
    ci.values = arr->n_buffers > 1 ? (const uint8_t *)arr->buffers[1] : nullptr;
  } else {
    ci.values = arr->n_buffers > 1 && arr->buffers[1] ? (const uint8_t *)arr->buffers[1] + (size_t)off * (size_t)ci.w_in : nullptr;
  }
}

const char *nested_name(const char *fmt) {
  if (strcmp(fmt, "+l") == 0 || strcmp(fmt, "+L") == 0) return "LIST";
  if (strcmp(fmt, "+s") == 0) return "STRUCT";
  if (strcmp(fmt, "+m") == 0) return "MAP";
  if (strcmp(fmt, "+vl") == 0 || strcmp(fmt, "+vL") == 0) return "list view";
  if (strncmp(fmt, "+w:", 3) == 0) return "fixed_size_list";
  return "nested type";
}

// Arrow list / large_list -> a LIST column whose child type the table declared (duckdb_mb_gpu_appender_set_list)
bool map_list(App *a, int j, const ArrowArray *arr, const ArrowSchema *sch, ColInput *ci, ColInput *child) {
  const char *fmt = sch->format;
  if (strcmp(fmt, "+l") != 0 && strcmp(fmt, "+L") != 0) {
    if (fmt[0] == '+') fail(a, "column %d: an Arrow %s ('%s') cannot be appended to a LIST column", j, nested_name(fmt), fmt);
    else fail(a, "column %d: Arrow format '%s' cannot be appended to a LIST column", j, fmt);
    return false;
  }
  const ListDecl &d = a->lists[(size_t)j];
  if (!d.type_id) {
    fail(a, "column %d: the LIST column's child type is not declared (duckdb_mb_gpu_appender_set_list)", j);
    return false;
  }
  if (arr->n_children != 1 || sch->n_children != 1 || !arr->children[0] || !sch->children[0] || !sch->children[0]->format) {
    fail(a, "column %d: an Arrow list needs exactly one child array", j);
    return false;
  }
  const ArrowArray *carr = arr->children[0];
  const char *cfmt = sch->children[0]->format;
  if (cfmt[0] == '+') {
    fail(a, "column %d: LIST<%s> cannot be appended (Arrow child format '%s')", j, nested_name(cfmt), cfmt);
    return false;
  }
  int32_t dec_w = d.dec_width, dec_s = d.dec_scale;  // a DECIMAL child: set_list declared it
  if (!map_format(a, j, "list child format", cfmt, d.type_id, &dec_w, &dec_s, child)) {
    const bool decimal_child = d.type_id == DMB_TYPE_DECIMAL || d.type_id == DMB_TYPE_HUGEINT;
    if (!decimal_child || strncmp(cfmt, "d:", 2) != 0)  // map_decimal's refusal names its own reason
      fail(a, "column %d: Arrow list child format '%s' does not match the declared child type %d", j, cfmt, d.type_id);
    return false;
  }
  bind_buffers(*child, carr, carr->offset);
  child->child_len = carr->length;
  ci->is_list = true;
  ci->large = fmt[1] == 'L';
  ci->w_out = 16;  // duckdb_list_entry
  ci->child = child;
  ci->child_len = carr->length;
  if (carr->length > 0 && ((child->is_string && !child->offsets) || (!child->is_string && !child->values))) {
    fail(a, "column %d: the Arrow list child has no value buffer", j);
    return false;
  }
  return true;
}

}  // namespace
}  // namespace dmb

extern "C" duckdb_mb_gpu_appender *duckdb_mb_gpu_appender_create(duckdb_mb_gpu_ctx *ctx, int32_t ncols, const int32_t *type_ids,
                                                                 dmb_chunk_sink sink, void *user) {
  if (!ctx || !ctx->core) { set_error("duckdb_mb_gpu_appender_create: null context"); return nullptr; }
  if (ncols <= 0 || !type_ids) { set_error("duckdb_mb_gpu_appender_create: no columns"); return nullptr; }
  App *a = new App();
  a->core = ctx->core;
  a->ncols = ncols;
  a->type_ids.assign(type_ids, type_ids + ncols);
  a->sink = sink;
  a->user = user;
  a->rows.resize((size_t)ncols);
  a->lists.resize((size_t)ncols);
  for (int j = 0; j < ncols; ++j) {
    a->rows[(size_t)j].width = row_width(type_ids[j]);  // -1: column only reachable through Arrow batches
    a->rows[(size_t)j].offsets.assign(1, 0);
  }
  const char *env = getenv("DMB_REV_BATCH_ROWS");
  if (env && atoll(env) >= DMB_VECTOR_SIZE) a->sub_rows = (atoll(env) / DMB_VECTOR_SIZE) * DMB_VECTOR_SIZE;
  const char *cap = getenv("DMB_REV_LIST_CHILD_CAP");
  a->list_child_cap = cap && atoll(cap) > 0 ? atoll(cap) : kListChildCap;
  a->state = kReady;  // Create: NotCreated -> Ready
  return a;
}

extern "C" void duckdb_mb_gpu_appender_destroy(duckdb_mb_gpu_appender *a) {
  if (!a) return;
  if (a->on_destroy) a->on_destroy(a->user);
  delete a;
}

extern "C" void duckdb_mb_gpu_appender_set_hooks(duckdb_mb_gpu_appender *a, dmb_appender_flush_hook on_flush, dmb_appender_destroy_hook on_destroy) {
  if (!a) return;
  a->on_flush = on_flush;
  a->on_destroy = on_destroy;
}

extern "C" moonbit_bytes_t duckdb_mb_gpu_appender_error(duckdb_mb_gpu_appender *a) {
  const char *msg = a ? a->error : "";
  const size_t n = strlen(msg);
  moonbit_bytes_t b = moonbit_make_bytes_raw((int32_t)n);
  if (b) memcpy(b, msg, n);
  return b;
}

extern "C" int32_t duckdb_mb_gpu_appender_state(duckdb_mb_gpu_appender *a) { return a ? a->state : kNotCreated; }
extern "C" int64_t duckdb_mb_gpu_appender_row_count(duckdb_mb_gpu_appender *a) { return a ? a->row_count : 0; }
extern "C" int64_t duckdb_mb_gpu_appender_flushed_row_count(duckdb_mb_gpu_appender *a) { return a ? a->flushed_row_count : 0; }

extern "C" int32_t duckdb_mb_gpu_append_arrow_batch(duckdb_mb_gpu_appender *a, const struct ArrowArray *batch,
                                                    const struct ArrowSchema *schema) {
  NvtxRange nvtx("dmb::append_arrow_batch");
  if (!a) { set_error("null appender"); return 0; }
  if (a->state != kReady && a->state != kFlushed) return illegal(a, "append_arrow_batch");  // legal where BeginRow is
  if (!batch || !schema || !schema->format || strcmp(schema->format, "+s") != 0) {
    fail(a, "append_arrow_batch: expected a struct array (record batch)");
    a->state = kError;
    return 0;
  }
  if (batch->n_children != a->ncols || schema->n_children != a->ncols) {
    fail(a, "append_arrow_batch: batch has %lld columns, table has %d", (long long)batch->n_children, a->ncols);
    a->state = kError;
    return 0;
  }
  if (batch->null_count > 0) {
    fail(a, "append_arrow_batch: null struct rows are not supported");
    a->state = kError;
    return 0;
  }
  const int64_t n = batch->length;
  std::vector<ColInput> cols((size_t)a->ncols), children((size_t)a->ncols);
  for (int j = 0; j < a->ncols; ++j) {
    const ArrowArray *ch = batch->children[j];
    const ArrowSchema *cs = schema->children[j];
    ColInput &ci = cols[(size_t)j];
    const bool list = a->type_ids[(size_t)j] == DMB_TYPE_LIST;
    if (!ch || !cs || !cs->format ||
        !(list ? map_list(a, j, ch, cs, &ci, &children[(size_t)j])
               : map_format(a, j, "format", cs->format, a->type_ids[(size_t)j], &a->rows[(size_t)j].dec_prec, &a->rows[(size_t)j].dec_scale, &ci))) {
      if (!a->error[0]) fail(a, "append_arrow_batch: column %d is malformed", j);
      a->state = kError;
      return 0;
    }
    if (ch->length < batch->offset + n) {
      fail(a, "append_arrow_batch: column %d is shorter than the batch", j);
      a->state = kError;
      return 0;
    }
    bind_buffers(ci, ch, ch->offset + batch->offset);
    if (n > 0 && (((ci.is_string || ci.is_list) && !ci.offsets) || (!ci.is_string && !ci.is_list && !ci.values))) {
      fail(a, "append_arrow_batch: column %d has no value buffer", j);
      a->state = kError;
      return 0;
    }
  }
  if (!flush_rows(a)) { a->state = kError; return 0; }  // keep row order with earlier row-API appends
  if (!convert_rows(a, cols, n)) { a->state = kError; return 0; }
  a->row_count += n;
  a->state = kReady;
  return 1;
}

// ---- row-at-a-time protocol of the reference (src/duckdb_native.c:1100-1235), column-buffered
extern "C" int32_t duckdb_mb_gpu_begin_row(duckdb_mb_gpu_appender *a) {
  if (!a) return 0;
  if (a->state != kReady && a->state != kFlushed) return illegal(a, "begin_row");
  for (int j = 0; j < a->ncols; ++j)
    if (a->rows[(size_t)j].width < 0) { fail(a, "begin_row: column %d (type %d) is only appendable through Arrow batches", j, a->type_ids[(size_t)j]); a->state = kError; return 0; }
  a->state = kRowInProgress;
  a->cur_col = 0;
  return 1;
}

extern "C" int32_t duckdb_mb_gpu_append_int(duckdb_mb_gpu_appender *a, int32_t v) { return a ? push_number(a, "append_int", v, 0, false) : 0; }
extern "C" int32_t duckdb_mb_gpu_append_bigint(duckdb_mb_gpu_appender *a, int64_t v) { return a ? push_number(a, "append_bigint", v, 0, false) : 0; }
extern "C" int32_t duckdb_mb_gpu_append_double(duckdb_mb_gpu_appender *a, double v) { return a ? push_number(a, "append_double", 0, v, true) : 0; }
extern "C" int32_t duckdb_mb_gpu_append_date(duckdb_mb_gpu_appender *a, int32_t days) { return a ? push_number(a, "append_date", days, 0, false) : 0; }
extern "C" int32_t duckdb_mb_gpu_append_timestamp(duckdb_mb_gpu_appender *a, int64_t micros) { return a ? push_number(a, "append_timestamp", micros, 0, false) : 0; }

// BLOB cell (src/duckdb_native.c:1397-1415): the bytes as they are, no UTF-8 requirement
extern "C" int32_t duckdb_mb_gpu_append_blob(duckdb_mb_gpu_appender *a, const uint8_t *bytes, int32_t len) {
  return duckdb_mb_gpu_append_varchar(a, bytes, len);
}

// LIST / STRUCT / MAP cells of the reference's row protocol: the reference serialises them as text and appends that as
// a VARCHAR cell (src/duckdb_native.c:1735-1790 `["a", "b"]`, :1792-1858 and :1860-1926 `{"k": "v", ...}`; no escaping).
// The text reaches libduckdb through duckdb_append_varchar, a C string: it ends at the first NUL byte of any item.
namespace {
void put_quoted(std::vector<uint8_t> &t, const uint8_t *p, int32_t len) {
  t.push_back('"');
  if (p && len > 0) t.insert(t.end(), p, p + len);
  t.push_back('"');
}
int32_t append_text_cell(duckdb_mb_gpu_appender *a, std::vector<uint8_t> &t) {
  size_t n = 0;
  while (n < t.size() && t[n] != 0) ++n;  // strlen of the reference's buffer
  return duckdb_mb_gpu_append_varchar(a, t.data(), (int32_t)n);
}
}  // namespace

extern "C" int32_t duckdb_mb_gpu_append_list_varchar(duckdb_mb_gpu_appender *a, const uint8_t *const *values, const int32_t *lens, int32_t count) {
  if (!a) return 0;
  if (count < 0 || (count > 0 && (!values || !lens))) { fail(a, "append_list_varchar: bad arguments"); a->state = kError; return 0; }
  std::vector<uint8_t> t;
  t.push_back('[');
  for (int32_t i = 0; i < count; ++i) {
    if (i > 0) { t.push_back(','); t.push_back(' '); }
    put_quoted(t, values[i], lens[i]);
  }
  t.push_back(']');
  return append_text_cell(a, t);
}

static int32_t append_pairs(duckdb_mb_gpu_appender *a, const char *what, const uint8_t *const *keys, const int32_t *key_lens,
                            const uint8_t *const *values, const int32_t *value_lens, int32_t count) {
  if (!a) return 0;
  if (count < 0 || (count > 0 && (!keys || !key_lens || !values || !value_lens))) { fail(a, "%s: bad arguments", what); a->state = kError; return 0; }
  std::vector<uint8_t> t;
  t.push_back('{');
  for (int32_t i = 0; i < count; ++i) {
    if (i > 0) { t.push_back(','); t.push_back(' '); }
    put_quoted(t, keys[i], key_lens[i]);
    t.push_back(':');
    t.push_back(' ');
    put_quoted(t, values[i], value_lens[i]);
  }
  t.push_back('}');
  return append_text_cell(a, t);
}

extern "C" int32_t duckdb_mb_gpu_append_struct_varchar(duckdb_mb_gpu_appender *a, const uint8_t *const *names, const int32_t *name_lens,
                                                      const uint8_t *const *values, const int32_t *value_lens, int32_t count) {
  return append_pairs(a, "append_struct_varchar", names, name_lens, values, value_lens, count);
}

extern "C" int32_t duckdb_mb_gpu_append_map_varchar_varchar(duckdb_mb_gpu_appender *a, const uint8_t *const *keys, const int32_t *key_lens,
                                                           const uint8_t *const *values, const int32_t *value_lens, int32_t count) {
  return append_pairs(a, "append_map_varchar_varchar", keys, key_lens, values, value_lens, count);
}

// INTERVAL cell (src/duckdb_native.c:1511-1533): duckdb_interval {months, days, micros}
extern "C" int32_t duckdb_mb_gpu_append_interval(duckdb_mb_gpu_appender *a, int32_t months, int32_t days, int64_t micros) {
  if (!a) return 0;
  RowBuf *rb = cell(a, "append_interval");
  if (!rb) return 0;
  if (a->type_ids[(size_t)a->cur_col] != DMB_TYPE_INTERVAL) return type_mismatch(a, "append_interval");
  interval_t v{months, days, micros};
  const uint8_t *p = reinterpret_cast<const uint8_t *>(&v);
  rb->values.insert(rb->values.end(), p, p + sizeof(v));
  rb->valid.push_back(1);
  a->cur_col++;
  return 1;
}

// the table column's DECIMAL(width, scale) (duckdb_appender_column_type -> duckdb_decimal_width / _scale)
extern "C" int32_t duckdb_mb_gpu_appender_set_decimal(duckdb_mb_gpu_appender *a, int32_t col, int32_t width, int32_t scale) {
  if (!a) return 0;
  if (col < 0 || col >= a->ncols || a->type_ids[(size_t)col] != DMB_TYPE_DECIMAL || width < 1 || width > 38 || scale < 0 || scale > width) {
    fail(a, "appender_set_decimal: column %d is not a DECIMAL column or DECIMAL(%d,%d) is not a type", col, width, scale);
    return 0;
  }
  RowBuf &rb = a->rows[(size_t)col];
  if (rb.dec_prec && (rb.dec_prec != width || rb.dec_scale != scale)) {
    fail(a, "appender_set_decimal: column %d is already DECIMAL(%d,%d)", col, rb.dec_prec, rb.dec_scale);
    return 0;
  }
  rb.dec_prec = width;
  rb.dec_scale = scale;
  return 1;
}

// the table column's LIST child type (duckdb_list_type_child_type(duckdb_appender_column_type(..)))
extern "C" int32_t duckdb_mb_gpu_appender_set_list(duckdb_mb_gpu_appender *a, int32_t col, int32_t child_type_id, int32_t child_dec_width,
                                                   int32_t child_dec_scale) {
  if (!a) return 0;
  if (col < 0 || col >= a->ncols || a->type_ids[(size_t)col] != DMB_TYPE_LIST) return fail(a, "appender_set_list: column %d is not a LIST column", col);
  switch (child_type_id) {
    case DMB_TYPE_LIST: return fail(a, "appender_set_list: column %d: LIST<LIST> cannot be appended", col);
    case DMB_TYPE_STRUCT: return fail(a, "appender_set_list: column %d: LIST<STRUCT> cannot be appended", col);
    case DMB_TYPE_MAP: return fail(a, "appender_set_list: column %d: LIST<MAP> cannot be appended", col);
    case DMB_TYPE_DECIMAL:
      if (child_dec_width < 1 || child_dec_width > 38 || child_dec_scale < 0 || child_dec_scale > child_dec_width)
        return fail(a, "appender_set_list: column %d: DECIMAL(%d,%d) is not a type", col, child_dec_width, child_dec_scale);
      break;
    case DMB_TYPE_BOOLEAN: case DMB_TYPE_TINYINT: case DMB_TYPE_SMALLINT: case DMB_TYPE_INTEGER: case DMB_TYPE_BIGINT:
    case DMB_TYPE_UTINYINT: case DMB_TYPE_USMALLINT: case DMB_TYPE_UINTEGER: case DMB_TYPE_UBIGINT: case DMB_TYPE_FLOAT:
    case DMB_TYPE_DOUBLE: case DMB_TYPE_DATE: case DMB_TYPE_TIME: case DMB_TYPE_TIME_NS: case DMB_TYPE_TIME_TZ:
    case DMB_TYPE_TIMESTAMP: case DMB_TYPE_TIMESTAMP_S: case DMB_TYPE_TIMESTAMP_MS: case DMB_TYPE_TIMESTAMP_NS:
    case DMB_TYPE_TIMESTAMP_TZ: case DMB_TYPE_HUGEINT: case DMB_TYPE_UHUGEINT: case DMB_TYPE_UUID: case DMB_TYPE_VARCHAR:
    case DMB_TYPE_BLOB:
      break;
    default:  // the child types map_format converts, and nothing else
      return fail(a, "appender_set_list: column %d: LIST child type %d cannot be appended", col, child_type_id);
  }
  if (child_type_id != DMB_TYPE_DECIMAL) child_dec_width = child_dec_scale = 0;
  ListDecl &d = a->lists[(size_t)col];
  if (d.type_id && (d.type_id != child_type_id || d.dec_width != child_dec_width || d.dec_scale != child_dec_scale))
    return fail(a, "appender_set_list: column %d already has LIST child type %d", col, d.type_id);
  d = ListDecl{child_type_id, child_dec_width, child_dec_scale};
  return 1;
}

// during a sink call: the child vector of LIST column `col` for the chunk being handed over
extern "C" int32_t duckdb_mb_gpu_appender_list_child(duckdb_mb_gpu_appender *a, int32_t col, const void **data, const uint64_t **validity,
                                                     uint64_t *size) {
  if (!a || !data || !validity || !size) return 0;
  if (a->sink_chunk < 0 || col < 0 || col >= a->ncols || (size_t)col >= a->sink_lists.size() || !a->sink_lists[(size_t)col].bounds)
    return fail(a, "appender_list_child: column %d is not a LIST column of a chunk being handed to the sink", col);
  const SinkList &l = a->sink_lists[(size_t)col];
  const int64_t k = a->sink_chunk;
  *data = l.values + (size_t)(l.bounds[k] - l.bounds[0]) * (size_t)l.w;
  *validity = l.words + l.cword[k];
  *size = (uint64_t)(l.bounds[k + 1] - l.bounds[k]);
  return 1;
}

// DECIMAL cell from hugeint parts (src/duckdb_native.c:1447-1481: duckdb_create_decimal + duckdb_append_value).
// The value is brought to the column's scale like DuckDB's decimal -> decimal cast (exact when the scale grows,
// round half away from zero when it shrinks) and must fit the column's precision.
extern "C" int32_t duckdb_mb_gpu_append_decimal(duckdb_mb_gpu_appender *a, int32_t width, int32_t scale, int64_t lower, int64_t upper) {
  if (!a) return 0;
  RowBuf *rb = cell(a, "append_decimal");
  if (!rb) return 0;
  if (a->type_ids[(size_t)a->cur_col] != DMB_TYPE_DECIMAL) return type_mismatch(a, "append_decimal");
  if (width < 1 || width > 38 || scale < 0 || scale > width) { fail(a, "append_decimal: DECIMAL(%d,%d) is not a type", width, scale); a->state = kError; return 0; }
  if (rb->dec_prec == 0) { rb->dec_prec = width; rb->dec_scale = scale; }  // first value declares the column
  __int128 v = (__int128)(((unsigned __int128)(uint64_t)upper << 64) | (unsigned __int128)(uint64_t)lower);
  auto pow10 = [](int e) { __int128 p = 1; while (e-- > 0) p *= 10; return p; };
  if (scale < rb->dec_scale) {
    const int up = rb->dec_scale - scale;
    const __int128 lim = pow10(38 - up);
    if (v >= lim || v <= -lim) { fail(a, "append_decimal: value out of range for DECIMAL(%d,%d)", rb->dec_prec, rb->dec_scale); a->state = kError; return 0; }
    v *= pow10(up);
  } else if (scale > rb->dec_scale) {
    const __int128 d = pow10(scale - rb->dec_scale), half = d / 2;
    v = v >= 0 ? (v + half) / d : -((-v + half) / d);
  }
  const __int128 bound = pow10(rb->dec_prec);
  if (v >= bound || v <= -bound) { fail(a, "append_decimal: value out of range for DECIMAL(%d,%d)", rb->dec_prec, rb->dec_scale); a->state = kError; return 0; }
  const uint8_t *p = reinterpret_cast<const uint8_t *>(&v);
  rb->values.insert(rb->values.end(), p, p + 16);
  rb->valid.push_back(1);
  a->cur_col++;
  return 1;
}

extern "C" int32_t duckdb_mb_gpu_append_bool(duckdb_mb_gpu_appender *a, int32_t v) {
  if (!a) return 0;
  RowBuf *rb = cell(a, "append_bool");
  if (!rb) return 0;
  if (a->type_ids[(size_t)a->cur_col] != DMB_TYPE_BOOLEAN) return type_mismatch(a, "append_bool");
  rb->values.push_back(v ? 1 : 0);
  rb->valid.push_back(1);
  a->cur_col++;
  return 1;
}

extern "C" int32_t duckdb_mb_gpu_append_varchar(duckdb_mb_gpu_appender *a, const uint8_t *bytes, int32_t len) {
  if (!a) return 0;
  RowBuf *rb = cell(a, "append_varchar");
  if (!rb) return 0;
  if (rb->width != 0) return type_mismatch(a, "append_varchar");
  if (len < 0 || (len > 0 && !bytes)) { fail(a, "append_varchar: bad buffer"); a->state = kError; return 0; }
  if ((int64_t)rb->data.size() + len > 0x7fffffffll) { fail(a, "append_varchar: more than 2 GiB of buffered string data; flush first"); a->state = kError; return 0; }
  rb->data.insert(rb->data.end(), bytes, bytes + len);
  rb->offsets.push_back((int32_t)rb->data.size());
  rb->valid.push_back(1);
  a->cur_col++;
  return 1;
}

extern "C" int32_t duckdb_mb_gpu_append_null(duckdb_mb_gpu_appender *a) {
  if (!a) return 0;
  RowBuf *rb = cell(a, "append_null");
  if (!rb) return 0;
  if (rb->width == 0) rb->offsets.push_back((int32_t)rb->data.size());
  else rb->values.resize(rb->values.size() + (size_t)rb->width, 0);
  rb->valid.push_back(0);
  a->cur_col++;
  return 1;
}

extern "C" int32_t duckdb_mb_gpu_end_row(duckdb_mb_gpu_appender *a) {
  if (!a) return 0;
  if (a->state != kRowInProgress) return illegal(a, "end_row");
  if (a->cur_col != a->ncols) {  // under-filled row (src/duckdb_appender_state_machine.mbt:160-177)
    fail(a, "end_row: row has %d of %d values", a->cur_col, a->ncols);
    a->state = kError;
    return 0;
  }
  a->state = kReady;
  a->row_count++;
  a->buffered_rows++;
  if (a->buffered_rows >= (1 << 20) && !flush_rows(a)) { a->state = kError; return 0; }
  return 1;
}

extern "C" int32_t duckdb_mb_gpu_appender_flush(duckdb_mb_gpu_appender *a) {
  if (!a) { set_error("null appender"); return 0; }
  if (a->state != kReady && a->state != kFlushed) return illegal(a, "flush");
  if (!flush_rows(a)) { a->state = kError; return 0; }
  if (a->on_flush && !a->on_flush(a->user)) { fail(a, "flush: the sink's flush hook failed"); a->state = kError; return 0; }
  a->flushed_row_count = a->row_count;
  a->state = kFlushed;
  return 1;
}

extern "C" int32_t duckdb_mb_gpu_appender_close(duckdb_mb_gpu_appender *a) {
  if (!a) { set_error("null appender"); return 0; }
  if (a->state == kClosed) return 1;  // Closed is terminal: the command is a no-op
  int32_t ok = 1;
  // complete buffered rows still reach the table, like duckdb_appender_destroy's implicit flush;
  // a row in progress is dropped
  if (a->state == kReady || a->state == kFlushed) ok = flush_rows(a);
  a->state = kClosed;
  return ok;
}

extern "C" int32_t duckdb_mb_gpu_appender_timings(duckdb_mb_gpu_appender *a, double *out4) {
  if (!a || !out4) return 0;
  for (int i = 0; i < 4; ++i) out4[i] = a->t[i];
  return 1;
}

extern "C" int32_t duckdb_mb_gpu_appender_link_bytes(duckdb_mb_gpu_appender *a, uint64_t *out2) {
  if (!a || !out2) return 0;
  out2[0] = a->bytes_h2d;
  out2[1] = a->bytes_d2h;
  return 1;
}

// =====================================================================================  L2 drop-in: the appender set
// The reference's own symbols (src/duckdb_native.c:1083-1251, 1313-1533, 1735-1926; MoonBit externs
// src/duckdb_native.mbt:44-110,134-144,165-217,266-288) with the reference's signatures: `duckdb_mb_appender` is this
// library's appender handle, Bytes arrive as moonbit_bytes_t (length from the object header, Moonbit_array_length),
// Array[Bytes] as moonbit_bytes_t*.  All parameters are #borrow: nothing is decref'd.  duckdb_mb_appender_create itself
// needs libduckdb (duckdb_appender_create) and lives in glue/duckdb_gpu_glue.c.
extern "C" void duckdb_mb_appender_destroy(duckdb_mb_appender *a) {  // :1083-1091
  if (!a) return;
  duckdb_mb_gpu_appender_close(a);  // complete rows still reach the table, like duckdb_appender_destroy's implicit flush
  duckdb_mb_gpu_appender_destroy(a);
}
extern "C" moonbit_bytes_t duckdb_mb_appender_error(duckdb_mb_appender *a) { return duckdb_mb_gpu_appender_error(a); }  // :1093-1098
extern "C" int32_t duckdb_mb_is_null_appender(duckdb_mb_appender *a) { return a == nullptr ? 1 : 0; }                    // :1253-1255
extern "C" int32_t duckdb_mb_begin_row(duckdb_mb_appender *a) { return duckdb_mb_gpu_begin_row(a); }                     // :1100
extern "C" int32_t duckdb_mb_append_int(duckdb_mb_appender *a, int32_t v) { return duckdb_mb_gpu_append_int(a, v); }     // :1116
extern "C" int32_t duckdb_mb_append_bigint(duckdb_mb_appender *a, int64_t v) { return duckdb_mb_gpu_append_bigint(a, v); }  // :1132
extern "C" int32_t duckdb_mb_append_double(duckdb_mb_appender *a, double v) { return duckdb_mb_gpu_append_double(a, v); }   // :1148
extern "C" int32_t duckdb_mb_append_varchar(duckdb_mb_appender *a, moonbit_bytes_t value) {                              // :1164
  if (!a) return 0;
  if (!value) { fail(a, "append_varchar: null Bytes"); return 0; }
  return duckdb_mb_gpu_append_varchar(a, value, Moonbit_array_length(value));
}
extern "C" int32_t duckdb_mb_append_bool(duckdb_mb_appender *a, bool v) { return duckdb_mb_gpu_append_bool(a, v ? 1 : 0); }  // :1189
extern "C" int32_t duckdb_mb_append_null(duckdb_mb_appender *a) { return duckdb_mb_gpu_append_null(a); }                 // :1205
extern "C" int32_t duckdb_mb_end_row(duckdb_mb_appender *a) { return duckdb_mb_gpu_end_row(a); }                         // :1221
extern "C" int32_t duckdb_mb_flush(duckdb_mb_appender *a) { return a ? duckdb_mb_gpu_appender_flush(a) : 0; }            // :1237
// exact days / micros into the vectors: the reference's approximate-string path (:1299-1367) is a defect, not a contract
extern "C" int32_t duckdb_mb_append_date(duckdb_mb_appender *a, int32_t days) { return duckdb_mb_gpu_append_date(a, days); }            // :1313
extern "C" int32_t duckdb_mb_append_timestamp(duckdb_mb_appender *a, int64_t micros) { return duckdb_mb_gpu_append_timestamp(a, micros); }  // :1350
extern "C" int32_t duckdb_mb_append_blob(duckdb_mb_appender *a, moonbit_bytes_t data, int32_t length) {                  // :1397
  if (!a) return 0;
  if (!data || length < 0 || length > Moonbit_array_length(data)) { fail(a, "append_blob: bad length"); return 0; }
  return duckdb_mb_gpu_append_blob(a, data, length);
}
extern "C" int32_t duckdb_mb_append_decimal(duckdb_mb_appender *a, uint8_t width, uint8_t scale, int64_t lower, int64_t upper) {  // :1447
  return duckdb_mb_gpu_append_decimal(a, width, scale, lower, upper);
}
extern "C" int32_t duckdb_mb_append_interval(duckdb_mb_appender *a, int32_t months, int32_t days, int64_t micros) {      // :1511
  return duckdb_mb_gpu_append_interval(a, months, days, micros);
}

namespace {
// Array[Bytes] (moonbit_bytes_t *) -> pointer + length tables
bool bytes_array(duckdb_mb_gpu_appender *a, const char *cmd, moonbit_bytes_t *items, int32_t count, std::vector<const uint8_t *> *ptrs,
                 std::vector<int32_t> *lens) {
  if (count < 0 || (count > 0 && !items)) { fail(a, "%s: bad arguments", cmd); return false; }
  ptrs->resize((size_t)count);
  lens->resize((size_t)count);
  for (int32_t i = 0; i < count; ++i) {
    if (!items[i]) { fail(a, "%s: element %d is null", cmd, i); return false; }
    (*ptrs)[(size_t)i] = items[i];
    (*lens)[(size_t)i] = Moonbit_array_length(items[i]);
  }
  return true;
}
}  // namespace

extern "C" int32_t duckdb_mb_append_list_varchar(duckdb_mb_appender *a, moonbit_bytes_t *values, int32_t count) {        // :1735
  if (!a) return 0;
  std::vector<const uint8_t *> p;
  std::vector<int32_t> l;
  if (!bytes_array(a, "append_list_varchar", values, count, &p, &l)) return 0;
  return duckdb_mb_gpu_append_list_varchar(a, p.data(), l.data(), count);
}
extern "C" int32_t duckdb_mb_append_struct_varchar(duckdb_mb_appender *a, moonbit_bytes_t *field_names, moonbit_bytes_t *field_values,
                                                  int32_t field_count) {                                                 // :1792
  if (!a) return 0;
  std::vector<const uint8_t *> pn, pv;
  std::vector<int32_t> ln, lv;
  if (!bytes_array(a, "append_struct_varchar", field_names, field_count, &pn, &ln) ||
      !bytes_array(a, "append_struct_varchar", field_values, field_count, &pv, &lv)) return 0;
  return duckdb_mb_gpu_append_struct_varchar(a, pn.data(), ln.data(), pv.data(), lv.data(), field_count);
}
extern "C" int32_t duckdb_mb_append_map_varchar_varchar(duckdb_mb_appender *a, moonbit_bytes_t *keys, moonbit_bytes_t *values,
                                                       int32_t entry_count) {                                            // :1860
  if (!a) return 0;
  std::vector<const uint8_t *> pk, pv;
  std::vector<int32_t> lk, lv;
  if (!bytes_array(a, "append_map_varchar_varchar", keys, entry_count, &pk, &lk) ||
      !bytes_array(a, "append_map_varchar_varchar", values, entry_count, &pv, &lv)) return 0;
  return duckdb_mb_gpu_append_map_varchar_varchar(a, pk.data(), lk.data(), pv.data(), lv.data(), entry_count);
}
