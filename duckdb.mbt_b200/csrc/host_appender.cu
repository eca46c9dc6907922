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

#include <string>

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
  // ENUM: labels (is_string) or Arrow dictionary indices (w_in bytes each) -> positions of w_out bytes
  bool is_enum = false, index_signed = false, dict_large = false;
  const uint8_t *dict_offsets = nullptr;  // dictionary indices: the Arrow dictionary's offsets (views when dict_view) at its own offset
  const uint8_t *dict_data = nullptr, *dict_validity = nullptr;
  int64_t dict_bit_offset = 0, dict_len = 0;
  // VARCHAR / BLOB from Arrow string views (is_view: `values` the 16-byte views of the slice) or from an Arrow dictionary of
  // strings (is_dict: `values` the indices, the dictionary in the dict_* fields; dict_view: its values are views).
  // view_bufs / view_sizes / nviews: the data buffers of those views and their sizes
  bool is_view = false, is_dict = false, dict_view = false;
  const void *const *view_bufs = nullptr;
  const int64_t *view_sizes = nullptr;
  int64_t nviews = 0;
  // STRUCT: a mask and no payload (w_out 0).  Field columns follow the table's columns; `parent`: the STRUCT column
  // whose masks a field column's rows are ANDed with (-1: a table column)
  bool is_struct = false;
  int parent = -1;
};

// an ENUM column's labels and internal width (duckdb_mb_gpu_appender_set_enum); width 0: not declared
struct EnumDecl {
  int32_t width = 0;
  std::vector<uint32_t> offsets;
  std::vector<uint8_t> data;
  std::vector<uint4> slots;  // the lookup table (dmb_rev_enum_table), two uint4 per slot
  uint32_t table_size = 0;
};

// the table's child type of a LIST column (duckdb_mb_gpu_appender_set_list); type_id 0: not declared
struct ListDecl {
  int32_t type_id = 0, dec_width = 0, dec_scale = 0;
};

// a STRUCT column's fields (duckdb_mb_gpu_appender_set_struct): field columns first .. first + types.size() - 1;
// first -1: not declared
struct StructDecl {
  int32_t first = -1;
  std::vector<int32_t> types;
};

// what duckdb_mb_gpu_appender_struct_field hands out during a sink call, per column: the sub-batch's vectors and masks
struct SinkCol {
  const uint8_t *data = nullptr;  // NULL for a STRUCT column
  const uint64_t *masks = nullptr;
  int w = 0;
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
  int32_t ncols = 0;                    // table columns; field columns of STRUCTs follow them in the per-column vectors
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
  std::vector<EnumDecl> enums;
  std::vector<StructDecl> structs;
  std::vector<int32_t> parent, field_index;  // field columns: the STRUCT column and the position in it (-1: table column)
  std::vector<SinkList> sink_lists;
  std::vector<SinkCol> sink_cols;  // valid while sink_chunk >= 0, every column and field column  // valid while sink_chunk >= 0: chunk sink_chunk of the sub-batch being handed over
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

// how messages name column c: "column 3", or for a field column the table column and the field path, "column 2, field 1.0"
std::string col_name(const App *a, int c) {
  std::string path;
  for (; c >= a->ncols; c = a->parent[(size_t)c]) path = std::to_string(a->field_index[(size_t)c]) + (path.empty() ? "" : "." + path);
  return "column " + std::to_string(c) + (path.empty() ? "" : ", field " + path);
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
bool map_decimal(App *a, const char *cn, const char *what, const char *fmt, int32_t type_id, int32_t *w, int32_t *s, ColInput *in) {
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
    fail(a, "%s: Arrow %s '%s' is not a decimal format", cn, what, fmt);
    return false;
  }
  if (bits != 128) {
    fail(a, "%s: Arrow %s '%s' is a %ld-bit decimal; only decimal128 can be appended to a %s column", cn, what, fmt, bits, col);
    return false;
  }
  if (p < 1 || p > 38 || sc > p) {
    fail(a, "%s: Arrow %s '%s' is not a DECIMAL(width, scale) DuckDB can store", cn, what, fmt);
    return false;
  }
  if (*w == 0) { *w = (int32_t)p; *s = (int32_t)sc; }
  if (sc != *s) {
    fail(a, "%s: Arrow %s '%s' has scale %ld; the column is %s", cn, what, fmt, sc, col);
    return false;
  }
  if (p > *w) {
    fail(a, "%s: Arrow %s '%s' has precision %ld; the column is %s", cn, what, fmt, p, col);
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
bool map_format(App *a, const char *cn, const char *what, const char *fmt, int32_t type_id, int32_t *dec_w, int32_t *dec_s, ColInput *in) {
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
        return map_decimal(a, cn, what, fmt, type_id, &w, &s, in);
      }
      break;
    case DMB_TYPE_UHUGEINT: case DMB_TYPE_UUID: if (is("w:16")) return fixed(16); break;
    case DMB_TYPE_DECIMAL: if (starts("d:")) return map_decimal(a, cn, what, fmt, type_id, dec_w, dec_s, in); break;
    case DMB_TYPE_VARCHAR:
      if (is("u") || is("U")) { in->is_string = true; in->large = is("U"); in->w_out = 16; return true; }
      if (is("vu")) { fixed(16); in->is_view = true; return true; }
      break;
    case DMB_TYPE_BLOB:
      if (is("z") || is("Z")) { in->is_string = true; in->large = is("Z"); in->w_out = 16; return true; }
      if (is("vz")) { fixed(16); in->is_view = true; return true; }
      break;
    default: break;
  }
  fail(a, "%s: Arrow %s '%s' cannot be appended to a column of DuckDB type %d", cn, what, fmt, type_id);
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
  uint8_t *d_dense = nullptr;  // a dictionary child: the element validity the gather writes, bit 0 = element e0
  size_t child_cap = 0, h_child_cap = 0, words_cap = 0, h_words_cap = 0, dense_cap = 0;
  int64_t *d_cword = nullptr, *h_cword = nullptr;
  int64_t child_bytes = 0, words = 0, e0 = 0;
};

struct Slot {  // device + pinned buffers of one in-flight sub-batch
  std::vector<uint8_t *> d_out, h_out;
  std::vector<uint64_t *> d_val, h_val;
  std::vector<ListOut> lists;                     // [ncols], used by LIST columns
  unsigned int *d_err = nullptr, *h_err = nullptr;  // [ncols]: rev_list_kernel error flags
  // [ncols]: the first offending row of an ENUM, view or dictionary column, or element of a LIST column's view or
  // dictionary child (~0: none)
  unsigned long long *d_eerr = nullptr, *h_eerr = nullptr;
  cudaEvent_t ev_out = nullptr;
  int64_t r0 = 0, r1 = 0;
  bool busy = false;
};

// Arrow offset of `row` (strings, lists), read on the host
int64_t offset_at(const ColInput &ci, int64_t row) {
  if (ci.large) { int64_t v; memcpy(&v, ci.offsets + 8 * row, 8); return v; }
  int32_t v; memcpy(&v, ci.offsets + 4 * row, 4); return v;
}

// the Arrow dictionary index of `row`, read on the host; false (with the appender error, `what` naming the row) when it
// is outside the dictionary
bool dict_index_at(App *a, const char *cn, const char *what, const ColInput &ci, int64_t row, int64_t *idx) {
  uint64_t raw = 0;
  memcpy(&raw, ci.values + (size_t)row * (size_t)ci.w_in, (size_t)ci.w_in);
  const int sh = 64 - 8 * ci.w_in;
  *idx = ci.index_signed ? (int64_t)(raw << sh) >> sh : (int64_t)raw;
  if (*idx >= 0 && *idx < ci.dict_len) return true;
  fail(a, "%s, %s %lld: dictionary index %lld is outside the Arrow dictionary (%lld entries)", cn, what, (long long)row, (long long)*idx,
       (long long)ci.dict_len);
  return false;
}

// the appender error for the first offending row of a VARCHAR / BLOB column read from string views or a dictionary,
// rendered from the host buffers (`what`: "row", "list element" or "dictionary entry")
int32_t string_error(App *a, const char *cn, const char *what, const ColInput &ci, int64_t row) {
  int64_t idx;
  if (ci.is_dict) return dict_index_at(a, cn, what, ci, row, &idx) ? fail(a, "%s, %s %lld: malformed", cn, what, (long long)row) : 0;
  int32_t v[4];
  memcpy(v, ci.values + (size_t)row * 16, 16);
  const long long r = (long long)row;
  if (v[0] < 0) return fail(a, "%s, %s %lld: string view length %d is negative", cn, what, r, v[0]);
  if ((uint32_t)v[2] >= (uint64_t)ci.nviews)
    return fail(a, "%s, %s %lld: string view buffer index %u is outside the array's %lld data buffers", cn, what, r, (uint32_t)v[2], (long long)ci.nviews);
  if (v[3] < 0) return fail(a, "%s, %s %lld: string view offset %d is negative", cn, what, r, v[3]);
  return fail(a, "%s, %s %lld: string view bytes [%d, %lld) pass the end of data buffer %d (%lld bytes)", cn, what, r, v[3],
              (long long)v[3] + v[0], v[2], (long long)ci.view_sizes[v[2]]);
}

// the appender error for the first offending row of an ENUM column, rendered from the host buffers
int32_t enum_error(App *a, const char *cn, const ColInput &ci, int64_t row) {
  const uint8_t *p;
  int64_t len;
  if (ci.is_string) {
    const int64_t o0 = offset_at(ci, row);
    p = ci.data + o0;
    len = offset_at(ci, row + 1) - o0;
  } else {
    int64_t idx;
    if (!dict_index_at(a, cn, "row", ci, row, &idx)) return 0;
    ColInput d;
    d.offsets = ci.dict_offsets;
    d.large = ci.dict_large;
    const int64_t o0 = offset_at(d, idx);
    p = ci.dict_data + o0;
    len = offset_at(d, idx + 1) - o0;
  }
  const int shown = len > 160 ? 160 : (int)len;  // the message fits the 256-byte error buffer
  return fail(a, "%s, row %lld: '%.*s'%s is not a label of the ENUM", cn, (long long)row, shown, (const char *)p,
              len > shown ? "..." : "");
}

// the conversion of column `ci` itself, or of its LIST child, reports its first offending row in the slot's error word
bool uses_error_word(const ColInput &ci) {
  const ColInput &x = ci.is_list ? *ci.child : ci;
  return x.is_enum || x.is_view || x.is_dict;
}

// the Arrow dictionary of a dictionary column as a column of its own: utf8 / large_utf8 / binary / large_binary or views
ColInput dict_values(const ColInput &ci) {
  ColInput d;
  d.is_string = !ci.dict_view;
  d.is_view = ci.dict_view;
  d.large = ci.dict_large;
  d.offsets = ci.dict_offsets;
  d.data = ci.dict_data;
  d.validity = ci.dict_validity;
  d.bit_offset = ci.dict_bit_offset;
  d.w_out = 16;
  if (ci.dict_view) {
    d.values = ci.dict_offsets;
    d.w_in = 16;
    d.rev_op = DMB_REV_COPY16;
    d.view_bufs = ci.view_bufs;
    d.view_sizes = ci.view_sizes;
    d.nviews = ci.nviews;
  }
  return d;
}

// `h_derr`: per column, the first malformed string view of a dictionary of views (~0: none; NULL: no such dictionary)
int32_t sink_slot(App *a, Slot &s, const std::vector<ColInput> &cols, const std::vector<std::vector<int64_t>> &bounds,
                  const unsigned long long *h_derr) {
  if (!s.busy) return 1;
  if (check_cuda(cudaEventSynchronize(s.ev_out), "appender copy-out wait")) return fail(a, "%s", duckdb_mb_gpu_last_error());
  s.busy = false;
  const int nc = (int)cols.size();
  for (int c = 0; c < nc; ++c) {  // a malformed sub-batch reaches no sink
    const ColInput &ci = cols[(size_t)c];
    const ColInput &x = ci.is_list ? *ci.child : ci;
    if (h_derr && h_derr[c] != ~0ull) return string_error(a, col_name(a, c).c_str(), "dictionary entry", dict_values(x), (int64_t)h_derr[c]);
    if (ci.is_list && s.h_err[c])
      return fail(a, "column %d: Arrow list offsets decrease within rows [%lld, %lld)", c, (long long)s.r0, (long long)s.r1);
    if (!uses_error_word(ci) || s.h_eerr[c] == ~0ull) continue;
    if (ci.is_enum) return enum_error(a, col_name(a, c).c_str(), ci, s.r0 + (int64_t)s.h_eerr[c]);
    if (ci.is_list) return string_error(a, col_name(a, c).c_str(), "list element", x, s.lists[(size_t)c].e0 + (int64_t)s.h_eerr[c]);
    return string_error(a, col_name(a, c).c_str(), "row", ci, s.r0 + (int64_t)s.h_eerr[c]);
  }
  if (!a->sink) return 1;
  const int nt = a->ncols;  // the sink sees the table's columns; field columns through duckdb_mb_gpu_appender_struct_field
  std::vector<const void *> vd((size_t)nt);
  std::vector<const uint64_t *> vv((size_t)nt);
  a->sink_lists.assign((size_t)nc, SinkList());
  a->sink_cols.assign((size_t)nc, SinkCol());
  for (int c = 0; c < nc; ++c) {
    const int w = cols[(size_t)c].w_out;
    a->sink_cols[(size_t)c] = SinkCol{w ? s.h_out[(size_t)c] : nullptr, s.h_val[(size_t)c], w};
  }
  for (int c = 0; c < nc; ++c)
    if (cols[(size_t)c].is_list) {
      const ListOut &lo = s.lists[(size_t)c];
      a->sink_lists[(size_t)c] = SinkList{lo.h_child, (const uint64_t *)lo.h_words, bounds[(size_t)c].data() + s.r0 / DMB_VECTOR_SIZE,
                                          lo.h_cword, cols[(size_t)c].child->w_out};
    }
  for (int64_t r = s.r0, k = 0; r < s.r1; r += DMB_VECTOR_SIZE, ++k) {
    const uint32_t count = (uint32_t)(s.r1 - r < DMB_VECTOR_SIZE ? s.r1 - r : DMB_VECTOR_SIZE);
    for (int c = 0; c < nt; ++c) {
      const int w = cols[(size_t)c].w_out;
      vd[(size_t)c] = w ? s.h_out[(size_t)c] + (size_t)k * DMB_VECTOR_SIZE * (size_t)w : nullptr;
      vv[(size_t)c] = s.h_val[(size_t)c] + (size_t)k * DMB_VALIDITY_WORDS;
    }
    a->sink_chunk = k;
    const int32_t ok = a->sink(a->user, nt, count, vd.data(), vv.data());
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

// per column, the job fields of its conversion (or its LIST child's) that do not change between sub-batches
struct CallTables {
  std::vector<dmb_rev_enum_job> enums;  // ENUM columns
  std::vector<dmb_rev_view_job> views;  // string views: the table of data buffers
  std::vector<dmb_rev_dict_job> dicts;  // dictionaries of strings: the string_t table of the entries
  unsigned long long *d_err = nullptr, *h_err = nullptr;  // a dictionary of views: its first malformed entry (~0: none)
};

// Once per conversion, before the first sub-batch's kernels:
//  * every ENUM column's lookup table and labels go to the device, and for a dictionary column the Arrow dictionary too,
//    whose labels the lookup kernel turns into the remap (one code per dictionary entry) that the index kernel of every
//    sub-batch reads;
//  * a string view column's data buffers become a device table of {host base, size};
//  * a VARCHAR / BLOB dictionary column's dictionary is converted to string_t by the string or view kernel, the table
//    every sub-batch's gather reads, and its NULL entries are marked.
int32_t stage_tables(App *a, Scope &sc, const std::vector<ColInput> &cols, CallTables *t) {
  CtxCore &c = *a->core;
  const size_t nc = cols.size();
  t->enums.assign(nc, dmb_rev_enum_job());
  t->views.assign(nc, dmb_rev_view_job());
  t->dicts.assign(nc, dmb_rev_dict_job());
  std::vector<dmb_rev_enum_job> remaps;
  std::vector<int64_t> remap_rows;
  std::vector<dmb_rev_string_job> str_builds;
  std::vector<dmb_rev_view_job> view_builds;
  std::vector<int64_t> str_rows, view_rows;
  std::vector<std::pair<dmb_string_t *, std::pair<const uint64_t *, int64_t>>> marks;
  // the {host base, size} table of a view array's data buffers
  auto buffer_table = [&](const ColInput &v, const dmb_view_buffer **out) {
    std::vector<dmb_view_buffer> hb((size_t)v.nviews);
    for (int64_t i = 0; i < v.nviews; ++i) hb[(size_t)i] = dmb_view_buffer{(uint64_t)(uintptr_t)v.view_bufs[i], v.view_sizes[i]};
    void *d = sc.dalloc(hb.size() * sizeof(dmb_view_buffer) + 16);
    if (!d || (!hb.empty() && stage_contiguous(c, c.s_in, d, hb.data(), hb.size() * sizeof(dmb_view_buffer), -1, &a->bytes_h2d))) return false;
    *out = (const dmb_view_buffer *)d;
    return true;
  };
  for (size_t j = 0; j < nc; ++j) {
    const ColInput &ci = cols[j].is_list ? *cols[j].child : cols[j];
    if (ci.is_view) {
      dmb_rev_view_job &vj = t->views[j];
      vj.nbuffers = ci.nviews;
      if (!buffer_table(ci, &vj.buffers)) return fail(a, "%s", duckdb_mb_gpu_last_error());
      continue;
    }
    if (ci.is_dict) {
      dmb_rev_dict_job &dj = t->dicts[j];
      dj.index_width = ci.w_in;
      dj.index_signed = ci.index_signed ? 1 : 0;
      dj.dict_len = ci.dict_len;
      if (ci.dict_len == 0) continue;  // every valid row is out of range
      const ColInput d = dict_values(ci);
      const int64_t cap = ((ci.dict_len + DMB_VECTOR_SIZE - 1) / DMB_VECTOR_SIZE) * DMB_VECTOR_SIZE;  // the kernels fill whole chunks
      dmb_string_t *table = (dmb_string_t *)sc.dalloc((size_t)cap * sizeof(dmb_string_t));
      uint64_t *masks = (uint64_t *)sc.dalloc((size_t)cap / 8);
      if (!table || !masks) return fail(a, "%s", duckdb_mb_gpu_last_error());
      InBuf ib;
      dmb_rev_fixed_job fj;
      dmb_rev_string_job sj;
      const uint8_t *d_validity = nullptr;
      int64_t bit_off = 0;
      if (!stage_rows(a, sc, d, ib, (int)j, 0, ci.dict_len, table, masks, &fj, &sj, &d_validity, &bit_off)) return 0;
      if (d.is_view) {
        if (!t->d_err) {
          t->d_err = (unsigned long long *)sc.dalloc(8 * nc);
          t->h_err = (unsigned long long *)sc.palloc(8 * nc);
          if (!t->d_err || !t->h_err) return fail(a, "%s", duckdb_mb_gpu_last_error());
        }
        dmb_rev_view_job vj;
        memset(&vj, 0, sizeof(vj));
        vj.nbuffers = d.nviews;
        if (!buffer_table(d, &vj.buffers)) return fail(a, "%s", duckdb_mb_gpu_last_error());
        vj.in_views = fj.in_values;
        vj.in_validity = d_validity;
        vj.in_bit_offset = bit_off;
        vj.out = table;
        vj.out_validity = masks;
        vj.error = t->d_err + j;
        view_builds.push_back(vj);
        view_rows.push_back(ci.dict_len);
      } else {
        str_builds.push_back(sj);
        str_rows.push_back(ci.dict_len);
      }
      if (d.validity) marks.push_back({table, {masks, ci.dict_len}});
      dj.table = table;
      continue;
    }
    if (!ci.is_enum) continue;
    const EnumDecl &e = a->enums[j];
    dmb_rev_enum_job &ej = t->enums[j];
    memset(&ej, 0, sizeof(ej));
    ej.out_width = e.width;
    const size_t tb = e.slots.size() * sizeof(uint4), ob = e.offsets.size() * 4;
    uint8_t *table = (uint8_t *)sc.dalloc(tb), *loff = (uint8_t *)sc.dalloc(ob), *ldata = (uint8_t *)sc.dalloc(e.data.size() + 16);
    if (!table || !loff || !ldata || stage_contiguous(c, c.s_in, table, e.slots.data(), tb, -1, &a->bytes_h2d) ||
        stage_contiguous(c, c.s_in, loff, e.offsets.data(), ob, -1, &a->bytes_h2d) ||
        (!e.data.empty() && stage_contiguous(c, c.s_in, ldata, e.data.data(), e.data.size(), -1, &a->bytes_h2d)))
      return fail(a, "%s", duckdb_mb_gpu_last_error());
    ej.table = table;
    ej.table_size = e.table_size;
    ej.label_offsets = (const uint32_t *)loff;
    ej.label_data = ldata;
    if (ci.is_string) continue;
    ej.index_width = ci.w_in;
    ej.index_signed = ci.index_signed ? 1 : 0;
    ej.dict_len = ci.dict_len;
    if (ci.dict_len == 0) continue;  // every valid row is out of range
    const ColInput d = dict_values(ci);  // its codes are the remap
    InBuf ib;
    dmb_rev_fixed_job fj;
    dmb_rev_string_job sj;
    const uint8_t *d_validity = nullptr;
    int64_t bit_off = 0;
    uint32_t *remap = (uint32_t *)sc.dalloc(4 * (size_t)ci.dict_len);
    if (!remap) return fail(a, "%s", duckdb_mb_gpu_last_error());
    if (!stage_rows(a, sc, d, ib, (int)j, 0, ci.dict_len, nullptr, nullptr, &fj, &sj, &d_validity, &bit_off)) return 0;
    dmb_rev_enum_job rj = ej;
    rj.index_width = 0;
    rj.out_width = 0;
    rj.in_offsets = sj.in_offsets;
    rj.in_data = sj.in_data;
    rj.large_offsets = sj.large_offsets;
    rj.in_validity = d_validity;
    rj.in_bit_offset = bit_off;
    rj.out = remap;
    remaps.push_back(rj);
    remap_rows.push_back(ci.dict_len);
    ej.remap = remap;
  }
  if (remaps.empty() && str_builds.empty() && view_builds.empty()) return 1;
  cudaEvent_t ev = sc.event(false);
  if (!ev || check_cuda(cudaEventRecord(ev, c.s_in), "dictionary staging") || check_cuda(cudaStreamWaitEvent(c.s_compute, ev, 0), "wait dictionary staging"))
    return fail(a, "%s", duckdb_mb_gpu_last_error());
  for (size_t i = 0; i < remaps.size(); ++i)
    if (dmb_dev_rev_enum_batch(&remaps[i], remap_rows[i], c.s_compute)) return fail(a, "%s", duckdb_mb_gpu_last_error());
  for (size_t i = 0; i < str_builds.size(); ++i)
    if (dmb_dev_rev_string_batch(&str_builds[i], str_rows[i], c.s_compute)) return fail(a, "%s", duckdb_mb_gpu_last_error());
  if (t->d_err && check_cuda(cudaMemsetAsync(t->d_err, 0xff, 8 * nc, c.s_compute), "dictionary error words reset"))
    return fail(a, "%s", duckdb_mb_gpu_last_error());
  for (size_t i = 0; i < view_builds.size(); ++i)
    if (dmb_dev_rev_view_batch(&view_builds[i], view_rows[i], c.s_compute)) return fail(a, "%s", duckdb_mb_gpu_last_error());
  for (const auto &m : marks)
    if (dmb_dev_rev_dict_mark(m.first, m.second.first, m.second.second, c.s_compute)) return fail(a, "%s", duckdb_mb_gpu_last_error());
  // read back before the first sub-batch's kernels, so before its copy-out, which sink_slot waits for
  if (t->d_err && check_cuda(cudaMemcpyAsync(t->h_err, t->d_err, 8 * nc, cudaMemcpyDeviceToHost, c.s_compute), "dictionary error words D2H"))
    return fail(a, "%s", duckdb_mb_gpu_last_error());
  return 1;
}

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
    slots[s].d_eerr = (unsigned long long *)sc.dalloc(8 * (size_t)nc);
    slots[s].h_eerr = (unsigned long long *)sc.palloc(8 * (size_t)nc);
    if (!slots[s].ev_out || !slots[s].d_err || !slots[s].h_err || !slots[s].d_eerr || !slots[s].h_eerr) return fail(a, "%s", duckdb_mb_gpu_last_error());
    for (int j = 0; j < nc; ++j) {
      const size_t ob = (size_t)sub * (size_t)cols[(size_t)j].w_out, vb = (size_t)sub_chunks * DMB_VALIDITY_WORDS * 8;
      uint8_t *d = ob ? (uint8_t *)sc.dalloc(ob) : nullptr, *h = ob ? (uint8_t *)sc.palloc(ob) : nullptr;  // STRUCT: no payload
      uint64_t *dv = (uint64_t *)sc.dalloc(vb), *hv = (uint64_t *)sc.palloc(vb);
      if ((ob && (!d || !h)) || !dv || !hv) return fail(a, "%s", duckdb_mb_gpu_last_error());
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
  // STRUCT columns: a column is "masked" when it or an ancestor STRUCT has an Arrow bitmap.  Then rev_mask_kernel writes
  // its masks from its bitmap AND its parent's masks, and for each field that is not a STRUCT the parent's masks AND the
  // field's bitmap into comb[slot][field], which the field's conversion reads as its validity.  Jobs of nesting level d
  // read the masks of level d - 1: one launch per level.  (A field column's number is above its parent's.)
  std::vector<char> masked((size_t)nc, 0);
  std::vector<int> depth((size_t)nc, 0);
  int levels = 0;
  for (int j = 0; j < nc; ++j) {
    const ColInput &ci = cols[(size_t)j];
    const int p = ci.parent;
    depth[(size_t)j] = p < 0 ? 0 : depth[(size_t)p] + 1;
    if (ci.is_struct) masked[(size_t)j] = ci.validity != nullptr || (p >= 0 && masked[(size_t)p]);
    if (ci.is_struct || (p >= 0 && masked[(size_t)p])) levels = depth[(size_t)j] + 1 > levels ? depth[(size_t)j] + 1 : levels;
  }
  std::vector<uint64_t *> comb((size_t)nslots * (size_t)nc, nullptr);
  dmb_rev_mask_job *h_mjobs = nullptr, *d_mjobs = nullptr;
  if (levels) {
    h_mjobs = (dmb_rev_mask_job *)sc.palloc(sizeof(dmb_rev_mask_job) * (size_t)nc * 2);
    d_mjobs = (dmb_rev_mask_job *)sc.dalloc(sizeof(dmb_rev_mask_job) * (size_t)nc * 2);
    if (!h_mjobs || !d_mjobs) return fail(a, "%s", duckdb_mb_gpu_last_error());
    for (int s = 0; s < nslots; ++s)
      for (int j = 0; j < nc; ++j)
        if (!cols[(size_t)j].is_struct && cols[(size_t)j].parent >= 0 && masked[(size_t)cols[(size_t)j].parent]) {
          uint64_t *&cb = comb[(size_t)s * (size_t)nc + (size_t)j];
          cb = (uint64_t *)sc.dalloc((size_t)(sub_chunks + 1) * DMB_VALIDITY_WORDS * 8);  // + 1 chunk: a BOOLEAN field's bit phase
          if (!cb) return fail(a, "%s", duckdb_mb_gpu_last_error());
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
  CallTables tabs;
  if (!stage_tables(a, sc, cols, &tabs)) return 0;
  bool any_err = false;  // some conversion reports rows in the slot's error words
  for (const ColInput &ci : cols) any_err = any_err || uses_error_word(ci);
  for (size_t b = 0; b + 1 < cuts.size(); ++b) {
    const int64_t r0 = cuts[b] * DMB_VECTOR_SIZE, r1 = cuts[b + 1] * DMB_VECTOR_SIZE < nrows ? cuts[b + 1] * DMB_VECTOR_SIZE : nrows;
    const int64_t n = r1 - r0;
    const int64_t nch = cuts[b + 1] - cuts[b];
    const int si = (int)(b % (size_t)nslots);
    Slot &slot = slots[si];
    if (!sink_slot(a, slot, cols, bounds, tabs.h_err)) return 0;  // the slot's previous sub-batch leaves first
    // the job array of this slot is reused as well: its previous launch has completed (sink_slot waited)
    dmb_rev_fixed_job *hj = h_jobs + (size_t)si * (size_t)nc * 2, *dj = d_jobs + (size_t)si * (size_t)nc * 2;
    int nfixed = 0, nchild_fixed = 0;
    cudaEvent_t ev_in = sc.event(false), ev_k = sc.event(false), k0 = sc.event(true), k1 = sc.event(true);
    if (!ev_in || !ev_k || !k0 || !k1) return fail(a, "%s", duckdb_mb_gpu_last_error());
    std::vector<dmb_rev_string_job> strs;
    std::vector<dmb_rev_list_job> lists;
    std::vector<dmb_rev_enum_job> enums;
    std::vector<dmb_rev_view_job> views;
    std::vector<dmb_rev_dict_job> dicts;
    std::vector<int64_t> view_rows, dict_rows;
    std::vector<int64_t> child_rows;  // element count of each child job: fixed-width ones first, in job order
    std::vector<int64_t> str_rows;
    std::vector<int> masks_from_bytes;  // columns
    std::vector<std::vector<dmb_rev_mask_job>> mask_levels((size_t)levels);
    for (int j = 0; j < nc; ++j) {
      const ColInput &ci = cols[(size_t)j];
      InBuf &ib = inbuf[(size_t)si * (size_t)nc + (size_t)j];
      const uint8_t *d_validity = nullptr;
      int64_t bit_off = 0;
      const bool under_mask = ci.parent >= 0 && masked[(size_t)ci.parent];
      const uint8_t *parent_masks = under_mask ? (const uint8_t *)slot.d_val[(size_t)ci.parent] : nullptr;
      if (ci.is_struct) {  // its masks only: own bitmap AND the parent's masks
        if (ci.validity) {
          bit_off = stage_bits(a, sc, ib.validity, ib.validity_cap, ci.validity, ci.bit_offset + r0, ci.bit_offset + r1);
          if (bit_off < 0) return fail(a, "%s", duckdb_mb_gpu_last_error());
          d_validity = ib.validity;
        }
        mask_levels[(size_t)depth[(size_t)j]].push_back(dmb_rev_mask_job{parent_masks, 0, d_validity, bit_off, slot.d_val[(size_t)j], 0});
        continue;
      }
      if (!ci.is_list) {
        dmb_rev_string_job sj;
        if (!stage_rows(a, sc, ci, ib, j, r0, r1, slot.d_out[(size_t)j], slot.d_val[(size_t)j], &hj[nfixed], &sj, &d_validity, &bit_off)) return 0;
        if (ci.valid_bytes) masks_from_bytes.push_back(j);
        if (under_mask) {  // the conversion reads parent masks AND own bitmap; a BOOLEAN field at its values' bit phase
          uint64_t *cb = comb[(size_t)si * (size_t)nc + (size_t)j];
          const int64_t phase = ci.is_bits ? hj[nfixed].in_bit_offset : 0;
          mask_levels[(size_t)depth[(size_t)j]].push_back(dmb_rev_mask_job{parent_masks, 0, d_validity, bit_off, cb, phase});
          d_validity = (const uint8_t *)cb;
          bit_off = phase;
          hj[nfixed].in_validity = d_validity;
          hj[nfixed].in_bit_offset = phase;
          sj.in_validity = d_validity;
          sj.in_bit_offset = 0;
        }
        if (ci.is_enum) {
          dmb_rev_enum_job ej = tabs.enums[(size_t)j];
          if (ci.is_string) {
            ej.in_offsets = sj.in_offsets;
            ej.in_data = sj.in_data;
            ej.large_offsets = sj.large_offsets;
          } else {
            ej.in_indices = hj[nfixed].in_values;  // (that job slot is reused by the next fixed-width column)
          }
          ej.in_validity = d_validity;
          ej.in_bit_offset = bit_off;
          ej.out = slot.d_out[(size_t)j];
          ej.out_validity = slot.d_val[(size_t)j];
          ej.error = slot.d_eerr + j;
          enums.push_back(ej);
        } else if (ci.is_view) {
          dmb_rev_view_job vj = tabs.views[(size_t)j];
          vj.in_views = hj[nfixed].in_values;  // (that job slot is reused by the next fixed-width column)
          vj.in_validity = d_validity;
          vj.in_bit_offset = bit_off;
          vj.out = (dmb_string_t *)slot.d_out[(size_t)j];
          vj.out_validity = slot.d_val[(size_t)j];
          vj.error = slot.d_eerr + j;
          views.push_back(vj);
          view_rows.push_back(n);
        } else if (ci.is_dict) {
          dmb_rev_dict_job dj = tabs.dicts[(size_t)j];
          dj.in_indices = hj[nfixed].in_values;
          dj.in_validity = d_validity;
          dj.in_bit_offset = bit_off;
          dj.out = (dmb_string_t *)slot.d_out[(size_t)j];
          dj.out_validity = slot.d_val[(size_t)j];
          dj.error = slot.d_eerr + j;
          dicts.push_back(dj);
          dict_rows.push_back(n);
        } else if (ci.is_string) { strs.push_back(sj); str_rows.push_back(n); }
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
      // the string, view and dictionary kernels fill whole vectors
      const bool whole = cc.is_string || cc.is_view || cc.is_dict;
      const int64_t child_slots = whole ? ((ne + DMB_VECTOR_SIZE - 1) / DMB_VECTOR_SIZE) * DMB_VECTOR_SIZE : ne;
      lo.child_bytes = ne * cc.w_out;
      lo.e0 = e0;
      if (!grow(sc, lo.d_child, lo.child_cap, (size_t)child_slots * (size_t)cc.w_out + 64) ||
          (cc.is_dict && !grow(sc, lo.d_dense, lo.dense_cap, (size_t)child_slots / 8 + 64)) ||
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
        // A view or dictionary child is judged by its own bitmap alone: an element the child marks valid is checked even in
        // the segment of a NULL list row, which Arrow's validation of the child array requires as well.
        if (cc.is_view) {
          dmb_rev_view_job vj = tabs.views[(size_t)j];
          vj.in_views = fj->in_values;  // (that job slot is reused by the next child)
          vj.in_validity = d_cvalidity;
          vj.in_bit_offset = cbit_off;
          vj.out = (dmb_string_t *)lo.d_child;
          vj.error = slot.d_eerr + j;
          views.push_back(vj);
          view_rows.push_back(ne);
        } else if (cc.is_dict) {  // a NULL dictionary entry makes an element NULL: the list kernel reads the gather's bitmap
          dmb_rev_dict_job dj = tabs.dicts[(size_t)j];
          dj.in_indices = fj->in_values;
          dj.in_validity = d_cvalidity;
          dj.in_bit_offset = cbit_off;
          dj.out = (dmb_string_t *)lo.d_child;
          dj.out_validity = (uint64_t *)lo.d_dense;
          dj.error = slot.d_eerr + j;
          dicts.push_back(dj);
          dict_rows.push_back(ne);
          d_cvalidity = lo.d_dense;
          cbit_off = 0;
        } else if (cc.is_string) { strs.push_back(sj); str_rows.push_back(ne); }
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
    if (levels) {  // STRUCT masks and the combined bitmaps of the fields, level by level, before the conversions read them
      dmb_rev_mask_job *hm = h_mjobs + (size_t)si * (size_t)nc, *dm = d_mjobs + (size_t)si * (size_t)nc;
      size_t nm = 0;
      for (const auto &lv : mask_levels)
        for (const auto &mj : lv) hm[nm++] = mj;
      if (nm && check_cuda(cudaMemcpyAsync(dm, hm, sizeof(dmb_rev_mask_job) * nm, cudaMemcpyHostToDevice, c.s_compute), "mask job H2D"))
        return fail(a, "%s", duckdb_mb_gpu_last_error());
      for (size_t l = 0, at = 0; l < mask_levels.size(); at += mask_levels[l].size(), ++l)
        if (dmb_dev_rev_mask_batch(dm + at, hm + at, (int32_t)mask_levels[l].size(), n, c.s_compute)) return fail(a, "%s", duckdb_mb_gpu_last_error());
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
    if (any_err && check_cuda(cudaMemsetAsync(slot.d_eerr, 0xff, 8 * (size_t)nc, c.s_compute), "error words reset"))
      return fail(a, "%s", duckdb_mb_gpu_last_error());
    for (auto &ej : enums)
      if (dmb_dev_rev_enum_batch(&ej, n, c.s_compute)) return fail(a, "%s", duckdb_mb_gpu_last_error());
    for (size_t i = 0; i < views.size(); ++i)
      if (dmb_dev_rev_view_batch(&views[i], view_rows[i], c.s_compute)) return fail(a, "%s", duckdb_mb_gpu_last_error());
    for (size_t i = 0; i < dicts.size(); ++i)
      if (dmb_dev_rev_dict_batch(&dicts[i], dict_rows[i], c.s_compute)) return fail(a, "%s", duckdb_mb_gpu_last_error());
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
      if ((ob && check_cuda(cudaMemcpyAsync(slot.h_out[(size_t)j], slot.d_out[(size_t)j], ob, cudaMemcpyDeviceToHost, c.s_out), "vectors D2H")) ||
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
    if (any_err && check_cuda(cudaMemcpyAsync(slot.h_eerr, slot.d_eerr, 8 * (size_t)nc, cudaMemcpyDeviceToHost, c.s_out), "error words D2H"))
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
    if (!sink_slot(a, slot, cols, bounds, tabs.h_err)) return 0;
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
      if (a->type_ids[(size_t)j] == DMB_TYPE_ENUM) {  // labels -> positions (set_enum declared the column before begin_row)
        ci.is_enum = true;
        ci.w_out = a->enums[(size_t)j].width;
      }
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
  } else if (ci.is_view) {  // validity, views, the data buffers, their sizes
    ci.values = arr->n_buffers > 1 && arr->buffers[1] ? (const uint8_t *)arr->buffers[1] + (size_t)off * 16 : nullptr;
    ci.nviews = arr->n_buffers >= 3 ? arr->n_buffers - 3 : 0;
    ci.view_bufs = arr->buffers + 2;
    ci.view_sizes = arr->n_buffers >= 3 ? (const int64_t *)arr->buffers[arr->n_buffers - 1] : nullptr;
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

// a string view array's buffers: validity, views, k data buffers, then the k sizes.  With k = 0 the sizes buffer is empty,
// and Arrow C++ exports it as NULL: an all-NULL, empty or all-inline array.
bool check_views(App *a, const char *cn, const ArrowArray *arr) {
  if (arr->n_buffers < 3) {
    fail(a, "%s: the Arrow string view array is malformed: it has %lld buffers, and needs validity, views, its data buffers and "
         "their sizes (at least 3)", cn, (long long)arr->n_buffers);
    return false;
  }
  if (arr->n_buffers > 3 && !arr->buffers[arr->n_buffers - 1]) {
    fail(a, "%s: the Arrow string view array is malformed: its %lld data buffers come without their sizes", cn,
         (long long)(arr->n_buffers - 3));
    return false;
  }
  return true;
}

// the index width and signedness of an Arrow dictionary's index format, false when it is not an integer format
bool map_dict_indices(const char *fmt, ColInput *ci) {
  if (strlen(fmt) != 1 || !strchr("cCsSiIlL", fmt[0])) return false;
  const char f = fmt[0];
  ci->w_in = f == 'c' || f == 'C' ? 1 : f == 's' || f == 'S' ? 2 : f == 'i' || f == 'I' ? 4 : 8;
  ci->rev_op = copy_op(ci->w_in);
  ci->index_signed = f >= 'a' && f <= 'z';
  return true;
}

// the Arrow dictionary `d` (values of format `dfmt`: u U z Z, or vu vz) into the dict_* fields of `ci`
bool bind_dict(App *a, const char *cn, const ArrowArray *d, const char *dfmt, ColInput *ci) {
  static const uint8_t kNoData[16] = {0};
  if (!d) {
    fail(a, "%s: the Arrow dictionary array is missing", cn);
    return false;
  }
  ci->dict_view = dfmt[0] == 'v';
  ci->dict_large = dfmt[0] == 'U' || dfmt[0] == 'Z';
  ci->dict_len = d->length;
  ci->dict_bit_offset = d->offset;
  ci->dict_validity = (d->null_count != 0 && d->n_buffers > 0) ? (const uint8_t *)d->buffers[0] : nullptr;
  const int ew = ci->dict_view ? 16 : ci->dict_large ? 8 : 4;
  ci->dict_offsets = d->n_buffers > 1 && d->buffers[1] ? (const uint8_t *)d->buffers[1] + (size_t)d->offset * (size_t)ew : nullptr;
  if (ci->dict_view) {
    if (!check_views(a, cn, d)) return false;
    ci->nviews = d->n_buffers - 3;
    ci->view_bufs = d->buffers + 2;
    ci->view_sizes = (const int64_t *)d->buffers[d->n_buffers - 1];
  } else {
    ci->dict_data = d->n_buffers > 2 && d->buffers[2] ? (const uint8_t *)d->buffers[2] : kNoData;
  }
  if (d->length > 0 && !ci->dict_offsets) {
    fail(a, "%s: the Arrow dictionary has no %s buffer", cn, ci->dict_view ? "views" : "offsets");
    return false;
  }
  return true;
}

// an Arrow dictionary array (indices c C s S i I l L) of strings for a VARCHAR (u U vu) or BLOB (z Z vz) column, table column,
// field or LIST child
bool map_string_dict(App *a, const char *cn, const ArrowArray *arr, const ArrowSchema *sch, int32_t type_id, ColInput *ci) {
  const char *fmt = sch->format;
  const char *dfmt = sch->dictionary->format ? sch->dictionary->format : "";
  const bool blob = type_id == DMB_TYPE_BLOB;
  const char *col = blob ? "BLOB" : "VARCHAR";
  if (!map_dict_indices(fmt, ci)) {
    fail(a, "%s: Arrow dictionary index format '%s' cannot be appended to a %s column", cn, fmt, col);
    return false;
  }
  static const char *const kValues[2][3] = {{"u", "U", "vu"}, {"z", "Z", "vz"}};
  bool ok = false;
  for (const char *f : kValues[blob ? 1 : 0]) ok = ok || strcmp(dfmt, f) == 0;
  if (!ok) {
    fail(a, "%s: an Arrow dictionary of '%s' values cannot be appended to a %s column", cn, dfmt, col);
    return false;
  }
  if (!bind_dict(a, cn, arr->dictionary, dfmt, ci)) return false;
  ci->is_dict = true;
  ci->w_out = 16;
  return true;
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
  const std::string cn = col_name(a, j);
  if ((d.type_id == DMB_TYPE_VARCHAR || d.type_id == DMB_TYPE_BLOB) && sch->children[0]->dictionary) {
    if (!map_string_dict(a, cn.c_str(), carr, sch->children[0], d.type_id, child)) return false;
  } else if (!map_format(a, cn.c_str(), "list child format", cfmt, d.type_id, &dec_w, &dec_s, child)) {
    const bool decimal_child = d.type_id == DMB_TYPE_DECIMAL || d.type_id == DMB_TYPE_HUGEINT;
    if (!decimal_child || strncmp(cfmt, "d:", 2) != 0)  // map_decimal's refusal names its own reason
      fail(a, "column %d: Arrow list child format '%s' does not match the declared child type %d", j, cfmt, d.type_id);
    return false;
  }
  bind_buffers(*child, carr, carr->offset);
  if (child->is_view && !check_views(a, cn.c_str(), carr)) return false;
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

// an Arrow struct array for a STRUCT column whose fields are declared (duckdb_mb_gpu_appender_set_struct); map_column maps
// the fields
bool map_struct(App *a, int j, const char *cn, const ArrowArray *arr, const ArrowSchema *sch, ColInput *ci) {
  const char *fmt = sch->format;
  if (strcmp(fmt, "+s") != 0) {
    if (fmt[0] == '+') fail(a, "%s: an Arrow %s ('%s') cannot be appended to a STRUCT column", cn, nested_name(fmt), fmt);
    else fail(a, "%s: Arrow format '%s' cannot be appended to a STRUCT column", cn, fmt);
    return false;
  }
  const StructDecl &d = a->structs[(size_t)j];
  if (d.first < 0) {
    fail(a, "%s: the STRUCT column's fields are not declared (duckdb_mb_gpu_appender_set_struct)", cn);
    return false;
  }
  if (arr->n_children != (int64_t)d.types.size() || sch->n_children != (int64_t)d.types.size() || !arr->children || !sch->children) {
    fail(a, "%s: the Arrow struct has %lld fields, the STRUCT column %d", cn, (long long)arr->n_children, (int)d.types.size());
    return false;
  }
  ci->is_struct = true;
  ci->w_out = 0;
  return true;
}

// an Arrow array for an ENUM column: a dictionary array (indices c C s S i I l L, labels u / U) or plain u / U labels
bool map_enum(App *a, int j, const char *cn, const ArrowArray *arr, const ArrowSchema *sch, ColInput *ci) {
  const char *fmt = sch->format;
  const EnumDecl &e = a->enums[(size_t)j];
  if (!e.width) {
    fail(a, "%s: the ENUM column's labels are not declared (duckdb_mb_gpu_appender_set_enum)", cn);
    return false;
  }
  ci->is_enum = true;
  ci->w_out = e.width;
  const bool integer = strlen(fmt) == 1 && strchr("cCsSiIlL", fmt[0]);
  if (!sch->dictionary) {
    if (strcmp(fmt, "u") == 0 || strcmp(fmt, "U") == 0) {
      ci->is_string = true;
      ci->large = fmt[0] == 'U';
      return true;
    }
    if (strcmp(fmt, "vu") == 0) fail(a, "%s: Arrow string views ('vu') cannot be appended to an ENUM column", cn);
    else if (integer) fail(a, "%s: a bare Arrow integer array ('%s') cannot be appended to an ENUM column: pass a dictionary array or utf8 labels", cn, fmt);
    else if (fmt[0] == '+') fail(a, "%s: an Arrow %s ('%s') cannot be appended to an ENUM column", cn, nested_name(fmt), fmt);
    else fail(a, "%s: Arrow format '%s' cannot be appended to an ENUM column", cn, fmt);
    return false;
  }
  const char *dfmt = sch->dictionary->format ? sch->dictionary->format : "";
  if (!integer) {
    fail(a, "%s: Arrow dictionary index format '%s' cannot be appended to an ENUM column", cn, fmt);
    return false;
  }
  if (strcmp(dfmt, "u") != 0 && strcmp(dfmt, "U") != 0) {
    fail(a, "%s: an Arrow dictionary of '%s' values cannot be appended to an ENUM column (the labels must be utf8 or large_utf8)", cn, dfmt);
    return false;
  }
  map_dict_indices(fmt, ci);
  return bind_dict(a, cn, arr->dictionary, dfmt, ci);
}

// Arrow array `arr` -> column j (a table column or a field column) of `cols`: row i of the batch is logical row at + i of
// `arr`.  A STRUCT maps its fields the same way, at arr->offset + at: in the Arrow C data interface a struct's offset is not
// applied to its children.
bool map_column(App *a, int j, const ArrowArray *arr, const ArrowSchema *sch, int64_t at, int64_t n, std::vector<ColInput> &cols,
                std::vector<ColInput> &children) {
  const std::string name = col_name(a, j);
  const char *cn = name.c_str();
  const bool field = j >= a->ncols;
  ColInput &ci = cols[(size_t)j];
  const int32_t t = a->type_ids[(size_t)j];
  if (arr && sch && sch->format && field && sch->format[0] == '+' && t != DMB_TYPE_STRUCT) {
    fail(a, "%s: an Arrow %s field ('%s') cannot be appended to a STRUCT", cn, nested_name(sch->format), sch->format);
    return false;
  }
  if (!arr || !sch || !sch->format ||
      !(t == DMB_TYPE_LIST ? map_list(a, j, arr, sch, &ci, &children[(size_t)j])
        : t == DMB_TYPE_ENUM ? map_enum(a, j, cn, arr, sch, &ci)
        : t == DMB_TYPE_STRUCT ? map_struct(a, j, cn, arr, sch, &ci)
        : (t == DMB_TYPE_VARCHAR || t == DMB_TYPE_BLOB) && sch->dictionary ? map_string_dict(a, cn, arr, sch, t, &ci)
                               : map_format(a, cn, field ? "field format" : "format", sch->format, t, &a->rows[(size_t)j].dec_prec,
                                            &a->rows[(size_t)j].dec_scale, &ci))) {
    if (!a->error[0]) fail(a, "append_arrow_batch: %s is malformed", cn);
    return false;
  }
  if (arr->length < at + n) {
    if (field) fail(a, "append_arrow_batch: %s is shorter than the rows it is read at (%lld of %lld)", cn, (long long)arr->length, (long long)(at + n));
    else fail(a, "append_arrow_batch: %s is shorter than the batch", cn);
    return false;
  }
  bind_buffers(ci, arr, arr->offset + at);
  if (ci.is_view && !check_views(a, cn, arr)) return false;
  if (ci.is_struct) {
    const StructDecl &d = a->structs[(size_t)j];
    for (int f = 0; f < (int)d.types.size(); ++f) {
      cols[(size_t)(d.first + f)].parent = j;
      if (!map_column(a, d.first + f, arr->children[f], sch->children[f], arr->offset + at, n, cols, children)) return false;
    }
    return true;
  }
  if (n > 0 && (((ci.is_string || ci.is_list) && !ci.offsets) || (!ci.is_string && !ci.is_list && !ci.values))) {
    fail(a, "append_arrow_batch: %s has no value buffer", cn);
    return false;
  }
  return true;
}

// the current cell of a row in progress belongs to an ENUM column
bool enum_cell(App *a) {
  return a->state == kRowInProgress && a->cur_col < a->ncols && a->type_ids[(size_t)a->cur_col] == DMB_TYPE_ENUM;
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
  a->enums.resize((size_t)ncols);
  a->structs.resize((size_t)ncols);
  a->parent.assign((size_t)ncols, -1);
  a->field_index.assign((size_t)ncols, -1);
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
  const size_t total = a->type_ids.size();  // table columns and field columns
  std::vector<ColInput> cols(total), children(total);
  for (int j = 0; j < a->ncols; ++j)
    if (!map_column(a, j, batch->children[j], schema->children[j], batch->offset, n, cols, children)) {
      a->state = kError;
      return 0;
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
  for (int j = 0; j < a->ncols; ++j) {
    if (a->type_ids[(size_t)j] == DMB_TYPE_ENUM && !a->enums[(size_t)j].width) {
      fail(a, "begin_row: ENUM column %d has no declared labels (duckdb_mb_gpu_appender_set_enum)", j);
      a->state = kError;
      return 0;
    }
    if (a->rows[(size_t)j].width < 0) { fail(a, "begin_row: column %d (type %d) is only appendable through Arrow batches", j, a->type_ids[(size_t)j]); a->state = kError; return 0; }
  }
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
  if (a && enum_cell(a)) return type_mismatch(a, "append_blob");  // an ENUM cell takes VARCHAR labels only
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
int32_t append_text_cell(duckdb_mb_gpu_appender *a, const char *cmd, std::vector<uint8_t> &t) {
  if (enum_cell(a)) return type_mismatch(a, cmd);
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
  return append_text_cell(a, "append_list_varchar", t);
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
  return append_text_cell(a, what, t);
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
  if (col < 0 || col >= (int32_t)a->type_ids.size() || a->type_ids[(size_t)col] != DMB_TYPE_DECIMAL || width < 1 || width > 38 || scale < 0 || scale > width) {
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

// the table column's ENUM type (duckdb_enum_dictionary_size / _value, duckdb_enum_internal_type of duckdb_appender_column_type)
extern "C" int32_t duckdb_mb_gpu_appender_set_enum(duckdb_mb_gpu_appender *a, int32_t col, int32_t internal_type_id, const dmb_enum_dict *dict) {
  if (!a) return 0;
  if (col < 0 || col >= (int32_t)a->type_ids.size() || a->type_ids[(size_t)col] != DMB_TYPE_ENUM) return fail(a, "appender_set_enum: column %d is not an ENUM column", col);
  int32_t w;
  uint64_t most;
  switch (internal_type_id) {
    case DMB_TYPE_UTINYINT: w = 1; most = 1ull << 8; break;
    case DMB_TYPE_USMALLINT: w = 2; most = 1ull << 16; break;
    case DMB_TYPE_UINTEGER: w = 4; most = 1ull << 30; break;  // (the lookup table takes 2^31 slots at most)
    default: return fail(a, "appender_set_enum: column %d: internal type %d is not UTINYINT, USMALLINT or UINTEGER", col, internal_type_id);
  }
  if (!dict) return fail(a, "appender_set_enum: column %d: no dictionary", col);
  if ((uint64_t)dict->size > most)
    return fail(a, "appender_set_enum: column %d: %u labels are more than internal type %d can index (%llu)", col, dict->size, internal_type_id,
                (unsigned long long)most);
  if (dict->size && (!dict->offsets || dict->offsets[0] != 0)) return fail(a, "appender_set_enum: column %d: malformed offsets (offsets[0] must be 0)", col);
  for (uint32_t i = 0; i < dict->size; ++i)
    if (dict->offsets[i + 1] < dict->offsets[i]) return fail(a, "appender_set_enum: column %d: malformed offsets (decreasing at label %u)", col, i);
  const uint32_t bytes = dict->size ? dict->offsets[dict->size] : 0;
  if (bytes && !dict->data) return fail(a, "appender_set_enum: column %d: malformed offsets (labels without data)", col);
  EnumDecl e;
  e.width = w;
  e.offsets.assign(dict->offsets ? dict->offsets : nullptr, dict->offsets ? dict->offsets + dict->size + 1 : nullptr);
  if (e.offsets.empty()) e.offsets.push_back(0);
  e.data.assign((const uint8_t *)dict->data, (const uint8_t *)dict->data + bytes);
  EnumDecl &cur = a->enums[(size_t)col];
  if (cur.width) {
    if (cur.width != e.width || cur.offsets != e.offsets || cur.data != e.data)
      return fail(a, "appender_set_enum: column %d already has a different ENUM declaration", col);
    return 1;
  }
  e.table_size = 16;
  while (e.table_size < 2 * (uint64_t)dict->size) e.table_size *= 2;
  e.slots.resize(2 * (size_t)e.table_size);
  const dmb_enum_dict copy{dict->size, 0, e.offsets.data(), (const char *)e.data.data()};
  if (!dmb_rev_enum_table(&copy, e.table_size, e.slots.data())) return fail(a, "appender_set_enum: column %d: %s", col, duckdb_mb_gpu_last_error());
  cur = std::move(e);
  a->rows[(size_t)col].width = 0;  // the row protocol buffers VARCHAR labels
  return 1;
}

// the table's field types of a STRUCT column (duckdb_struct_type_child_count / _child_type), or of a STRUCT field column:
// they become field columns, numbered from the current column count on
extern "C" int32_t duckdb_mb_gpu_appender_set_struct(duckdb_mb_gpu_appender *a, int32_t col, int32_t nfields, const int32_t *field_type_ids,
                                                     int32_t *first_field) {
  if (!a) return 0;
  if (col < 0 || col >= (int32_t)a->type_ids.size() || a->type_ids[(size_t)col] != DMB_TYPE_STRUCT)
    return fail(a, "appender_set_struct: column %d is not a STRUCT column", col);
  if (nfields <= 0 || !field_type_ids) return fail(a, "appender_set_struct: column %d: a STRUCT needs at least one field", col);
  for (int32_t f = 0; f < nfields; ++f) {
    const int32_t t = field_type_ids[f];
    switch (t) {
      case DMB_TYPE_LIST: return fail(a, "appender_set_struct: column %d, field %d: LIST fields cannot be appended", col, f);
      case DMB_TYPE_MAP: return fail(a, "appender_set_struct: column %d, field %d: MAP fields cannot be appended", col, f);
      case DMB_TYPE_BOOLEAN: case DMB_TYPE_TINYINT: case DMB_TYPE_SMALLINT: case DMB_TYPE_INTEGER: case DMB_TYPE_BIGINT:
      case DMB_TYPE_UTINYINT: case DMB_TYPE_USMALLINT: case DMB_TYPE_UINTEGER: case DMB_TYPE_UBIGINT: case DMB_TYPE_FLOAT:
      case DMB_TYPE_DOUBLE: case DMB_TYPE_DATE: case DMB_TYPE_TIME: case DMB_TYPE_TIME_NS: case DMB_TYPE_TIME_TZ:
      case DMB_TYPE_TIMESTAMP: case DMB_TYPE_TIMESTAMP_S: case DMB_TYPE_TIMESTAMP_MS: case DMB_TYPE_TIMESTAMP_NS:
      case DMB_TYPE_TIMESTAMP_TZ: case DMB_TYPE_HUGEINT: case DMB_TYPE_UHUGEINT: case DMB_TYPE_UUID: case DMB_TYPE_VARCHAR:
      case DMB_TYPE_BLOB: case DMB_TYPE_DECIMAL: case DMB_TYPE_ENUM: case DMB_TYPE_STRUCT:
        break;
      default:  // the types map_column converts, and nothing else
        return fail(a, "appender_set_struct: column %d, field %d: field type %d cannot be appended", col, f, t);
    }
  }
  StructDecl &d = a->structs[(size_t)col];
  if (d.first >= 0) {
    if (d.types != std::vector<int32_t>(field_type_ids, field_type_ids + nfields))
      return fail(a, "appender_set_struct: column %d already has a different STRUCT declaration (%d fields)", col, (int)d.types.size());
    if (first_field) *first_field = d.first;
    return 1;
  }
  const int32_t first = (int32_t)a->type_ids.size();
  d.first = first;
  d.types.assign(field_type_ids, field_type_ids + nfields);
  for (int32_t f = 0; f < nfields; ++f) {
    a->type_ids.push_back(field_type_ids[f]);
    a->parent.push_back(col);
    a->field_index.push_back(f);
    RowBuf rb;
    rb.width = row_width(field_type_ids[f]);
    rb.offsets.assign(1, 0);
    a->rows.push_back(std::move(rb));
    a->lists.emplace_back();
    a->enums.emplace_back();
    a->structs.emplace_back();  // (moves `d`)
  }
  if (first_field) *first_field = first;
  return 1;
}

// during a sink call: field `field` of STRUCT column `col` for the chunk being handed over
extern "C" int32_t duckdb_mb_gpu_appender_struct_field(duckdb_mb_gpu_appender *a, int32_t col, int32_t field, const void **data,
                                                       const uint64_t **validity) {
  if (!a || !data || !validity) return 0;
  if (a->sink_chunk < 0 || col < 0 || (size_t)col >= a->sink_cols.size() || a->type_ids[(size_t)col] != DMB_TYPE_STRUCT)
    return fail(a, "appender_struct_field: column %d is not a STRUCT column of a chunk being handed to the sink", col);
  const StructDecl &d = a->structs[(size_t)col];
  if (field < 0 || field >= (int32_t)d.types.size()) return fail(a, "appender_struct_field: column %d has no field %d", col, field);
  const SinkCol &f = a->sink_cols[(size_t)(d.first + field)];
  const int64_t k = a->sink_chunk;
  *data = f.data ? f.data + (size_t)k * DMB_VECTOR_SIZE * (size_t)f.w : nullptr;
  *validity = f.masks + (size_t)k * DMB_VALIDITY_WORDS;
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
