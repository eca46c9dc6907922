/*
 * oracle.c — CPU restatement of the reference's result/ingest boundary.  TEST INFRASTRUCTURE ONLY.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
 * load this file.  The product path (libduckdb_mb_gpu.so) never links or calls it.
 *
 * PARITY PINNING.  The reference itself (MoonBit native + libduckdb) cannot be built in this image
 * (no moon, no moonbit.h, no libduckdb; SURVEY.md §8c), so there is no oracle/_ref.  The oracle is
 * pinned against the reference's own golden vectors re-expressed as chunk inputs:
 *   src/duckdb_arrow_test.mbt:210-518, src/duckdb_fixture_cases.mbt:4-262,
 *   src/duckdb_test.mbt:1031-1316, src/pbt_generated_test.mbt:178-280   (tests/test_oracle_golden.py)
 * Conversions that run inside un-vendored libduckdb and that no reference test exercises
 * (double->int64 rounding, DECIMAL->int64, text rendering of doubles beyond the fixtures) are
 * "parity unpinned": they follow DuckDB's documented semantics and are marked UNPINNED below.
 *
 * Each function cites the reference lines it follows (paths relative to /root/reference).
 * The per-cell call structure of the reference is kept on purpose: it is what the CPU baseline times.
 */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define ORA_VECTOR_SIZE 2048

enum { /* DUCKDB_TYPE ids, src/duckdb_parsing.mbt:8-52 */
  T_INVALID = 0, T_BOOLEAN = 1, T_TINYINT = 2, T_SMALLINT = 3, T_INTEGER = 4, T_BIGINT = 5,
  T_UTINYINT = 6, T_USMALLINT = 7, T_UINTEGER = 8, T_UBIGINT = 9, T_FLOAT = 10, T_DOUBLE = 11,
  T_TIMESTAMP = 12, T_DATE = 13, T_TIME = 14, T_INTERVAL = 15, T_HUGEINT = 16, T_VARCHAR = 17,
  T_BLOB = 18, T_DECIMAL = 19, T_TIMESTAMP_S = 20, T_TIMESTAMP_MS = 21, T_TIMESTAMP_NS = 22,
  T_UUID = 27, T_TIME_TZ = 30, T_TIMESTAMP_TZ = 31, T_UHUGEINT = 32, T_TIME_NS = 39
};
enum { P_BOOL, P_I8, P_I16, P_I32, P_I64, P_U8, P_U16, P_U32, P_U64, P_F32, P_F64, P_I128, P_U128, P_INTERVAL, P_STRING };
static const int PHYS_W[] = {1, 1, 2, 4, 8, 1, 2, 4, 8, 4, 8, 16, 16, 16, 16};

typedef struct {
  int32_t type_id, phys, dec_width, dec_scale;
  const uint8_t *data;      /* column slab */
  const uint64_t *data_off; /* [nchunks] */
  const uint64_t *validity; /* slab or NULL */
  const int64_t *val_off;   /* [nchunks], -1 = NULL pointer */
  const char *name;
  /* ENUM (type 23): the type's dictionary as duckdb_enum_dictionary_value returns it, packed:
   * label i = dict_data[dict_offsets[i] .. dict_offsets[i+1]); vectors hold uint8/16/32 indices */
  const uint32_t *dict_offsets;
  const char *dict_data;
  uint32_t dict_size;
} ora_column;

typedef struct {
  int64_t nchunks;
  const uint32_t *counts;
  int32_t ncols;
  const ora_column *cols;
} ora_batch;

typedef struct { /* duckdb_string_t, read like src/duckdb_native.c:597-603 */
  uint32_t length;
  char rest[12]; /* inlined[12]  |  prefix[4] + ptr */
} ora_string_t;

/* stand-in for the reference's handle {duckdb_result, column_count, row_count}
 * (src/duckdb_native.c:2211-2217) plus what libduckdb's deprecated value API materialises on the
 * first duckdb_value_* call: row-addressable column arrays with a bool nullmask (external
 * knowledge of duckdb_translate_result; the work is part of what the reference pays). */
typedef struct {
  ora_batch batch;
  int64_t *row_off;
  int64_t nrows;
  int32_t column_count, row_count; /* (int32_t) casts, :2264-2265 */
  uint8_t **dep_data;              /* per column contiguous payload (strings: char* array) */
  uint8_t **dep_null;              /* per column bool nullmask */
  int materialised;
} ora_result;

/* ------------------------------------------------------------------ chunk accessors */
static inline const uint8_t *vec_data(const ora_column *c, int64_t k) { return c->data + c->data_off[k]; }

/* duckdb_mb_chunk_is_null, src/duckdb_native.c:520-535: NULL validity => valid, else bit test */
static inline int chunk_is_null(const ora_column *c, int64_t k, int32_t row) {
  if (c->val_off[k] < 0) return 0;
  const uint64_t *validity = c->validity + c->val_off[k];
  return ((validity[row / 64] >> (row % 64)) & 1ull) ? 0 : 1;
}

static inline const char *string_t_data(const ora_string_t *s) { /* duckdb_string_t_data */
  if (s->length <= 12) return s->rest;
  const char *p;
  memcpy(&p, s->rest + 4, sizeof(p));
  return p;
}

ora_result *ora_result_create(const ora_batch *b) {
  ora_result *r = (ora_result *)calloc(1, sizeof(ora_result));
  r->batch = *b;
  r->row_off = (int64_t *)malloc(sizeof(int64_t) * (size_t)(b->nchunks + 1));
  int64_t acc = 0;
  for (int64_t k = 0; k < b->nchunks; k++) { r->row_off[k] = acc; acc += b->counts[k]; }
  r->row_off[b->nchunks] = acc;
  r->nrows = acc;
  r->column_count = b->ncols;
  r->row_count = (int32_t)acc;
  r->dep_data = (uint8_t **)calloc((size_t)(b->ncols > 0 ? b->ncols : 1), sizeof(uint8_t *));
  r->dep_null = (uint8_t **)calloc((size_t)(b->ncols > 0 ? b->ncols : 1), sizeof(uint8_t *));
  return r;
}

static void ora_free_dep(ora_result *r) {
  for (int32_t c = 0; c < r->batch.ncols; c++) {
    if (r->dep_data[c] && r->batch.cols[c].phys == P_STRING) {
      char **arr = (char **)r->dep_data[c];
      for (int64_t i = 0; i < r->nrows; i++) free(arr[i]);
    }
    free(r->dep_data[c]); r->dep_data[c] = NULL;
    free(r->dep_null[c]); r->dep_null[c] = NULL;
  }
  r->materialised = 0;
}

void ora_result_destroy(ora_result *r) {
  if (!r) return;
  ora_free_dep(r);
  free(r->dep_data); free(r->dep_null); free(r->row_off); free(r);
}

int64_t ora_result_rows(ora_result *r) { return r ? r->nrows : 0; }

/* what libduckdb does on the first deprecated duckdb_value_* call */
static void ora_materialise(ora_result *r) {
  if (r->materialised) return;
  const ora_batch *b = &r->batch;
  for (int32_t c = 0; c < b->ncols; c++) {
    const ora_column *col = &b->cols[c];
    int w = PHYS_W[col->phys];
    size_t n = (size_t)(r->nrows > 0 ? r->nrows : 1);
    r->dep_null[c] = (uint8_t *)malloc(n);
    if (col->phys == P_STRING) {
      char **arr = (char **)calloc(n, sizeof(char *));
      r->dep_data[c] = (uint8_t *)arr;
      for (int64_t k = 0; k < b->nchunks; k++) {
        const ora_string_t *v = (const ora_string_t *)vec_data(col, k);
        for (uint32_t i = 0; i < b->counts[k]; i++) {
          int64_t row = r->row_off[k] + i;
          int isnull = chunk_is_null(col, k, (int32_t)i);
          r->dep_null[c][row] = (uint8_t)isnull;
          if (!isnull) {
            uint32_t len = v[i].length;
            char *s = (char *)malloc((size_t)len + 1);
            memcpy(s, string_t_data(&v[i]), len);
            s[len] = '\0';
            arr[row] = s;
          }
        }
      }
    } else {
      r->dep_data[c] = (uint8_t *)malloc(n * (size_t)w);
      for (int64_t k = 0; k < b->nchunks; k++) {
        const uint8_t *v = vec_data(col, k);
        for (uint32_t i = 0; i < b->counts[k]; i++) {
          int64_t row = r->row_off[k] + i;
          r->dep_null[c][row] = (uint8_t)chunk_is_null(col, k, (int32_t)i);
          memcpy(r->dep_data[c] + (size_t)row * (size_t)w, v + (size_t)i * (size_t)w, (size_t)w);
        }
      }
    }
  }
  r->materialised = 1;
}

/* ------------------------------------------------------------------ duckdb_value_* stand-ins
 * (libduckdb, un-vendored.  Call sites: src/duckdb_native.c:2380,2384,2414,2417,2446,2449,2475,
 * 2478,2538,2541.)  Same-family casts are pinned by src/duckdb_arrow_test.mbt; the rest UNPINNED. */
typedef struct { uint64_t lo; int64_t hi; } ora_hugeint;
int ora_render_cell(const ora_column *c, const uint8_t *p, char *out);
int ora_render_time(int64_t v, int64_t unit_per_sec, char *out);
int ora_render_uuid(const uint8_t *p, char *out);
int ora_render_time_tz(uint64_t bits, char *out);
int ora_render_interval(int32_t months, int32_t days, int64_t micros, char *out);
int ora_render_decimal128(unsigned __int128 u, int is_signed, int scale, char *out);

__attribute__((noinline)) int ora_value_is_null(ora_result *r, int32_t col, int64_t row) {
  if (!r->materialised) ora_materialise(r);
  if (col < 0 || col >= r->column_count || row < 0 || row >= r->nrows) return 0;
  return r->dep_null[col][row];
}

static int64_t double_to_i64(double v) { /* UNPINNED: DuckDB TryCast double->int64, nearbyint */
  if (!(v >= -9223372036854775808.0 && v < 9223372036854775808.0)) return 0;
  return (int64_t)nearbyint(v);
}

/* libduckdb casts a cell by the column's LOGICAL type (GetInternalCValue switches on the deprecated column type):
 * integers / floats / HUGEINT / UHUGEINT by TryCast (failure -> 0), DECIMAL by TryCastFromDecimal (the stored integer
 * divided by 10^scale), and DATE / TIME* / TIMESTAMP* / INTERVAL / UUID / ENUM have no cast to a number (TryCast throws,
 * the C API catches and returns 0).  VARCHAR -> number parses the text in libduckdb; not restated: 0.  UNPINNED except
 * the same-family integer / double / boolean reads (src/duckdb_arrow_test.mbt). */
static int numeric_castable(const ora_column *c) {
  switch (c->type_id) {
    case T_BOOLEAN: case T_TINYINT: case T_SMALLINT: case T_INTEGER: case T_BIGINT: case T_UTINYINT: case T_USMALLINT:
    case T_UINTEGER: case T_UBIGINT: case T_FLOAT: case T_DOUBLE: case T_HUGEINT: case T_UHUGEINT: case T_DECIMAL:
      return 1;
    default: return 0;
  }
}

/* DuckDB Hugeint::TryCast<double> (CastBigintToFloating) */
static double hugeint_to_double(uint64_t lo, int64_t hi) {
  if (hi == -1) return -(double)(0xffffffffffffffffull - lo) - 1.0;
  return (double)lo + (double)hi * 18446744073709551616.0;
}
static double int128_to_double(__int128 x) { return hugeint_to_double((uint64_t)x, (int64_t)(x >> 64)); }

static const double DOUBLE_POW10[39] = {
    1e0,  1e1,  1e2,  1e3,  1e4,  1e5,  1e6,  1e7,  1e8,  1e9,  1e10, 1e11, 1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19,
    1e20, 1e21, 1e22, 1e23, 1e24, 1e25, 1e26, 1e27, 1e28, 1e29, 1e30, 1e31, 1e32, 1e33, 1e34, 1e35, 1e36, 1e37, 1e38};
static __int128 pow10_i128(int scale) {
  __int128 p = 1;
  for (int k = 0; k < scale && k < 38; k++) p *= 10;
  return p;
}
static __int128 decimal_stored(const ora_column *c, const uint8_t *p) {
  switch (c->phys) {
    case P_I16: { int16_t v; memcpy(&v, p, 2); return v; }
    case P_I32: { int32_t v; memcpy(&v, p, 4); return v; }
    case P_I64: { int64_t v; memcpy(&v, p, 8); return v; }
    default: { ora_hugeint v; memcpy(&v, p, 16); return ((__int128)v.hi << 64) | (__int128)(unsigned __int128)v.lo; }
  }
}
/* TryCastFromDecimal -> integer: round half away from zero, truncating division; out of range -> the cast fails -> 0 */
static int64_t decimal_to_i64(const ora_column *c, const uint8_t *p) {
  __int128 power = pow10_i128(c->dec_scale), x = decimal_stored(c, p);
  __int128 rounding = (x < 0 ? -power : power) / 2;
  __int128 q = (x + rounding) / power;
  return (q >= -(__int128)9223372036854775807ll - 1 && q <= (__int128)9223372036854775807ll) ? (int64_t)q : 0;
}
/* TryCastDecimalToFloatingPoint: exact integers (|x| <= 2^53) or scale 0 divide directly, the rest split in two */
static double decimal_to_double(const ora_column *c, const uint8_t *p) {
  __int128 x = decimal_stored(c, p);
  int scale = c->dec_scale < 0 ? 0 : (c->dec_scale > 38 ? 38 : c->dec_scale);
  double dp = DOUBLE_POW10[scale];
  if (scale == 0 || (x <= (__int128)9007199254740992ll && x >= -(__int128)9007199254740992ll)) return int128_to_double(x) / dp;
  __int128 power = pow10_i128(scale);
  return int128_to_double(x / power) + int128_to_double(x % power) / dp;
}

__attribute__((noinline)) int64_t ora_value_int64(ora_result *r, int32_t col, int64_t row) {
  if (!r->materialised) ora_materialise(r);
  if (col < 0 || col >= r->column_count || row < 0 || row >= r->nrows) return 0;
  if (r->dep_null[col][row]) return 0;
  const ora_column *c = &r->batch.cols[col];
  const uint8_t *p = r->dep_data[col] + (size_t)row * (size_t)PHYS_W[c->phys];
  if (!numeric_castable(c)) return 0;
  if (c->type_id == T_DECIMAL) return decimal_to_i64(c, p); /* UNPINNED */
  switch (c->phys) {
    case P_BOOL: return *(const uint8_t *)p ? 1 : 0;
    case P_I8: return *(const int8_t *)p;
    case P_I16: { int16_t v; memcpy(&v, p, 2); return v; }
    case P_I32: { int32_t v; memcpy(&v, p, 4); return v; }
    case P_I64: { int64_t v; memcpy(&v, p, 8); return v; }
    case P_U8: return *(const uint8_t *)p;
    case P_U16: { uint16_t v; memcpy(&v, p, 2); return v; }
    case P_U32: { uint32_t v; memcpy(&v, p, 4); return v; }
    case P_U64: { uint64_t v; memcpy(&v, p, 8); return v > 0x7fffffffffffffffull ? 0 : (int64_t)v; } /* UNPINNED */
    case P_F32: { float v; memcpy(&v, p, 4); return double_to_i64((double)v); }                      /* UNPINNED */
    case P_F64: { double v; memcpy(&v, p, 8); return double_to_i64(v); }                             /* UNPINNED */
    case P_I128: { ora_hugeint v; memcpy(&v, p, 16);                                                 /* UNPINNED */
      int fits = (v.hi == 0 && (int64_t)v.lo >= 0) || (v.hi == -1 && (int64_t)v.lo < 0);
      return fits ? (int64_t)v.lo : 0; }
    case P_U128: { ora_hugeint v; memcpy(&v, p, 16);                                                 /* UNPINNED: UHUGEINT */
      return (v.hi == 0 && v.lo <= 0x7fffffffffffffffull) ? (int64_t)v.lo : 0; }
    default: return 0;
  }
}

__attribute__((noinline)) double ora_value_double(ora_result *r, int32_t col, int64_t row) {
  if (!r->materialised) ora_materialise(r);
  if (col < 0 || col >= r->column_count || row < 0 || row >= r->nrows) return 0.0;
  if (r->dep_null[col][row]) return 0.0;
  const ora_column *c = &r->batch.cols[col];
  const uint8_t *p = r->dep_data[col] + (size_t)row * (size_t)PHYS_W[c->phys];
  if (!numeric_castable(c)) return 0.0;
  if (c->type_id == T_DECIMAL) return decimal_to_double(c, p); /* UNPINNED */
  switch (c->phys) {
    case P_F64: { double v; memcpy(&v, p, 8); return v; }
    case P_F32: { float v; memcpy(&v, p, 4); return (double)v; }
    case P_U64: { uint64_t v; memcpy(&v, p, 8); return (double)v; }
    case P_I128: { ora_hugeint v; memcpy(&v, p, 16); return hugeint_to_double(v.lo, v.hi); }          /* UNPINNED: what SUM() returns */
    case P_U128: { ora_hugeint v; memcpy(&v, p, 16); return (double)v.lo + (double)(uint64_t)v.hi * 18446744073709551616.0; }
    default: return (double)ora_value_int64(r, col, row);
  }
}

__attribute__((noinline)) int ora_value_boolean(ora_result *r, int32_t col, int64_t row) {
  if (!r->materialised) ora_materialise(r);
  if (col < 0 || col >= r->column_count || row < 0 || row >= r->nrows) return 0;
  if (r->dep_null[col][row]) return 0;
  const ora_column *c = &r->batch.cols[col];
  if (!numeric_castable(c)) return 0;
  if (c->type_id == T_DECIMAL) return ora_value_int64(r, col, row) != 0; /* TryCastDecimalToNumeric<.., bool>: the rounded integer */
  if (c->phys == P_F32 || c->phys == P_F64) return ora_value_double(r, col, row) != 0.0;
  if (c->phys == P_U64) { uint64_t u; memcpy(&u, r->dep_data[col] + (size_t)row * 8, 8); return u != 0; }
  if (c->phys == P_I128 || c->phys == P_U128) { ora_hugeint v; memcpy(&v, r->dep_data[col] + (size_t)row * 16, 16); return (v.lo | (uint64_t)v.hi) != 0; }
  return ora_value_int64(r, col, row) != 0;
}

/* duckdb_value_varchar: a malloc'ed NUL-terminated copy the caller frees with duckdb_free */
__attribute__((noinline)) char *ora_value_varchar(ora_result *r, int32_t col, int64_t row) {
  if (!r->materialised) ora_materialise(r);
  if (col < 0 || col >= r->column_count || row < 0 || row >= r->nrows) return NULL;
  if (r->dep_null[col][row]) return NULL;
  const ora_column *c = &r->batch.cols[col];
  if (c->phys == P_STRING && c->type_id == T_BLOB) {
    /* duckdb_value_varchar of a BLOB cell is its VARCHAR cast, DuckDB Blob::ToString: printable ASCII except backslash and
     * the quote characters as it is, every other byte as \xHH (upper-case hex).  The bytes come from the chunk vector (the
     * deprecated column keeps {data, size}, so embedded NULs survive).  UNPINNED: no reference test reads a BLOB as text. */
    int64_t k = 0;
    while (k + 1 < r->batch.nchunks && r->row_off[k + 1] <= row) k++;
    const ora_string_t *e = (const ora_string_t *)vec_data(c, k) + (row - r->row_off[k]);
    const uint8_t *src = (const uint8_t *)string_t_data(e);
    char *out = (char *)malloc((size_t)e->length * 4 + 1);
    size_t n = 0;
    for (uint32_t i = 0; i < e->length; i++) {
      uint8_t ch = src[i];
      if (ch >= 32 && ch <= 126 && ch != '\\' && ch != '\'' && ch != '"') out[n++] = (char)ch;
      else { static const char hex[] = "0123456789ABCDEF"; out[n++] = '\\'; out[n++] = 'x'; out[n++] = hex[ch >> 4]; out[n++] = hex[ch & 15]; }
    }
    out[n] = 0;
    return out;
  }
  if (c->phys == P_STRING) {
    const char *s = ((char **)r->dep_data[col])[row];
    /* the deprecated column keeps a C string, so the copy stops at the first NUL */
    size_t len = strlen(s);
    char *out = (char *)malloc(len + 1);
    memcpy(out, s, len + 1);
    return out;
  }
  if (c->type_id == 23) {
    /* ENUM: the cell's VARCHAR cast is its dictionary label; the reference keeps it as Value::String
     * (src/duckdb_parsing.mbt:119-122).  UNPINNED: no reference test or fixture holds an ENUM column. */
    const uint8_t *p = r->dep_data[col] + (size_t)row * (size_t)PHYS_W[c->phys];
    uint32_t idx = 0;
    memcpy(&idx, p, (size_t)PHYS_W[c->phys]); /* little endian: uint8 / uint16 / uint32 */
    if (!c->dict_offsets || idx >= c->dict_size) return NULL;
    size_t len = c->dict_offsets[idx + 1] - c->dict_offsets[idx];
    char *out = (char *)malloc(len + 1);
    memcpy(out, c->dict_data + c->dict_offsets[idx], len);
    out[len] = 0;
    return out;
  }
  char buf[96];
  /* DuckDB's VARCHAR cast of the cell (ora_render_cell below; formats pinned by the fixture strings) */
  if (ora_render_cell(c, r->dep_data[col] + (size_t)row * (size_t)PHYS_W[c->phys], buf) < 0) return NULL;
  size_t len = strlen(buf);
  char *out = (char *)malloc(len + 1);
  memcpy(out, buf, len + 1);
  return out;
}

/* ------------------------------------------------------------------ packed getters
 * Returned blob stands for the MoonBit Bytes; *out_len is its length. */
static uint8_t *make_bytes(int64_t len, int64_t *out_len) {
  *out_len = len;
  return (uint8_t *)malloc((size_t)(len > 0 ? len : 1));
}

/* src/duckdb_native.c:2359-2390 */
uint8_t *ora_arrow_get_column_int32(ora_result *r, int32_t col_idx, int64_t *out_len) {
  if (!r) return make_bytes(0, out_len);
  int32_t row_count = r->row_count;
  if (col_idx < 0 || col_idx >= r->column_count || row_count <= 0) return make_bytes(0, out_len);
  int32_t total_size = 4 + row_count * 4;
  uint8_t *result = make_bytes(total_size, out_len);
  int32_t *out = (int32_t *)result;
  out[0] = row_count;
  for (int32_t i = 0; i < row_count; i++) {
    if (ora_value_is_null(r, col_idx, i)) {
      out[i + 1] = 0;
    } else {
      int64_t val = ora_value_int64(r, col_idx, i);
      out[i + 1] = (int32_t)val;
    }
  }
  return result;
}

/* src/duckdb_native.c:2392-2422 (values start at byte 4: 4-byte aligned only) */
uint8_t *ora_arrow_get_column_int64(ora_result *r, int32_t col_idx, int64_t *out_len) {
  if (!r) return make_bytes(0, out_len);
  int32_t row_count = r->row_count;
  if (col_idx < 0 || col_idx >= r->column_count || row_count <= 0) return make_bytes(0, out_len);
  int32_t total_size = 4 + row_count * 8;
  uint8_t *result = make_bytes(total_size, out_len);
  ((int32_t *)result)[0] = row_count;
  uint8_t *out_data = result + 4;
  for (int32_t i = 0; i < row_count; i++) {
    int64_t v = ora_value_is_null(r, col_idx, i) ? 0 : ora_value_int64(r, col_idx, i);
    memcpy(out_data + (size_t)i * 8, &v, 8);
  }
  return result;
}

/* src/duckdb_native.c:2424-2454 */
uint8_t *ora_arrow_get_column_double(ora_result *r, int32_t col_idx, int64_t *out_len) {
  if (!r) return make_bytes(0, out_len);
  int32_t row_count = r->row_count;
  if (col_idx < 0 || col_idx >= r->column_count || row_count <= 0) return make_bytes(0, out_len);
  int32_t total_size = 4 + row_count * 8;
  uint8_t *result = make_bytes(total_size, out_len);
  ((int32_t *)result)[0] = row_count;
  uint8_t *out_data = result + 4;
  for (int32_t i = 0; i < row_count; i++) {
    double v = ora_value_is_null(r, col_idx, i) ? 0.0 : ora_value_double(r, col_idx, i);
    memcpy(out_data + (size_t)i * 8, &v, 8);
  }
  return result;
}

/* src/duckdb_native.c:2516-2546 */
uint8_t *ora_arrow_get_column_bool(ora_result *r, int32_t col_idx, int64_t *out_len) {
  if (!r) return make_bytes(0, out_len);
  int32_t row_count = r->row_count;
  if (col_idx < 0 || col_idx >= r->column_count || row_count <= 0) return make_bytes(0, out_len);
  int32_t total_size = 4 + row_count;
  uint8_t *result = make_bytes(total_size, out_len);
  ((int32_t *)result)[0] = row_count;
  uint8_t *out_data = result + 4;
  for (int32_t i = 0; i < row_count; i++) {
    if (ora_value_is_null(r, col_idx, i)) out_data[i] = 0;
    else out_data[i] = ora_value_boolean(r, col_idx, i) ? 1 : 0;
  }
  return result;
}

/* Shared body of src/duckdb_native.c:2456-2514 and :2687-2759.
 * Faithful to a defect of the reference: pass 1 adds nothing to total_data_len for a NULL row
 * (:2475-2476) but pass 2 still writes a '\0' for it (:2508-2510), so the stream is
 * total_data_len + null_count bytes long.  In the nullable getter the surplus lands in (and is then
 * overwritten by) the validity bytes (:2745-2755); in the plain getter it runs past the allocation
 * (undefined behaviour) — the in-bounds part, the first total_data_len bytes, is what we keep. */
static uint8_t *string_getter(ora_result *r, int32_t col_idx, int nullable, int64_t *out_len) {
  if (!r) return make_bytes(0, out_len);
  int32_t row_count = r->row_count;
  if (col_idx < 0 || col_idx >= r->column_count || row_count <= 0) return make_bytes(0, out_len);
  size_t total_data_len = 0;
  char **strings = (char **)malloc((size_t)row_count * sizeof(char *));
  if (!strings) return make_bytes(0, out_len);
  size_t null_rows = 0;
  for (int32_t i = 0; i < row_count; i++) {
    if (ora_value_is_null(r, col_idx, i)) {
      strings[i] = NULL;
      null_rows++;
    } else {
      strings[i] = ora_value_varchar(r, col_idx, i);
      if (strings[i]) total_data_len += strlen(strings[i]) + 1;
      else total_data_len += 1;
    }
  }
  int32_t total_size = 4 + 4 + (int32_t)total_data_len + (nullable ? row_count : 0);
  uint8_t *result = make_bytes(total_size, out_len);
  int32_t *out_header = (int32_t *)result;
  out_header[0] = row_count;
  out_header[1] = (int32_t)total_data_len;
  /* the reference writes the whole stream in place; emulate with a scratch stream and keep
   * what stays inside the allocation */
  uint8_t *stream = (uint8_t *)malloc(total_data_len + null_rows + 1);
  size_t out_pos = 0;
  for (int32_t i = 0; i < row_count; i++) {
    if (strings[i]) {
      size_t len = strlen(strings[i]);
      memcpy(stream + out_pos, strings[i], len);
      out_pos += len;
      stream[out_pos++] = '\0';
      free(strings[i]);
    } else {
      stream[out_pos++] = '\0';
    }
  }
  size_t room = (size_t)total_size - 8;
  memcpy(result + 8, stream, out_pos < room ? out_pos : room);
  free(stream);
  if (nullable) {
    uint8_t *validity_out = result + 8 + total_data_len;
    for (int32_t i = 0; i < row_count; i++) validity_out[i] = ora_value_is_null(r, col_idx, i) ? 0 : 1;
  }
  free(strings);
  return result;
}
uint8_t *ora_arrow_get_column_string(ora_result *r, int32_t col, int64_t *out_len) { return string_getter(r, col, 0, out_len); }
uint8_t *ora_arrow_get_column_string_nullable(ora_result *r, int32_t col, int64_t *out_len) { return string_getter(r, col, 1, out_len); }

/* src/duckdb_native.c:2572-2609 */
uint8_t *ora_arrow_get_column_int32_nullable(ora_result *r, int32_t col_idx, int64_t *out_len) {
  if (!r) return make_bytes(0, out_len);
  int32_t row_count = r->row_count;
  if (col_idx < 0 || col_idx >= r->column_count || row_count <= 0) return make_bytes(0, out_len);
  int32_t total_size = 4 + row_count * 4 + row_count;
  uint8_t *result = make_bytes(total_size, out_len);
  int32_t *out = (int32_t *)result;
  out[0] = row_count;
  int32_t *values_out = out + 1;
  uint8_t *validity_out = result + 4 + (size_t)row_count * 4;
  for (int32_t i = 0; i < row_count; i++) {
    if (ora_value_is_null(r, col_idx, i)) {
      values_out[i] = 0;
      validity_out[i] = 0;
    } else {
      int64_t val = ora_value_int64(r, col_idx, i);
      values_out[i] = (int32_t)val;
      validity_out[i] = 1;
    }
  }
  return result;
}

/* src/duckdb_native.c:2611-2647 */
uint8_t *ora_arrow_get_column_int64_nullable(ora_result *r, int32_t col_idx, int64_t *out_len) {
  if (!r) return make_bytes(0, out_len);
  int32_t row_count = r->row_count;
  if (col_idx < 0 || col_idx >= r->column_count || row_count <= 0) return make_bytes(0, out_len);
  int32_t total_size = 4 + row_count * 8 + row_count;
  uint8_t *result = make_bytes(total_size, out_len);
  ((int32_t *)result)[0] = row_count;
  uint8_t *values_out = result + 4;
  uint8_t *validity_out = result + 4 + (size_t)row_count * 8;
  for (int32_t i = 0; i < row_count; i++) {
    int64_t v = 0;
    if (ora_value_is_null(r, col_idx, i)) validity_out[i] = 0;
    else { v = ora_value_int64(r, col_idx, i); validity_out[i] = 1; }
    memcpy(values_out + (size_t)i * 8, &v, 8);
  }
  return result;
}

/* src/duckdb_native.c:2649-2685 */
uint8_t *ora_arrow_get_column_double_nullable(ora_result *r, int32_t col_idx, int64_t *out_len) {
  if (!r) return make_bytes(0, out_len);
  int32_t row_count = r->row_count;
  if (col_idx < 0 || col_idx >= r->column_count || row_count <= 0) return make_bytes(0, out_len);
  int32_t total_size = 4 + row_count * 8 + row_count;
  uint8_t *result = make_bytes(total_size, out_len);
  ((int32_t *)result)[0] = row_count;
  uint8_t *values_out = result + 4;
  uint8_t *validity_out = result + 4 + (size_t)row_count * 8;
  for (int32_t i = 0; i < row_count; i++) {
    double v = 0.0;
    if (ora_value_is_null(r, col_idx, i)) validity_out[i] = 0;
    else { v = ora_value_double(r, col_idx, i); validity_out[i] = 1; }
    memcpy(values_out + (size_t)i * 8, &v, 8);
  }
  return result;
}

/* src/duckdb_native.c:2761-2797 */
uint8_t *ora_arrow_get_column_bool_nullable(ora_result *r, int32_t col_idx, int64_t *out_len) {
  if (!r) return make_bytes(0, out_len);
  int32_t row_count = r->row_count;
  if (col_idx < 0 || col_idx >= r->column_count || row_count <= 0) return make_bytes(0, out_len);
  int32_t total_size = 4 + row_count + row_count;
  uint8_t *result = make_bytes(total_size, out_len);
  ((int32_t *)result)[0] = row_count;
  uint8_t *values_out = result + 4;
  uint8_t *validity_out = values_out + row_count;
  for (int32_t i = 0; i < row_count; i++) {
    if (ora_value_is_null(r, col_idx, i)) { values_out[i] = 0; validity_out[i] = 0; }
    else { values_out[i] = ora_value_boolean(r, col_idx, i) ? 1 : 0; validity_out[i] = 1; }
  }
  return result;
}

void ora_free(void *p) { free(p); }

/* src/duckdb_native.c:2285-2355 (type map :2314-2339; names not escaped, nullable always true) */
uint8_t *ora_arrow_schema(ora_result *r, int64_t *out_len) {
  if (!r || r->column_count <= 0) { uint8_t *b = make_bytes(2, out_len); memcpy(b, "[]", 2); return b; }
  int32_t col_count = r->column_count;
  size_t cap = (size_t)col_count * 200 + 10;
  char *json = (char *)malloc(cap);
  size_t pos = 0;
  json[pos++] = '[';
  for (int32_t i = 0; i < col_count; i++) {
    const char *name = r->batch.cols[i].name ? r->batch.cols[i].name : "";
    const char *type_id = "string";
    switch (r->batch.cols[i].type_id) {
      case T_BOOLEAN: type_id = "bool"; break;
      case T_TINYINT: case T_SMALLINT: case T_INTEGER: type_id = "int32"; break;
      case T_BIGINT: type_id = "int64"; break;
      case T_FLOAT: case T_DOUBLE: type_id = "double"; break;
      default: type_id = "string"; break;
    }
    pos += (size_t)snprintf(json + pos, cap - pos, "%s{\"name\":\"%s\",\"nullable\":true,\"type_id\":\"%s\"}",
                            (i == 0) ? "" : ",", name, type_id);
  }
  json[pos++] = ']';
  uint8_t *out = make_bytes((int64_t)pos, out_len);
  memcpy(out, json, pos);
  free(json);
  return out;
}

/* ------------------------------------------------------------------ MoonBit decoder loops
 * src/duckdb_arrow_native.mbt:430-822, restated for the CPU baseline: byte-assembled
 * read_int32_le (:452-462), count cap 1,000,000 (:435), NUL scanning (:559-574). */
static inline int32_t read_int32_le(const uint8_t *data, int64_t len, int64_t offset) {
  if (offset + 4 > len) return 0;
  uint32_t b0 = data[offset], b1 = data[offset + 1], b2 = data[offset + 2], b3 = data[offset + 3];
  return (int32_t)(b0 | (b1 << 8) | (b2 << 16) | (b3 << 24));
}

/* decode_int32_array / decode_int32_nullable_array; returns count decoded (0 = the `[]` result) */
int64_t ora_decode_int32(const uint8_t *data, int64_t len, int nullable, int32_t *values, uint8_t *validity) {
  if (len < 4) return 0;
  int32_t count = read_int32_le(data, len, 0);
  if (count <= 0 || count > 1000000) return 0;
  int64_t expected = 4 + (int64_t)count * 4 + (nullable ? count : 0);
  if (len < expected) return 0;
  int64_t validity_start = 4 + (int64_t)count * 4;
  for (int32_t i = 0; i < count; i++) {
    values[i] = read_int32_le(data, len, 4 + (int64_t)i * 4);
    if (nullable) validity[i] = data[validity_start + i] != 0;
  }
  return count;
}

/* get_column_int64 (:466-505): MoonBit Int is 32-bit on native, shifts >= 32 drop out (Appendix B.1);
 * the value that survives is the low 32 bits. */
int64_t ora_decode_int64_as_int(const uint8_t *data, int64_t len, int nullable, int32_t *values, uint8_t *validity) {
  if (len < 4) return 0;
  int32_t count = read_int32_le(data, len, 0);
  if (count <= 0 || count > 1000000) return 0;
  int64_t expected = 4 + (int64_t)count * 8 + (nullable ? count : 0);
  if (len < expected) return 0;
  int64_t validity_start = 4 + (int64_t)count * 8;
  for (int32_t i = 0; i < count; i++) {
    int64_t base = 4 + (int64_t)i * 8;
    uint32_t b0 = data[base], b1 = data[base + 1], b2 = data[base + 2], b3 = data[base + 3];
    values[i] = (int32_t)(b0 | (b1 << 8) | (b2 << 16) | (b3 << 24));
    if (nullable) validity[i] = data[validity_start + i] != 0;
  }
  return count;
}

/* duckdb_mb_bytes_to_double, src/duckdb_native.c:2561-2565: one FFI call per value (:537-543) */
__attribute__((noinline)) double ora_bytes_to_double(const char *bytes, int32_t offset) {
  double result;
  memcpy(&result, bytes + offset, sizeof(double));
  return result;
}

int64_t ora_decode_double(const uint8_t *data, int64_t len, int nullable, double *values, uint8_t *validity) {
  if (len < 4) return 0;
  int32_t count = read_int32_le(data, len, 0);
  if (count <= 0 || count > 1000000) return 0;
  int64_t expected = 4 + (int64_t)count * 8 + (nullable ? count : 0);
  if (len < expected) return 0;
  int64_t validity_start = 4 + (int64_t)count * 8;
  for (int32_t i = 0; i < count; i++) {
    int64_t base = 4 + (int64_t)i * 8;
    values[i] = (base + 8 > len) ? 0.0 : ora_bytes_to_double((const char *)data, (int32_t)base);
    if (nullable) validity[i] = data[validity_start + i] != 0;
  }
  return count;
}

int64_t ora_decode_bool(const uint8_t *data, int64_t len, int nullable, uint8_t *values, uint8_t *validity) {
  if (len < 4) return 0;
  int32_t count = read_int32_le(data, len, 0);
  if (count <= 0 || count > 1000000) return 0;
  int64_t expected = 4 + (int64_t)count + (nullable ? count : 0);
  if (len < expected) return 0;
  for (int32_t i = 0; i < count; i++) {
    values[i] = data[4 + i] != 0;
    if (nullable) validity[i] = data[4 + count + i] != 0;
  }
  return count;
}

/* get_column_string / decode_string_nullable_array (:546-575, :752-784): NUL scan from byte 8.
 * Writes (start,end) byte positions per string; returns count. */
int64_t ora_decode_string(const uint8_t *data, int64_t len, int nullable, int64_t *starts, int64_t *ends, uint8_t *validity) {
  if (len < 8) return 0;
  int32_t count = read_int32_le(data, len, 0);
  int32_t total_data_len = read_int32_le(data, len, 4);
  if (count <= 0 || count > 1000000) return 0;
  if (nullable && len < 8 + (int64_t)total_data_len + count) return 0;
  int64_t validity_start = 8 + (int64_t)total_data_len;
  int64_t pos = 8;
  for (int32_t i = 0; i < count; i++) {
    int64_t start_pos = pos;
    while (pos < len && data[pos] != 0) pos++;
    if (start_pos < len) { starts[i] = start_pos; ends[i] = pos; }
    else { starts[i] = len; ends[i] = len; }
    pos++;
    if (nullable) validity[i] = data[validity_start + i] != 0;
  }
  return count;
}

/* ------------------------------------------------------------------ Arrow-layout oracle
 * Per-cell restatement on the chunk path: null test src/duckdb_native.c:520-535, payload load
 * :553-662, string_t read :597-603.  Output layouts are the Arrow columnar spec (SURVEY.md
 * Appendix A): LSB validity bitmap, dense little-endian values, NULL slots zero, NULL strings
 * zero-length.  dst kinds mirror enum dmb_dst of include/duckdb_mb_gpu.h. */
enum { D_SAME, D_I32_TRUNC, D_I64, D_F64, D_BOOL_BYTE, D_BOOL_BITS, D_I128, D_I32_SAT,
       D_TS_US_FROM_S, D_TS_US_FROM_MS, D_TS_US_FROM_NS, D_MONTH_DAY_NANO, D_DATE_REF,
       D_DEC_I64 = 17, D_DEC_I32_TRUNC = 18, D_DEC_F64 = 19, D_DEC_BOOL_BYTE = 20 };

static int64_t load_i64(const ora_column *c, const uint8_t *p, int *ok) {
  *ok = 1;
  switch (c->phys) {
    case P_BOOL: return *p ? 1 : 0;
    case P_I8: return *(const int8_t *)p;
    case P_I16: { int16_t v; memcpy(&v, p, 2); return v; }
    case P_I32: { int32_t v; memcpy(&v, p, 4); return v; }
    case P_I64: { int64_t v; memcpy(&v, p, 8); return v; }
    case P_U8: return *p;
    case P_U16: { uint16_t v; memcpy(&v, p, 2); return v; }
    case P_U32: { uint32_t v; memcpy(&v, p, 4); return v; }
    case P_U64: { uint64_t v; memcpy(&v, p, 8); if (v > 0x7fffffffffffffffull) { *ok = 0; return 0; } return (int64_t)v; }
    case P_F32: { float v; memcpy(&v, p, 4); return double_to_i64((double)v); }
    case P_F64: { double v; memcpy(&v, p, 8); return double_to_i64(v); }
    case P_I128: { ora_hugeint v; memcpy(&v, p, 16);
      int fits = (v.hi == 0 && (int64_t)v.lo >= 0) || (v.hi == -1 && (int64_t)v.lo < 0);
      if (!fits) { *ok = 0; return 0; } return (int64_t)v.lo; }
    case P_U128: { ora_hugeint v; memcpy(&v, p, 16);
      if (!(v.hi == 0 && v.lo <= 0x7fffffffffffffffull)) { *ok = 0; return 0; } return (int64_t)v.lo; }
    default: *ok = 0; return 0;
  }
}

static int64_t floor_div64(int64_t a, int64_t b) {
  int64_t q = a / b;
  if ((a % b != 0) && ((a < 0) != (b < 0))) q -= 1;
  return q;
}

/* parse_int, src/duckdb_parsing.mbt:203-237 (Int32-saturating, skips non-digits) */
int32_t ora_parse_int(const char *s, int64_t len) {
  int32_t result = 0;
  int negative = 0;
  int64_t start = 0;
  if (len > 0) {
    if (s[0] == '-') { negative = 1; start = 1; }
    else if (s[0] == '+') start = 1;
  }
  int32_t limit = negative ? INT32_MIN : -INT32_MAX;
  int32_t multmin = limit / 10;
  for (int64_t i = start; i < len; i++) {
    char c = s[i];
    if (c >= '0' && c <= '9') {
      int32_t digit = c - '0';
      if (result < multmin) return negative ? INT32_MIN : INT32_MAX;
      result = result * 10;
      /* next = result - digit; compare without signed overflow */
      if (result < limit + digit) return negative ? INT32_MIN : INT32_MAX;
      result = result - digit;
    }
  }
  return negative ? result : -result;
}

/* parse_fractional + parse_double, src/duckdb_parsing.mbt:241-283 (not correctly rounded) */
double ora_parse_double(const char *s, int64_t len) {
  int64_t dot = -1;
  for (int64_t i = 0; i < len; i++) if (s[i] == '.') { dot = i; break; }
  if (dot < 0) return (double)ora_parse_int(s, len);
  int32_t int_val = ora_parse_int(s, dot);
  double result = 0.0, divisor = 1.0;
  for (int64_t i = dot + 1; i < len; i++) {
    char c = s[i];
    if (c >= '0' && c <= '9') { divisor = divisor * 10.0; result = result + (double)(c - '0') / divisor; }
  }
  double sign = (len > 0 && s[0] == '-') ? -1.0 : 1.0;
  /* int_val.abs(): Int32 abs, MIN stays MIN */
  int32_t a = int_val < 0 ? (int_val == INT32_MIN ? INT32_MIN : -int_val) : int_val;
  return sign * ((double)a + result);
}

static int is_leap(int32_t y) { return (y % 4 == 0 && y % 100 != 0) || y % 400 == 0; }
static int days_in_month(int32_t y, int32_t m) {
  if (m == 2) return is_leap(y) ? 29 : 28;
  if (m == 4 || m == 6 || m == 9 || m == 11) return 30;
  return 31;
}
/* date_to_days, src/duckdb_parsing.mbt:318-338 (leap loop is empty for year < 1970) */
int32_t ora_date_to_days(int32_t year, int32_t month, int32_t day) {
  int32_t y = year - 1970;
  int32_t days = y * 365;
  int32_t leap_years = 0;
  for (int32_t ly = 1970; ly < year; ly++) if (is_leap(ly)) leap_years++;
  days += leap_years;
  for (int32_t m = 1; m < month; m++) days += days_in_month(year, m);
  days += day - 1;
  return days;
}
/* parse_date, src/duckdb_parsing.mbt:293-316; returns 0 and *ok=0 on Err */
int32_t ora_parse_date(const char *s, int64_t len, int *ok) {
  *ok = 0;
  if (!(len == 10 && s[4] == '-' && s[7] == '-')) return 0;
  int32_t year = ora_parse_int(s, 4), month = ora_parse_int(s + 5, 2), day = ora_parse_int(s + 8, 2);
  if (month < 1 || month > 12) return 0;
  if (day < 1 || day > days_in_month(year, month)) return 0;
  *ok = 1;
  return ora_date_to_days(year, month, day);
}
/* parse_fraction_to_micros, src/duckdb_parsing.mbt:402-417 */
static int32_t parse_fraction_to_micros(const char *s, int64_t len) {
  int32_t micros = 0, factor = 100000;
  for (int64_t i = 0; i < len; i++) {
    char c = s[i];
    if (c < '0' || c > '9') break;
    if (factor >= 1) { micros += (c - '0') * factor; factor /= 10; }
  }
  return micros;
}
/* parse_time_to_micros, src/duckdb_parsing.mbt:421-470 */
static int64_t parse_time_to_micros(const char *s, int64_t len, int *ok) {
  int colon_count = 0; int64_t colon1 = -1, colon2 = -1;
  for (int64_t i = 0; i < len; i++) if (s[i] == ':') { if (colon1 < 0) colon1 = i; else colon2 = i; colon_count++; }
  if (colon_count < 2) { *ok = 0; return 0; }
  *ok = 1;
  const char *sec = s + colon2 + 1; int64_t seclen = len - colon2 - 1;
  int64_t dot = -1;
  for (int64_t i = 0; i < seclen; i++) if (sec[i] == '.') { dot = i; break; }
  int32_t second, frac = 0;
  if (dot >= 0) { second = ora_parse_int(sec, dot); frac = parse_fraction_to_micros(sec + dot + 1, seclen - dot - 1); }
  else second = ora_parse_int(sec, seclen);
  int32_t hour = ora_parse_int(s, colon1), minute = ora_parse_int(s + colon1 + 1, colon2 - colon1 - 1);
  return ((int64_t)hour * 3600 + (int64_t)minute * 60 + (int64_t)second) * 1000000 + (int64_t)frac;
}
/* parse_timestamp, src/duckdb_parsing.mbt:375-398 */
int64_t ora_parse_timestamp(const char *s, int64_t len, int *ok) {
  *ok = 0;
  if (!(len >= 19 && s[4] == '-' && s[7] == '-' && s[10] == ' ' && s[13] == ':' && s[16] == ':')) return 0;
  int dok; int32_t days = ora_parse_date(s, 10, &dok);
  if (!dok) return 0;
  int tok; int64_t micros = parse_time_to_micros(s + 11, len - 11, &tok);
  if (!tok) return 0;
  *ok = 1;
  return (int64_t)days * 86400 * 1000000 + micros;
}

/* ---- DuckDB VARCHAR renderings (libduckdb, un-vendored).  Pinned by the fixture strings of
 * src/duckdb_fixture_cases.mbt (ints :27-32,83-102; DATE :41-46; TIMESTAMP :55-60; epoch±1 :62-67;
 * DECIMAL :69-81); anything beyond those shapes is UNPINNED. */
static void civil_from_days(int64_t z, int64_t *y, int *m, int *d) {
  z += 719468;
  int64_t era = (z >= 0 ? z : z - 146096) / 146097;
  int64_t doe = z - era * 146097;
  int64_t yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
  int64_t yy = yoe + era * 400;
  int64_t doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
  int64_t mp = (5 * doy + 2) / 153;
  *d = (int)(doy - (153 * mp + 2) / 5 + 1);
  *m = (int)(mp < 10 ? mp + 3 : mp - 9);
  *y = yy + (*m <= 2);
}
int ora_render_date(int32_t days, char *out) {
  int64_t y; int m, d;
  civil_from_days(days, &y, &m, &d);
  if (y >= 1 && y <= 9999) return sprintf(out, "%04lld-%02d-%02d", (long long)y, m, d);
  if (y > 9999) return sprintf(out, "%lld-%02d-%02d", (long long)y, m, d);
  return sprintf(out, "%04lld-%02d-%02d (BC)", (long long)(1 - y), m, d);
}
/* unit_per_sec: 1 (S), 1000 (MS), 1000000 (US), 1000000000 (NS); fraction digits trimmed */
int ora_render_timestamp(int64_t v, int64_t unit_per_sec, int tz, char *out) {
  int64_t secs = floor_div64(v, unit_per_sec);
  int64_t frac = v - secs * unit_per_sec;
  int64_t days = floor_div64(secs, 86400);
  int64_t sod = secs - days * 86400;
  int n = ora_render_date((int32_t)days, out);
  n += sprintf(out + n, " %02d:%02d:%02d", (int)(sod / 3600), (int)(sod / 60 % 60), (int)(sod % 60));
  if (frac != 0) {
    int digits = unit_per_sec == 1000 ? 3 : unit_per_sec == 1000000 ? 6 : 9;
    char f[16];
    sprintf(f, "%0*lld", digits, (long long)frac);
    int L = digits;
    while (L > 0 && f[L - 1] == '0') L--;
    f[L] = 0;
    n += sprintf(out + n, ".%s", f);
  }
  if (tz) n += sprintf(out + n, "+00");
  return n;
}
/* TIME: HH:MM:SS[.fraction], fraction digits trimmed like the time part of a TIMESTAMP */
int ora_render_time(int64_t v, int64_t unit_per_sec, char *out) {
  int64_t secs = v / unit_per_sec, frac = v % unit_per_sec;
  int n = sprintf(out, "%02d:%02d:%02d", (int)(secs / 3600), (int)(secs / 60 % 60), (int)(secs % 60));
  if (frac != 0) {
    int digits = unit_per_sec == 1000000 ? 6 : 9;
    char f[16];
    sprintf(f, "%0*lld", digits, (long long)frac);
    int L = digits;
    while (L > 0 && f[L - 1] == '0') L--;
    f[L] = 0;
    n += sprintf(out + n, ".%s", f);
  }
  return n;
}
/* UUID / TIME WITH TIME ZONE / INTERVAL: cells the reference's stream whitelist lets through
 * (src/duckdb_native.c:271-303, loaded at :615-662) and hands to libduckdb for text.  No reference test or
 * fixture holds such a string: UNPINNED, restated from DuckDB's documented storage and VARCHAR casts.
 * UUID: hugeint with the top bit flipped, lowercase hex 8-4-4-4-12. */
int ora_render_uuid(const uint8_t *p, char *out) {
  uint64_t lo, hi;
  memcpy(&lo, p, 8);
  memcpy(&hi, p + 8, 8);
  hi ^= 1ull << 63;
  return sprintf(out, "%08llx-%04llx-%04llx-%04llx-%012llx", (unsigned long long)(hi >> 32), (unsigned long long)((hi >> 16) & 0xffff),
                 (unsigned long long)(hi & 0xffff), (unsigned long long)(lo >> 48), (unsigned long long)(lo & 0xffffffffffffull));
}
/* TIME_TZ: micros << 24 | (57599 - utc offset seconds); "+HH", then ":MM" / ":SS" only when non-zero */
int ora_render_time_tz(uint64_t bits, char *out) {
  int n = ora_render_time((int64_t)(bits >> 24), 1000000, out);
  int off = 57599 - (int)(bits & 0xffffffull);
  out[n++] = off < 0 ? '-' : '+';
  if (off < 0) off = -off;
  n += sprintf(out + n, "%02d", off / 3600);
  if (off % 3600 / 60) n += sprintf(out + n, ":%02d", off % 3600 / 60);
  if (off % 60) n += sprintf(out + n, ":%02d", off % 60);
  return n;
}
/* INTERVAL: years/months from `months`, days, then [-]HH:MM:SS[.ffffff]; zero parts omitted, all zero = 00:00:00 */
static int interval_part(char *out, int n, long long v, const char *name) {
  if (v == 0) return n;
  if (n) out[n++] = ' ';
  n += sprintf(out + n, "%lld%s", v, name);
  if (v != 1 && v != -1) out[n++] = 's';
  return n;
}
int ora_render_interval(int32_t months, int32_t days, int64_t micros, char *out) {
  int n = 0;
  int32_t years = months / 12;
  n = interval_part(out, n, years, " year");
  n = interval_part(out, n, months - years * 12, " month");
  n = interval_part(out, n, days, " day");
  if (micros != 0) {
    if (n) out[n++] = ' ';
    int64_t m = micros; /* kept non-positive (INT64_MIN) */
    if (m < 0) out[n++] = '-'; else m = -m;
    int64_t hour = -(m / 3600000000ll); m += hour * 3600000000ll;
    int64_t min = -(m / 60000000ll); m += min * 60000000ll;
    int64_t sec = -(m / 1000000ll); m += sec * 1000000ll;
    n += sprintf(out + n, "%02lld:%02lld:%02lld", (long long)hour, (long long)min, (long long)sec);
    if (m) {
      char f[8];
      sprintf(f, "%06lld", (long long)-m);
      int L = 6;
      while (L > 0 && f[L - 1] == '0') L--;
      f[L] = 0;
      n += sprintf(out + n, ".%s", f);
    }
  } else if (n == 0) {
    n = sprintf(out, "00:00:00");
  }
  out[n] = 0;
  return n;
}
/* 128-bit integers (HUGEINT, UHUGEINT, DECIMAL(19..38, scale)): sign, digits, '.' before the last `scale` digits */
int ora_render_decimal128(unsigned __int128 u, int is_signed, int scale, char *out) {
  char digits[48];
  int neg = is_signed && (__int128)u < 0;
  unsigned __int128 a = neg ? (unsigned __int128)0 - u : u;
  int n = 0;
  do { digits[n++] = (char)('0' + (int)(a % 10)); a /= 10; } while (a != 0);
  while (n <= scale) digits[n++] = '0';  /* at least one digit before the point */
  int pos = 0;
  if (neg) out[pos++] = '-';
  for (int i = n - 1; i >= 0; i--) {
    out[pos++] = digits[i];
    if (scale > 0 && i == scale) out[pos++] = '.';
  }
  out[pos] = 0;
  return pos;
}
int ora_render_decimal64(int64_t v, int scale, char *out) {
  char digits[32];
  int neg = v < 0;
  uint64_t a = neg ? (uint64_t)0 - (uint64_t)v : (uint64_t)v;
  int n = sprintf(digits, "%llu", (unsigned long long)a);
  int pos = 0;
  if (neg) out[pos++] = '-';
  if (scale == 0) { memcpy(out + pos, digits, (size_t)n); pos += n; out[pos] = 0; return pos; }
  if (n <= scale) {
    out[pos++] = '0'; out[pos++] = '.';
    for (int i = 0; i < scale - n; i++) out[pos++] = '0';
    memcpy(out + pos, digits, (size_t)n); pos += n;
  } else {
    memcpy(out + pos, digits, (size_t)(n - scale)); pos += n - scale;
    out[pos++] = '.';
    memcpy(out + pos, digits + n - scale, (size_t)scale); pos += scale;
  }
  out[pos] = 0;
  return pos;
}
/* does the decimal text read back as v: as a double, or for FLOAT as the float v holds exactly */
static int reads_back(const char *text, double v, int is_float) { return is_float ? strtof(text, NULL) == (float)v : strtod(text, NULL) == v; }

/* shortest round-trip double (FLOAT: shortest round-trip float, DuckDB prints 0.1f as "0.1"), fmt-style
 * (UNPINNED beyond "3.5", "5.333333333333333", "nan", "inf") */
static int render_shortest(double v, int is_float, char *out) {
  if (isnan(v)) return sprintf(out, "nan");
  if (isinf(v)) return sprintf(out, v < 0 ? "-inf" : "inf");
  char buf[40];
  int prec;
  for (prec = 1; prec <= (is_float ? 9 : 17); prec++) {
    snprintf(buf, sizeof buf, "%.*e", prec - 1, v);
    if (reads_back(buf, v, is_float)) break;
    /* the correctly rounded prec-digit decimal is the closest one, but below a power of two the
     * rounding interval is half as wide as above it: the next prec-digit decimal up (or down) may
     * still read back as v although the closest does not.  Shortest round trip takes it. */
    {
      char *ee = strchr(buf, 'e');
      int x10 = atoi(ee + 1), ng = buf[0] == '-';
      unsigned long long m = 0;
      for (char *q = buf + ng; q < ee; q++) if (*q != '.') m = m * 10ull + (unsigned long long)(*q - '0');
      int found = 0;
      for (int step = 1; step >= -1 && !found; step -= 2) {
        unsigned long long m2 = m + (unsigned long long)(long long)step;
        char cand[48];
        snprintf(cand, sizeof cand, "%s%llue%d", ng ? "-" : "", m2, x10 - (prec - 1));
        if (m2 != 0 && reads_back(cand, v, is_float)) {
          /* renormalise: m2 may have gained a digit (99 -> 100) */
          char digits[24];
          int nd2 = snprintf(digits, sizeof digits, "%llu", m2);
          int e2 = x10 + (nd2 - prec);
          while (nd2 > 1 && digits[nd2 - 1] == '0') nd2--;
          int pos2 = 0;
          if (ng) buf[pos2++] = '-';
          buf[pos2++] = digits[0];
          if (nd2 > 1) { buf[pos2++] = '.'; memcpy(buf + pos2, digits + 1, (size_t)(nd2 - 1)); pos2 += nd2 - 1; }
          snprintf(buf + pos2, sizeof buf - (size_t)pos2, "e%+03d", e2);
          found = 1;
        }
      }
      if (found) break;
    }
  }
  /* buf = d.ddddde[+-]XX */
  char *e = strchr(buf, 'e');
  int exp10 = atoi(e + 1);
  char mant[24]; int nd = 0; int neg = buf[0] == '-';
  for (char *p = buf + neg; p < e; p++) if (*p != '.') mant[nd++] = *p;
  mant[nd] = 0;
  int pos = 0;
  if (neg) out[pos++] = '-';
  if (exp10 >= -5 && exp10 < 16) {
    if (exp10 >= 0) {
      for (int i = 0; i <= exp10; i++) out[pos++] = i < nd ? mant[i] : '0';
      out[pos++] = '.';
      if (nd > exp10 + 1) for (int i = exp10 + 1; i < nd; i++) out[pos++] = mant[i];
      else out[pos++] = '0';
    } else {
      out[pos++] = '0'; out[pos++] = '.';
      for (int i = 0; i < -exp10 - 1; i++) out[pos++] = '0';
      for (int i = 0; i < nd; i++) out[pos++] = mant[i];
    }
    out[pos] = 0;
    return pos;
  }
  out[pos++] = mant[0];
  if (nd > 1) { out[pos++] = '.'; for (int i = 1; i < nd; i++) out[pos++] = mant[i]; }
  pos += sprintf(out + pos, "e%c%02d", exp10 < 0 ? '-' : '+', exp10 < 0 ? -exp10 : exp10);
  return pos;
}
int ora_render_double(double v, char *out) { return render_shortest(v, 0, out); }
int ora_render_float(float v, char *out) { return render_shortest((double)v, 1, out); }

/* one fixed-width cell -> DuckDB text (what duckdb_value_varchar / the chunk path's
 * duckdb_value_to_string hand to MoonBit, src/duckdb_native.c:224-238).  Returns length, -1 if the
 * type has no renderer here. */
int ora_render_cell(const ora_column *c, const uint8_t *p, char *out) {
  int ok;
  switch (c->type_id) {
    case T_BOOLEAN: return sprintf(out, "%s", *p ? "true" : "false");
    case T_TINYINT: case T_SMALLINT: case T_INTEGER: case T_BIGINT:
    case T_UTINYINT: case T_USMALLINT: case T_UINTEGER:
      return sprintf(out, "%lld", (long long)load_i64(c, p, &ok));
    case T_UBIGINT: { uint64_t v; memcpy(&v, p, 8); return sprintf(out, "%llu", (unsigned long long)v); }
    case T_FLOAT: { float v; memcpy(&v, p, 4); return ora_render_float(v, out); } /* UNPINNED layout; digits float shortest */
    case T_DOUBLE: { double v; memcpy(&v, p, 8); return ora_render_double(v, out); }
    /* DuckDB stores 'infinity' / '-infinity' as DATE +-INT32_MAX and TIMESTAMP / TIMESTAMPTZ +-INT64_MAX and prints the words */
    case T_DATE: { int32_t v; memcpy(&v, p, 4);
      if (v == INT32_MAX || v == -INT32_MAX) return sprintf(out, "%s", v < 0 ? "-infinity" : "infinity");
      return ora_render_date(v, out); }
    case T_TIMESTAMP: case T_TIMESTAMP_TZ: { int64_t v; memcpy(&v, p, 8);
      if (v == INT64_MAX || v == -INT64_MAX) return sprintf(out, "%s", v < 0 ? "-infinity" : "infinity");
      return ora_render_timestamp(v, 1000000, c->type_id == T_TIMESTAMP_TZ, out); }
    case T_TIMESTAMP_S: { int64_t v; memcpy(&v, p, 8); return ora_render_timestamp(v, 1, 0, out); }
    case T_TIMESTAMP_MS: { int64_t v; memcpy(&v, p, 8); return ora_render_timestamp(v, 1000, 0, out); }
    case T_TIMESTAMP_NS: { int64_t v; memcpy(&v, p, 8); return ora_render_timestamp(v, 1000000000, 0, out); }
    case T_DECIMAL:
      if (c->phys == P_I128) { unsigned __int128 u; memcpy(&u, p, 16); return ora_render_decimal128(u, 1, c->dec_scale, out); }
      return ora_render_decimal64(load_i64(c, p, &ok), c->dec_scale, out);
    /* HUGEINT: what SUM() of an integer column returns (fixtures :34-37, :174-177) */
    case T_HUGEINT: { unsigned __int128 u; memcpy(&u, p, 16); return ora_render_decimal128(u, 1, 0, out); }
    case T_UHUGEINT: { unsigned __int128 u; memcpy(&u, p, 16); return ora_render_decimal128(u, 0, 0, out); }
    case T_TIME: { int64_t v; memcpy(&v, p, 8); return ora_render_time(v, 1000000, out); }   /* fixture :48-51 */
    case T_TIME_NS: { int64_t v; memcpy(&v, p, 8); return ora_render_time(v, 1000000000, out); }
    case T_TIME_TZ: { uint64_t v; memcpy(&v, p, 8); return ora_render_time_tz(v, out); }              /* UNPINNED */
    case T_UUID: return ora_render_uuid(p, out);                                                       /* UNPINNED */
    case T_INTERVAL: { int32_t mo, d; int64_t us; memcpy(&mo, p, 4); memcpy(&d, p + 4, 4); memcpy(&us, p + 8, 8);
                       return ora_render_interval(mo, d, us, out); }                                   /* UNPINNED */
    default: return -1;
  }
}

/* typed Value of one cell: render -> parse_value_with_type (src/duckdb_parsing.mbt:82-144), as
 * Connection::query + QueryResult::to_typed do (src/duckdb_native.mbt:477-497,
 * src/duckdb_typed_result.mbt:8-43).  Tags follow enum dmb_value_tag.
 * Returns tag; *ival for Int/Bool/Date/Timestamp, *dval for Double; text holds the string form. */
enum { V_INT = 0, V_DOUBLE = 1, V_BOOL = 2, V_STRING = 3, V_DATE = 4, V_TIMESTAMP = 5, V_DECIMAL = 6, V_BLOB = 7, V_NULL = 8 };

static int is_special_float(const char *s, int n) {
  return (n == 3 && (!memcmp(s, "nan", 3) || !memcmp(s, "NaN", 3) || !memcmp(s, "inf", 3))) ||
         (n == 8 && !memcmp(s, "Infinity", 8)) || (n == 4 && !memcmp(s, "-inf", 4)) || (n == 9 && !memcmp(s, "-Infinity", 9));
}

int ora_typed_from_text(int32_t type_id, const char *s, int n, int64_t *ival, double *dval) {
  int ok;
  switch (type_id) {
    case T_BOOLEAN:
      if (n == 4 && !memcmp(s, "true", 4)) { *ival = 1; return V_BOOL; }
      if (n == 5 && !memcmp(s, "false", 5)) { *ival = 0; return V_BOOL; }
      return V_STRING;
    case T_TINYINT: case T_SMALLINT: case T_INTEGER: case T_BIGINT:
    case T_UTINYINT: case T_USMALLINT: case T_UINTEGER: case T_UBIGINT:
      *ival = ora_parse_int(s, n); return V_INT;
    case T_FLOAT: case T_DOUBLE:
      if (is_special_float(s, n)) return V_STRING;
      *dval = ora_parse_double(s, n); return V_DOUBLE;
    case T_DATE: { int32_t d = ora_parse_date(s, n, &ok); if (!ok) return V_STRING; *ival = d; return V_DATE; }
    case T_TIMESTAMP: case T_TIMESTAMP_S: case T_TIMESTAMP_MS: case T_TIMESTAMP_NS: case T_TIMESTAMP_TZ: {
      int64_t t = ora_parse_timestamp(s, n, &ok); if (!ok) return V_STRING; *ival = t; return V_TIMESTAMP; }
    default: return V_STRING;
  }
}

/* typed column of a fixed-width column through the text round trip.
 * tags[n], ivals[n], dvals[n]; text not retained.  Returns 0, or -1 if a cell has no renderer. */
int ora_typed_fixed_column(ora_result *r, int32_t col, uint8_t *tags, int64_t *ivals, double *dvals) {
  const ora_column *c = &r->batch.cols[col];
  int w = PHYS_W[c->phys];
  char text[96];
  for (int64_t k = 0; k < r->batch.nchunks; k++) {
    const uint8_t *v = vec_data(c, k);
    for (uint32_t i = 0; i < r->batch.counts[k]; i++) {
      int64_t row = r->row_off[k] + i;
      ivals[row] = 0; dvals[row] = 0.0;
      if (chunk_is_null(c, k, (int32_t)i)) { tags[row] = V_NULL; continue; }
      int n = ora_render_cell(c, v + (size_t)i * (size_t)w, text);
      if (n < 0) return -1;
      tags[row] = (uint8_t)ora_typed_from_text(c->type_id, text, n, &ivals[row], &dvals[row]);
    }
  }
  return 0;
}

/* Arrow / typed fixed-width column, per cell.  out_values width is implied by dst.
 * Returns 0, -1 on unsupported. */
int ora_arrow_fixed(ora_result *r, int32_t col, int dst, uint8_t *out_values, uint8_t *out_bitmap,
                    uint8_t *out_valid_bytes, int64_t *null_count) {
  const ora_column *c = &r->batch.cols[col];
  int w = PHYS_W[c->phys];
  int64_t nulls = 0;
  if (out_bitmap) memset(out_bitmap, 0, (size_t)((r->nrows + 63) / 64 * 8));
  if (dst == D_BOOL_BITS && out_values) memset(out_values, 0, (size_t)((r->nrows + 7) / 8));
  for (int64_t k = 0; k < r->batch.nchunks; k++) {
    const uint8_t *v = vec_data(c, k);
    for (uint32_t i = 0; i < r->batch.counts[k]; i++) {
      int64_t row = r->row_off[k] + i;
      int isnull = chunk_is_null(c, k, (int32_t)i);
      if (isnull) nulls++;
      else if (out_bitmap) out_bitmap[row >> 3] |= (uint8_t)(1u << (row & 7));
      if (out_valid_bytes) out_valid_bytes[row] = isnull ? 0 : 1;
      if (!out_values) continue;
      const uint8_t *p = v + (size_t)i * (size_t)w;
      int ok = 1;
      switch (dst) {
        case D_SAME:
          if (isnull) memset(out_values + (size_t)row * (size_t)w, 0, (size_t)w);
          else memcpy(out_values + (size_t)row * (size_t)w, p, (size_t)w);
          break;
        case D_I32_TRUNC: { int32_t x = isnull ? 0 : (int32_t)load_i64(c, p, &ok); memcpy(out_values + row * 4, &x, 4); break; }
        case D_I64: { int64_t x = isnull ? 0 : load_i64(c, p, &ok); memcpy(out_values + row * 8, &x, 8); break; }
        case D_F64: {
          double x = 0.0;
          if (!isnull) {
            if (c->phys == P_F64) memcpy(&x, p, 8);
            else if (c->phys == P_F32) { float f; memcpy(&f, p, 4); x = (double)f; }
            else if (c->phys == P_U64) { uint64_t u; memcpy(&u, p, 8); x = (double)u; }
            else if (c->phys == P_I128) { ora_hugeint h; memcpy(&h, p, 16); x = hugeint_to_double(h.lo, h.hi); }
            else if (c->phys == P_U128) { ora_hugeint h; memcpy(&h, p, 16); x = (double)h.lo + (double)(uint64_t)h.hi * 18446744073709551616.0; }
            else x = (double)load_i64(c, p, &ok);
          }
          memcpy(out_values + row * 8, &x, 8); break; }
        case D_DEC_I64: { int64_t x = isnull ? 0 : decimal_to_i64(c, p); memcpy(out_values + row * 8, &x, 8); break; }
        case D_DEC_I32_TRUNC: { int32_t x = isnull ? 0 : (int32_t)decimal_to_i64(c, p); memcpy(out_values + row * 4, &x, 4); break; }
        case D_DEC_F64: { double x = isnull ? 0.0 : decimal_to_double(c, p); memcpy(out_values + row * 8, &x, 8); break; }
        case D_DEC_BOOL_BYTE: out_values[row] = (uint8_t)(!isnull && decimal_to_i64(c, p) != 0); break;
        case D_BOOL_BYTE: {
          uint8_t x = 0;
          if (!isnull) {
            if (c->phys == P_F64) { double d; memcpy(&d, p, 8); x = d != 0.0; }
            else if (c->phys == P_F32) { float f; memcpy(&f, p, 4); x = f != 0.0f; }
            else if (c->phys == P_U64) { uint64_t u; memcpy(&u, p, 8); x = u != 0; }
            else if (c->phys == P_I128 || c->phys == P_U128) { ora_hugeint h; memcpy(&h, p, 16); x = (h.lo | (uint64_t)h.hi) != 0; }
            else x = load_i64(c, p, &ok) != 0;
          }
          out_values[row] = x; break; }
        case D_BOOL_BITS:
          if (!isnull && *p) out_values[row >> 3] |= (uint8_t)(1u << (row & 7));
          break;
        case D_I128: {
          ora_hugeint x = {0, 0};
          if (!isnull) {
            if (c->phys == P_I128) memcpy(&x, p, 16);
            else { int64_t s = load_i64(c, p, &ok); x.lo = (uint64_t)s; x.hi = s < 0 ? -1 : 0; }
          }
          memcpy(out_values + row * 16, &x, 16); break; }
        case D_I32_SAT: {
          int32_t x = 0;
          if (!isnull) {
            if (c->phys == P_U64) { uint64_t u; memcpy(&u, p, 8); x = u > 2147483647ull ? INT32_MAX : (int32_t)u; }
            else { int64_t s = load_i64(c, p, &ok); x = s > INT32_MAX ? INT32_MAX : s < INT32_MIN ? INT32_MIN : (int32_t)s; }
          }
          memcpy(out_values + row * 4, &x, 4); break; }
        case D_TS_US_FROM_S: case D_TS_US_FROM_MS: case D_TS_US_FROM_NS: {
          int64_t x = 0;
          if (!isnull) {
            int64_t s; memcpy(&s, p, 8);
            x = dst == D_TS_US_FROM_S ? (int64_t)((uint64_t)s * 1000000ull)
              : dst == D_TS_US_FROM_MS ? (int64_t)((uint64_t)s * 1000ull) : floor_div64(s, 1000);
          }
          memcpy(out_values + row * 8, &x, 8); break; }
        case D_MONTH_DAY_NANO: {
          uint8_t x[16] = {0};
          if (!isnull) { memcpy(x, p, 8); int64_t us; memcpy(&us, p + 8, 8); int64_t ns = (int64_t)((uint64_t)us * 1000ull); memcpy(x + 8, &ns, 8); }
          memcpy(out_values + row * 16, x, 16); break; }
        case D_DATE_REF: { /* the reference's own path: text -> parse_date */
          int32_t x = 0;
          if (!isnull) {
            int32_t d; memcpy(&d, p, 4);
            char text[40]; int n = ora_render_date(d, text); int pok;
            int32_t parsed = ora_parse_date(text, n, &pok);
            x = pok ? parsed : d; /* non 10-char dates fall back to Value::String in the reference */
          }
          memcpy(out_values + row * 4, &x, 4); break; }
        default: return -1;
      }
      (void)ok;
    }
  }
  if (null_count) *null_count = nulls;
  return 0;
}

/* Arrow utf8 of a VARCHAR/BLOB column.  mode 0: int32 offsets, 1: int64 offsets, 2: the reference's
 * NUL-terminated stream expressed as offsets (every row strnlen+1 bytes, NULL row a lone \0).
 * Call with out_data == NULL to size (*total). */
int ora_arrow_string(ora_result *r, int32_t col, int mode, void *out_offsets, uint8_t *out_data, int64_t *total) {
  const ora_column *c = &r->batch.cols[col];
  if (c->phys != P_STRING) return -1;
  int64_t pos = 0;
  for (int64_t k = 0; k < r->batch.nchunks; k++) {
    const ora_string_t *v = (const ora_string_t *)vec_data(c, k);
    for (uint32_t i = 0; i < r->batch.counts[k]; i++) {
      int64_t row = r->row_off[k] + i;
      if (out_offsets) { if (mode == 1) ((int64_t *)out_offsets)[row] = pos; else ((int32_t *)out_offsets)[row] = (int32_t)pos; }
      int isnull = chunk_is_null(c, k, (int32_t)i);
      if (!isnull) {
        ora_string_t str = v[i];
        const char *ptr = string_t_data(&str);
        uint32_t len = str.length;
        if (mode == 2) len = (uint32_t)strnlen(ptr, len);
        if (out_data) memcpy(out_data + pos, ptr, len);
        pos += len;
      }
      if (mode == 2) { if (out_data) out_data[pos] = 0; pos += 1; }
    }
  }
  if (out_offsets) { if (mode == 1) ((int64_t *)out_offsets)[r->nrows] = pos; else ((int32_t *)out_offsets)[r->nrows] = (int32_t)pos; }
  if (total) *total = pos;
  return 0;
}

/* ------------------------------------------------------------------ reverse path oracle
 * Arrow -> DataChunk vectors, per cell, the way the reference's appender feeds libduckdb one
 * value at a time (src/duckdb_native.c:1116-1235) — expressed on the vector layouts that
 * duckdb_append_data_chunk consumes (:2109-2132).  Chunk k = rows [2048k, 2048k+2048). */
static inline int arrow_bit(const uint8_t *bm, int64_t i) { return (bm[i >> 3] >> (i & 7)) & 1; }

/* fixed width: values[nrows*w] (already at the slice start), bitmap with bit offset, into slabs
 * out_data[nchunks*2048*w_out], out_validity[nchunks*32].  rev_op mirrors enum dmb_rev_op. */
int ora_rev_fixed(const uint8_t *values, const uint8_t *bitmap, int64_t bit_offset, int64_t nrows, int rev_op,
                  uint8_t *out_data, uint64_t *out_validity, int64_t *null_count) {
  static const int w_in[] = {1, 2, 4, 8, 16, 0, 16, 16, 16};
  static const int w_out[] = {1, 2, 4, 8, 16, 1, 8, 4, 2};
  int wi = w_in[rev_op], wo = w_out[rev_op];
  int64_t nchunks = (nrows + ORA_VECTOR_SIZE - 1) / ORA_VECTOR_SIZE;
  memset(out_validity, 0, (size_t)nchunks * 32 * 8);
  memset(out_data, 0, (size_t)nchunks * ORA_VECTOR_SIZE * (size_t)wo);
  int64_t nulls = 0;
  for (int64_t i = 0; i < nrows; i++) {
    int valid = bitmap ? arrow_bit(bitmap, bit_offset + i) : 1;
    if (valid) out_validity[i >> 6] |= 1ull << (i & 63); else nulls++;
    uint8_t *dst = out_data + (size_t)i * (size_t)wo;
    if (!valid) continue; /* payload under NULL: zero */
    if (rev_op == 5) dst[0] = (uint8_t)arrow_bit(values, bit_offset + i);
    else if (rev_op >= 6) memcpy(dst, values + (size_t)i * 16, (size_t)wo); /* low bytes of decimal128 */
    else memcpy(dst, values + (size_t)i * (size_t)wi, (size_t)wi);
  }
  if (null_count) *null_count = nulls;
  return 0;
}

/* utf8 -> duckdb_string_t: length <= 12 inlined with zero padding, else 4-byte prefix + pointer
 * to the bytes in place in the Arrow data buffer at host address data_host_base. */
int ora_rev_string(const void *offsets, int large, const uint8_t *data, uint64_t data_host_base,
                   const uint8_t *bitmap, int64_t bit_offset, int64_t nrows, uint8_t *out,
                   uint64_t *out_validity, int64_t *null_count) {
  int64_t nchunks = (nrows + ORA_VECTOR_SIZE - 1) / ORA_VECTOR_SIZE;
  memset(out_validity, 0, (size_t)nchunks * 32 * 8);
  memset(out, 0, (size_t)nchunks * ORA_VECTOR_SIZE * 16);
  int64_t nulls = 0;
  for (int64_t i = 0; i < nrows; i++) {
    int valid = bitmap ? arrow_bit(bitmap, bit_offset + i) : 1;
    if (!valid) { nulls++; continue; }
    out_validity[i >> 6] |= 1ull << (i & 63);
    int64_t o0 = large ? ((const int64_t *)offsets)[i] : ((const int32_t *)offsets)[i];
    int64_t o1 = large ? ((const int64_t *)offsets)[i + 1] : ((const int32_t *)offsets)[i + 1];
    uint32_t len = (uint32_t)(o1 - o0);
    uint8_t *e = out + (size_t)i * 16;
    memcpy(e, &len, 4);
    if (len <= 12) memcpy(e + 4, data + o0, len);
    else { memcpy(e + 4, data + o0, 4); uint64_t p = data_host_base + (uint64_t)o0; memcpy(e + 8, &p, 8); }
  }
  if (null_count) *null_count = nulls;
  return 0;
}

/* ------------------------------------------------------------------ LIST / STRUCT / MAP cells of the row appender
 * The reference serialises them as text and appends the text as one VARCHAR cell (src/duckdb_native.c:1735-1790
 * list, :1792-1858 struct, :1860-1926 map): items between double quotes, no escaping, ", " between entries, ": "
 * between a key and its value.  duckdb_append_varchar takes a C string, so the cell ends at the first NUL byte.
 * Returns the cell's length (strlen of the buffer); out needs room for the full serialisation + 1. */
static size_t ora_put_quoted(char *out, size_t pos, const uint8_t *p, int32_t len) {
  out[pos++] = '"';
  for (int32_t j = 0; j < len; j++) out[pos++] = (char)p[j];
  out[pos++] = '"';
  return pos;
}

int64_t ora_list_varchar_text(const uint8_t *const *values, const int32_t *lens, int32_t count, char *out) {
  size_t pos = 0;
  out[pos++] = '[';
  for (int32_t i = 0; i < count; i++) {
    if (i > 0) { out[pos++] = ','; out[pos++] = ' '; }
    pos = ora_put_quoted(out, pos, values[i], values[i] ? lens[i] : 0);
  }
  out[pos++] = ']';
  out[pos] = '\0';
  return (int64_t)strlen(out);
}

/* struct (field names / values) and map (keys / values) share the form */
int64_t ora_pairs_varchar_text(const uint8_t *const *keys, const int32_t *key_lens, const uint8_t *const *values,
                               const int32_t *value_lens, int32_t count, char *out) {
  size_t pos = 0;
  out[pos++] = '{';
  for (int32_t i = 0; i < count; i++) {
    if (i > 0) { out[pos++] = ','; out[pos++] = ' '; }
    pos = ora_put_quoted(out, pos, keys[i], keys[i] ? key_lens[i] : 0);
    out[pos++] = ':';
    out[pos++] = ' ';
    pos = ora_put_quoted(out, pos, values[i], values[i] ? value_lens[i] : 0);
  }
  out[pos++] = '}';
  out[pos] = '\0';
  return (int64_t)strlen(out);
}

/* ------------------------------------------------------------------ LIST vectors -> Arrow list<child>
 * (SURVEY.md 8f item 3; the reference rejects LIST on its chunk path, src/duckdb_native.c:271-303, so this restates
 * the Arrow-format contract: what DuckDB's own Arrow appender produces for a LIST column of flat chunks.)
 * Per chunk k: entries {uint64 offset, uint64 length} at entries + data_off[k], the LIST validity mask, and the
 * chunk's child vector staged at element child_base[k] (mask words at child_val_off[k], -1 = all valid).
 * Rows in order: a valid row appends its child elements [offset, offset + length); a NULL row appends nothing. */
int ora_list_arrow(const uint8_t *entries, const uint64_t *data_off, const uint64_t *validity, const int64_t *val_off,
                   const uint32_t *counts, int64_t nchunks, const uint64_t *child_base, const uint8_t *child_data,
                   const uint64_t *child_validity, const int64_t *child_val_off, int child_width, int large,
                   void *out_offsets, uint8_t *out_child, uint8_t *out_child_bitmap, int64_t *total, int64_t *child_nulls) {
  int64_t row = 0, pos = 0, nulls = 0;
  for (int64_t k = 0; k < nchunks; k++) {
    const uint64_t *ent = (const uint64_t *)(entries + data_off[k]);
    const uint64_t *mask = val_off[k] < 0 ? NULL : validity + val_off[k];
    const uint64_t *cmask = (child_validity && child_val_off && child_val_off[k] >= 0) ? child_validity + child_val_off[k] : NULL;
    for (uint32_t i = 0; i < counts[k]; i++, row++) {
      if (large) ((int64_t *)out_offsets)[row] = pos; else ((int32_t *)out_offsets)[row] = (int32_t)pos;
      if (mask && !((mask[i / 64] >> (i % 64)) & 1ull)) continue;
      uint64_t off = ent[2 * i], len = ent[2 * i + 1];
      for (uint64_t e = off; e < off + len; e++, pos++) {
        int valid = cmask ? (int)((cmask[e / 64] >> (e % 64)) & 1ull) : 1;
        if (valid) {
          memcpy(out_child + (size_t)pos * (size_t)child_width, child_data + (size_t)(child_base[k] + e) * (size_t)child_width, (size_t)child_width);
          out_child_bitmap[pos / 8] |= (uint8_t)(1u << (pos % 8));
        } else {
          memset(out_child + (size_t)pos * (size_t)child_width, 0, (size_t)child_width);
          nulls++;
        }
      }
    }
  }
  if (large) ((int64_t *)out_offsets)[row] = pos; else ((int32_t *)out_offsets)[row] = (int32_t)pos;
  if (total) *total = pos;
  if (child_nulls) *child_nulls = nulls;
  return 0;
}
