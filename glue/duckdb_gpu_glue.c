/*
 * duckdb_gpu_glue.c — the second native stub of the MoonBit package, "next to duckdb_native.c" (SURVEY.md §8b).
 *
 * It defines the entry points of the reference's stub that RUN SQL OR OPEN AN APPENDER and therefore need libduckdb:
 *
 *   duckdb_mb_query_arrow    src/duckdb_native.c:2219-2268   -> ArrowResult handle
 *   duckdb_mb_query          src/duckdb_native.c:142-172     -> materialised result handle
 *   duckdb_mb_query_stream   src/duckdb_native.c:355-397     -> stream handle
 *   duckdb_mb_appender_create src/duckdb_native.c:1032-1081  -> appender handle
 *
 * Each runs the statement through libduckdb exactly like the reference, then hands the result's DataChunks — the
 * pointers duckdb_vector_get_data / duckdb_vector_get_validity return (:529-530,547), duckdb_string_t with their host
 * pointers (:597-603), ENUM dictionaries, LIST child vectors — to libduckdb_mb_gpu.so as ONE dmb_host_batch.  Every other
 * symbol of the path (duckdb_mb_arrow_*, duckdb_mb_result_*, duckdb_mb_stream_*, duckdb_mb_chunk_*, duckdb_mb_begin_row /
 * append_* / end_row / flush, duckdb_mb_appender_destroy / _error) is exported by the library itself with the
 * reference's signatures, so the MoonBit `extern "C"` declarations stay as they are.
 *
 * In duckdb_native.c the maintainer deletes the functions this file and the library now define (the result / stream /
 * arrow / appender blocks) and keeps the connection, config, prepared-statement and logical-type blocks; see
 * INTEGRATION.md.  Built in this repository against glue/mock/duckdb.h + glue/mock/libduckdb_mock.c (libduckdb is
 * not in the image) and driven by tests/test_glue_mock.py; nothing here is mock specific.
 */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "duckdb.h"
#include "duckdb_mb_gpu.h"

/* same layout as the reference's handle (src/duckdb_native.c:10-13): the connection block of duckdb_native.c stays */
typedef struct {
  duckdb_database db;
  duckdb_connection conn;
} duckdb_mb_connection;

/* ---- error string: the reference keeps one process-global message read back by duckdb_mb_last_error (:22-40,240-246).
 * duckdb_native.c's setter is `static`; the maintainer makes it extern (INTEGRATION.md).  Standalone (the tests):
 * this file owns the message. */
#ifdef DMB_GLUE_STANDALONE
static char *g_last_error = NULL;
static void duckdb_mb_set_error(const char *message) {
  free(g_last_error);
  g_last_error = message ? strdup(message) : NULL;
}
moonbit_bytes_t duckdb_mb_last_error(void) {
  const char *m = g_last_error ? g_last_error : "";
  size_t n = strlen(m);
  moonbit_bytes_t b = moonbit_make_bytes_raw((int32_t)n);
  if (b && n) memcpy(b, m, n);
  return b;
}
#else
void duckdb_mb_set_error(const char *message);
#endif

static char *bytes_to_cstr(moonbit_bytes_t bytes) { /* like duckdb_mb_bytes_to_cstr, :51-65 */
  if (!bytes) return NULL;
  int32_t len = Moonbit_array_length(bytes);
  char *buf = (char *)malloc((size_t)len + 1);
  if (!buf) return NULL;
  if (len > 0) memcpy(buf, bytes, (size_t)len);
  buf[len] = '\0';
  return buf;
}

/* ---- one GPU context per process, created on first use (device: DMB_DEVICE, default 0) */
static duckdb_mb_gpu_ctx *g_ctx = NULL;
static duckdb_mb_gpu_ctx *glue_ctx(void) {
  if (!g_ctx) {
    const char *dev = getenv("DMB_DEVICE");
    g_ctx = duckdb_mb_gpu_ctx_create(dev ? atoi(dev) : 0);
    if (!g_ctx) duckdb_mb_set_error(duckdb_mb_gpu_last_error());
  }
  return g_ctx;
}

/* ---- what a result handle keeps alive: the duckdb_result, its chunks, and the pointer tables of the batch */
typedef struct {
  duckdb_result result;
  duckdb_data_chunk *chunks;
  int64_t nchunks, cap;
  uint32_t *counts;
  int32_t ncols;
  dmb_host_column *cols;
  const void ***data;          /* [ncols][nchunks] */
  const uint64_t ***validity;
  dmb_enum_dict *dicts;        /* [ncols] */
  uint32_t **dict_offsets;
  char **dict_data;
  dmb_host_list *lists;        /* [ncols] */
  const void ***child_data;
  const uint64_t ***child_validity;
  uint64_t **child_sizes;
} glue_owner;

static void owner_destroy(void *p) {
  glue_owner *o = (glue_owner *)p;
  if (!o) return;
  for (int64_t k = 0; k < o->nchunks; k++) duckdb_destroy_data_chunk(&o->chunks[k]);
  for (int32_t c = 0; c < o->ncols; c++) {
    if (o->data) free((void *)o->data[c]);
    if (o->validity) free((void *)o->validity[c]);
    if (o->dict_offsets) free(o->dict_offsets[c]);
    if (o->dict_data) free(o->dict_data[c]);
    if (o->child_data) free((void *)o->child_data[c]);
    if (o->child_validity) free((void *)o->child_validity[c]);
    if (o->child_sizes) free(o->child_sizes[c]);
  }
  free(o->chunks); free(o->counts); free(o->cols); free((void *)o->data); free((void *)o->validity); free(o->dicts);
  free(o->dict_offsets); free(o->dict_data); free(o->lists); free((void *)o->child_data); free((void *)o->child_validity);
  free(o->child_sizes);
  duckdb_destroy_result(&o->result);
  free(o);
}

static int32_t phys_of(duckdb_type t, duckdb_type internal) {
  switch (t) {
    case DUCKDB_TYPE_BOOLEAN: return DMB_PHYS_BOOL;
    case DUCKDB_TYPE_TINYINT: return DMB_PHYS_I8;
    case DUCKDB_TYPE_SMALLINT: return DMB_PHYS_I16;
    case DUCKDB_TYPE_INTEGER: case DUCKDB_TYPE_DATE: return DMB_PHYS_I32;
    case DUCKDB_TYPE_BIGINT: case DUCKDB_TYPE_TIMESTAMP: case DUCKDB_TYPE_TIME: case DUCKDB_TYPE_TIMESTAMP_S: case DUCKDB_TYPE_TIMESTAMP_MS:
    case DUCKDB_TYPE_TIMESTAMP_NS: case DUCKDB_TYPE_TIMESTAMP_TZ: case DUCKDB_TYPE_TIME_NS: return DMB_PHYS_I64;
    case DUCKDB_TYPE_UTINYINT: return DMB_PHYS_U8;
    case DUCKDB_TYPE_USMALLINT: return DMB_PHYS_U16;
    case DUCKDB_TYPE_UINTEGER: return DMB_PHYS_U32;
    case DUCKDB_TYPE_UBIGINT: case DUCKDB_TYPE_TIME_TZ: return DMB_PHYS_U64;
    case DUCKDB_TYPE_FLOAT: return DMB_PHYS_F32;
    case DUCKDB_TYPE_DOUBLE: return DMB_PHYS_F64;
    case DUCKDB_TYPE_HUGEINT: return DMB_PHYS_I128;
    case DUCKDB_TYPE_UHUGEINT: case DUCKDB_TYPE_UUID: case DUCKDB_TYPE_LIST: return DMB_PHYS_U128; /* LIST: duckdb_list_entry, 16 bytes */
    case DUCKDB_TYPE_INTERVAL: return DMB_PHYS_INTERVAL;
    case DUCKDB_TYPE_VARCHAR: case DUCKDB_TYPE_BLOB: return DMB_PHYS_STRING;
    case DUCKDB_TYPE_DECIMAL: case DUCKDB_TYPE_ENUM: return phys_of(internal, DUCKDB_TYPE_INVALID);
    default: return -1;
  }
}

/* Run `sql` and wrap every chunk of its result in a library result handle.  NULL + last error on failure. */
static duckdb_mb_arrow_result *glue_query(duckdb_mb_connection *handle, moonbit_bytes_t sql) {
  duckdb_mb_gpu_ctx *ctx = glue_ctx();
  if (!ctx) return NULL;
  char *sql_c = bytes_to_cstr(sql);
  if (!sql_c) { duckdb_mb_set_error("failed to allocate sql buffer"); return NULL; }
  glue_owner *o = (glue_owner *)calloc(1, sizeof(glue_owner));
  if (!o) { free(sql_c); duckdb_mb_set_error("failed to allocate result"); return NULL; }
  duckdb_state state = duckdb_query(handle->conn, sql_c, &o->result);
  free(sql_c);
  if (state != DuckDBSuccess) {
    const char *error = duckdb_result_error(&o->result);
    duckdb_mb_set_error(error ? error : "duckdb_query failed"); /* (the reference reads the message after freeing it, B.9: not reproduced) */
    owner_destroy(o);
    return NULL;
  }
  const int32_t ncols = (int32_t)duckdb_column_count(&o->result);
  o->ncols = ncols;
  for (;;) { /* every chunk of the materialised result */
    duckdb_data_chunk ch = duckdb_fetch_chunk(o->result);
    if (!ch) break;
    if (o->nchunks == o->cap) {
      o->cap = o->cap ? o->cap * 2 : 64;
      o->chunks = (duckdb_data_chunk *)realloc(o->chunks, sizeof(duckdb_data_chunk) * (size_t)o->cap);
      o->counts = (uint32_t *)realloc(o->counts, sizeof(uint32_t) * (size_t)o->cap);
    }
    o->chunks[o->nchunks] = ch;
    o->counts[o->nchunks] = (uint32_t)duckdb_data_chunk_get_size(ch);
    o->nchunks++;
  }
  const size_t nc = (size_t)(ncols > 0 ? ncols : 1), nk = (size_t)(o->nchunks > 0 ? o->nchunks : 1);
  o->cols = (dmb_host_column *)calloc(nc, sizeof(dmb_host_column));
  o->data = (const void ***)calloc(nc, sizeof(void *));
  o->validity = (const uint64_t ***)calloc(nc, sizeof(void *));
  o->dicts = (dmb_enum_dict *)calloc(nc, sizeof(dmb_enum_dict));
  o->dict_offsets = (uint32_t **)calloc(nc, sizeof(void *));
  o->dict_data = (char **)calloc(nc, sizeof(void *));
  o->lists = (dmb_host_list *)calloc(nc, sizeof(dmb_host_list));
  o->child_data = (const void ***)calloc(nc, sizeof(void *));
  o->child_validity = (const uint64_t ***)calloc(nc, sizeof(void *));
  o->child_sizes = (uint64_t **)calloc(nc, sizeof(void *));
  for (int32_t c = 0; c < ncols; c++) {
    dmb_host_column *col = &o->cols[c];
    const duckdb_type t = duckdb_column_type(&o->result, (idx_t)c);
    duckdb_logical_type lt = duckdb_column_logical_type(&o->result, (idx_t)c);
    duckdb_type internal = DUCKDB_TYPE_INVALID;
    col->name = duckdb_column_name(&o->result, (idx_t)c); /* owned by the duckdb_result, which the owner keeps */
    col->type_id = (int32_t)t;
    if (t == DUCKDB_TYPE_DECIMAL) {
      col->dec_width = duckdb_decimal_width(lt);
      col->dec_scale = duckdb_decimal_scale(lt);
      internal = duckdb_decimal_internal_type(lt);
    } else if (t == DUCKDB_TYPE_ENUM) {
      internal = duckdb_enum_internal_type(lt);
      const uint32_t size = duckdb_enum_dictionary_size(lt);
      uint32_t *offs = (uint32_t *)calloc((size_t)size + 1, sizeof(uint32_t));
      size_t cap = 64, pos = 0;
      char *bytes = (char *)malloc(cap);
      for (uint32_t i = 0; i < size; i++) {
        char *label = duckdb_enum_dictionary_value(lt, i);
        const size_t n = label ? strlen(label) : 0;
        if (pos + n + 1 > cap) { while (pos + n + 1 > cap) cap *= 2; bytes = (char *)realloc(bytes, cap); }
        if (n) memcpy(bytes + pos, label, n);
        pos += n;
        offs[i + 1] = (uint32_t)pos;
        duckdb_free(label);
      }
      o->dict_offsets[c] = offs;
      o->dict_data[c] = bytes;
      o->dicts[c].size = size;
      o->dicts[c].offsets = offs;
      o->dicts[c].data = bytes;
      col->dict = &o->dicts[c];
    }
    col->phys = phys_of(t, internal);
    o->data[c] = (const void **)calloc(nk, sizeof(void *));
    o->validity[c] = (const uint64_t **)calloc(nk, sizeof(void *));
    for (int64_t k = 0; k < o->nchunks; k++) {
      duckdb_vector v = duckdb_data_chunk_get_vector(o->chunks[k], (idx_t)c);
      o->data[c][k] = duckdb_vector_get_data(v);          /* :547 */
      o->validity[c][k] = duckdb_vector_get_validity(v);  /* :530, NULL = all valid */
    }
    col->data = o->data[c];
    col->validity = o->validity[c];
    /* VARCHAR / BLOB: every vector owns its own string heap, nobody knows a contiguous region: heap_len = 0, the
     * stager compacts what the pointers refer to (include/duckdb_mb_gpu.h, dmb_host_column) */
    if (t == DUCKDB_TYPE_LIST) {
      duckdb_logical_type child_lt = duckdb_list_type_child_type(lt);
      dmb_host_list *l = &o->lists[c];
      const duckdb_type ct = duckdb_get_type_id(child_lt);
      duckdb_type cinternal = DUCKDB_TYPE_INVALID;
      l->child_type_id = (int32_t)ct;
      if (ct == DUCKDB_TYPE_DECIMAL) {
        l->child_dec_width = duckdb_decimal_width(child_lt);
        l->child_dec_scale = duckdb_decimal_scale(child_lt);
        cinternal = duckdb_decimal_internal_type(child_lt);
      }
      l->child_phys = phys_of(ct, cinternal);
      o->child_data[c] = (const void **)calloc(nk, sizeof(void *));
      o->child_validity[c] = (const uint64_t **)calloc(nk, sizeof(void *));
      o->child_sizes[c] = (uint64_t *)calloc(nk, sizeof(uint64_t));
      for (int64_t k = 0; k < o->nchunks; k++) {
        duckdb_vector v = duckdb_data_chunk_get_vector(o->chunks[k], (idx_t)c);
        duckdb_vector child = duckdb_list_vector_get_child(v);
        o->child_sizes[c][k] = duckdb_list_vector_get_size(v);
        o->child_data[c][k] = child ? duckdb_vector_get_data(child) : NULL;
        o->child_validity[c][k] = child ? duckdb_vector_get_validity(child) : NULL;
      }
      l->child_data = o->child_data[c];
      l->child_validity = o->child_validity[c];
      l->child_sizes = o->child_sizes[c];
      col->list = l;
      duckdb_destroy_logical_type(&child_lt);
    }
    duckdb_destroy_logical_type(&lt);
  }
  dmb_host_batch batch;
  memset(&batch, 0, sizeof(batch));
  batch.ncols = ncols;
  batch.flags = 0; /* libduckdb's buffers are pageable */
  batch.nchunks = o->nchunks;
  batch.counts = o->counts;
  batch.cols = o->cols;
  duckdb_mb_arrow_result *r = duckdb_mb_gpu_result_from_chunks(ctx, &batch);
  if (!r) {
    duckdb_mb_set_error(duckdb_mb_gpu_last_error());
    owner_destroy(o);
    return NULL;
  }
  duckdb_mb_gpu_result_set_owner(r, o, owner_destroy);
  return r;
}

/* src/duckdb_native.c:2219-2268 */
duckdb_mb_arrow_result *duckdb_mb_query_arrow(duckdb_mb_connection *handle, moonbit_bytes_t sql) {
  if (!handle || !handle->conn) { duckdb_mb_set_error("invalid connection handle"); return NULL; }
  return glue_query(handle, sql);
}

/* src/duckdb_native.c:142-172.  The MoonBit side holds the handle as an #external type and only passes it back to
 * duckdb_mb_result_* (exported by the library), so the pointee may be the library's result object. */
duckdb_mb_arrow_result *duckdb_mb_query(duckdb_mb_connection *handle, moonbit_bytes_t sql) {
  if (!handle) { duckdb_mb_set_error("connection is null"); return NULL; }
  return glue_query(handle, sql);
}

/* src/duckdb_native.c:355-397.  The reference prepares the statement and executes it streaming, then checks the column
 * types against its whitelist (:319-353); here the result is collected chunk by chunk up front (one GPU pass renders a
 * whole column) and the same whitelist + error message apply (duckdb_mb_gpu_stream_from_result). */
duckdb_mb_stream *duckdb_mb_query_stream(duckdb_mb_connection *handle, moonbit_bytes_t sql) {
  if (!handle) { duckdb_mb_set_error("connection is null"); return NULL; }
  duckdb_mb_arrow_result *r = glue_query(handle, sql);
  if (!r) return NULL;
  duckdb_mb_stream *s = duckdb_mb_gpu_stream_from_result_owned(r); /* destroys r on failure */
  if (!s) duckdb_mb_set_error(duckdb_mb_gpu_last_error());
  return s;
}

/* ---- appender: the library converts rows / Arrow batches into DataChunk vectors on the GPU and calls this sink once
 * per finished 2048-row chunk; the sink fills a duckdb_data_chunk and appends it (the bulk door, :2109-2132). */
typedef struct {
  duckdb_appender appender;
  duckdb_mb_appender *lib; /* the library's handle: LIST children are read through it during a sink call */
  int32_t ncols;
  duckdb_logical_type *types;
  int32_t *type_ids;
  int32_t *widths;
  int32_t *child_type_ids, *child_widths; /* LIST columns */
  duckdb_data_chunk chunk; /* reused: duckdb_append_data_chunk copies */
} glue_sink;

static int32_t vector_width(duckdb_logical_type lt) {
  const duckdb_type t = duckdb_get_type_id(lt);
  switch (t) {
    case DUCKDB_TYPE_BOOLEAN: case DUCKDB_TYPE_TINYINT: case DUCKDB_TYPE_UTINYINT: return 1;
    case DUCKDB_TYPE_SMALLINT: case DUCKDB_TYPE_USMALLINT: return 2;
    case DUCKDB_TYPE_INTEGER: case DUCKDB_TYPE_UINTEGER: case DUCKDB_TYPE_FLOAT: case DUCKDB_TYPE_DATE: return 4;
    case DUCKDB_TYPE_DECIMAL: { const int w = duckdb_decimal_width(lt); return w <= 4 ? 2 : w <= 9 ? 4 : w <= 18 ? 8 : 16; }
    case DUCKDB_TYPE_VARCHAR: case DUCKDB_TYPE_BLOB: case DUCKDB_TYPE_INTERVAL: case DUCKDB_TYPE_HUGEINT: case DUCKDB_TYPE_UHUGEINT: case DUCKDB_TYPE_UUID:
    case DUCKDB_TYPE_LIST: return 16; /* LIST: duckdb_list_entry */
    default: return 8;
  }
}

/* `count` rows of values + mask into vector v */
static void fill_vector(duckdb_vector v, int32_t type_id, int32_t width, uint64_t count, const void *data, const uint64_t *mask) {
  const int is_str = type_id == DUCKDB_TYPE_VARCHAR || type_id == DUCKDB_TYPE_BLOB;
  if (!is_str) {
    if (count) memcpy(duckdb_vector_get_data(v), data, (size_t)count * (size_t)width);
  } else { /* the vector must own its strings: inlined entries are copied as they are, pointer entries assigned */
    const dmb_string_t *e = (const dmb_string_t *)data;
    dmb_string_t *out = (dmb_string_t *)duckdb_vector_get_data(v);
    for (uint64_t i = 0; i < count; i++) {
      if (mask && !((mask[i >> 6] >> (i & 63)) & 1ull)) continue;
      if (e[i].length <= 12) out[i] = e[i];
      else duckdb_vector_assign_string_element_len(v, i, (const char *)(uintptr_t)e[i].tail.ptr, e[i].length);
    }
  }
  if (mask) {
    duckdb_vector_ensure_validity_writable(v);
    memcpy(duckdb_vector_get_validity(v), mask, 8 * (((size_t)count + 63) / 64));
  }
}

static int32_t sink_chunk(void *user, int32_t ncols, uint32_t count, const void *const *vec_data, const uint64_t *const *vec_validity) {
  glue_sink *s = (glue_sink *)user;
  if (ncols != s->ncols) return 0;
  for (int32_t c = 0; c < ncols; c++) {
    duckdb_vector v = duckdb_data_chunk_get_vector(s->chunk, (idx_t)c);
    fill_vector(v, s->type_ids[c], s->widths[c], count, vec_data[c], vec_validity[c]);
    if (s->type_ids[c] == DUCKDB_TYPE_LIST) { /* the entries index this chunk's own child vector */
      const void *cdata = NULL;
      const uint64_t *cmask = NULL;
      uint64_t size = 0;
      if (!duckdb_mb_gpu_appender_list_child(s->lib, c, &cdata, &cmask, &size)) return 0;
      /* every call sets the size: the chunk is reused; the child is fetched after reserve, which may reallocate it */
      if (duckdb_list_vector_reserve(v, (idx_t)size) != DuckDBSuccess || duckdb_list_vector_set_size(v, (idx_t)size) != DuckDBSuccess) return 0;
      duckdb_vector child = duckdb_list_vector_get_child(v);
      if (!child) return 0;
      fill_vector(child, s->child_type_ids[c], s->child_widths[c], size, cdata, cmask);
    }
  }
  duckdb_data_chunk_set_size(s->chunk, count);
  return duckdb_append_data_chunk(s->appender, s->chunk) == DuckDBSuccess ? 1 : 0;
}

static int32_t sink_flush(void *user) { return duckdb_appender_flush(((glue_sink *)user)->appender) == DuckDBSuccess ? 1 : 0; }

static void sink_destroy(void *user) {
  glue_sink *s = (glue_sink *)user;
  if (!s) return;
  if (s->chunk) duckdb_destroy_data_chunk(&s->chunk);
  for (int32_t c = 0; c < s->ncols; c++) duckdb_destroy_logical_type(&s->types[c]);
  if (s->appender) duckdb_appender_destroy(&s->appender); /* (flushes what is left, like the reference's destroy :1083-1091) */
  free(s->types); free(s->type_ids); free(s->widths); free(s->child_type_ids); free(s->child_widths); free(s);
}

/* src/duckdb_native.c:1032-1081: NULL on failure (the reference sets no global error here either) */
duckdb_mb_appender *duckdb_mb_appender_create(duckdb_mb_connection *handle, moonbit_bytes_t schema, moonbit_bytes_t table) {
  if (!handle) return NULL;
  duckdb_mb_gpu_ctx *ctx = glue_ctx();
  if (!ctx) return NULL;
  char *schema_c = bytes_to_cstr(schema);
  if (!schema_c) return NULL;
  char *table_c = bytes_to_cstr(table);
  if (!table_c) { free(schema_c); return NULL; }
  glue_sink *s = (glue_sink *)calloc(1, sizeof(glue_sink));
  if (!s) { free(schema_c); free(table_c); return NULL; }
  duckdb_state state = duckdb_appender_create(handle->conn, schema_c[0] ? schema_c : NULL, table_c, &s->appender);
  free(schema_c);
  free(table_c);
  if (state != DuckDBSuccess) { sink_destroy(s); return NULL; }
  s->ncols = (int32_t)duckdb_appender_column_count(s->appender);
  const size_t nc = (size_t)(s->ncols > 0 ? s->ncols : 1);
  s->types = (duckdb_logical_type *)calloc(nc, sizeof(duckdb_logical_type));
  s->type_ids = (int32_t *)calloc(nc, sizeof(int32_t));
  s->widths = (int32_t *)calloc(nc, sizeof(int32_t));
  s->child_type_ids = (int32_t *)calloc(nc, sizeof(int32_t));
  s->child_widths = (int32_t *)calloc(nc, sizeof(int32_t));
  for (int32_t c = 0; c < s->ncols; c++) {
    s->types[c] = duckdb_appender_column_type(s->appender, (idx_t)c);
    s->type_ids[c] = (int32_t)duckdb_get_type_id(s->types[c]);
    s->widths[c] = vector_width(s->types[c]);
  }
  s->chunk = duckdb_create_data_chunk(s->types, (idx_t)s->ncols);
  duckdb_mb_appender *a = duckdb_mb_gpu_appender_create(ctx, s->ncols, s->type_ids, sink_chunk, s);
  if (!a) { sink_destroy(s); return NULL; }
  s->lib = a;
  duckdb_mb_gpu_appender_set_hooks(a, sink_flush, sink_destroy);
  for (int32_t c = 0; c < s->ncols; c++) {
    if (s->type_ids[c] == DUCKDB_TYPE_DECIMAL)
      duckdb_mb_gpu_appender_set_decimal(a, c, duckdb_decimal_width(s->types[c]), duckdb_decimal_scale(s->types[c]));
    if (s->type_ids[c] == DUCKDB_TYPE_LIST) {
      /* a child type the library refuses (LIST, STRUCT, ...) leaves the column undeclared: Arrow batches for it fail */
      duckdb_logical_type child = duckdb_list_type_child_type(s->types[c]);
      const duckdb_type ct = duckdb_get_type_id(child);
      s->child_type_ids[c] = (int32_t)ct;
      s->child_widths[c] = vector_width(child);
      duckdb_mb_gpu_appender_set_list(a, c, (int32_t)ct, ct == DUCKDB_TYPE_DECIMAL ? duckdb_decimal_width(child) : 0,
                                      ct == DUCKDB_TYPE_DECIMAL ? duckdb_decimal_scale(child) : 0);
      duckdb_destroy_logical_type(&child);
    }
  }
  return a;
}

/* tests / embedding hosts: drop the process-wide context (pools, streams) */
void duckdb_mb_glue_shutdown(void) {
  if (g_ctx) { duckdb_mb_gpu_ctx_destroy(g_ctx); g_ctx = NULL; }
}
