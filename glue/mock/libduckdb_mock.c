/*
 * libduckdb_mock.c — a stand-in for libduckdb that serves CANNED DataChunks (test infrastructure).
 *
 * The glue (glue/duckdb_gpu_glue.c) talks to DuckDB only through the C API declared in glue/mock/duckdb.h.  This
 * file implements that subset over tables a test registers: `duckdb_query(conn, sql)` looks the SQL text up in the
 * registry and the result hands out the registered vectors (payload, validity mask or NULL, duckdb_string_t with real
 * pointers, ENUM dictionaries, LIST child vectors) chunk by chunk — the layouts of SURVEY.md Appendix A.  The appender
 * side records every chunk passed to duckdb_append_data_chunk so the test can read back what reached the "table".
 * No SQL is parsed or executed here.
 */
#include "duckdb.h"

#include <stdlib.h>
#include <string.h>

#define MOCK_VECTOR_SIZE 2048

typedef struct {
  const char *name;
  int32_t type_id;
  int32_t width;                         /* bytes per row of the vector payload */
  int32_t dec_width, dec_scale;
  const void *const *data;               /* [nchunks] */
  const uint64_t *const *validity;       /* [nchunks] or NULL */
  uint32_t dict_size;                    /* ENUM */
  const char *const *dict_values;
  int32_t child_type_id, child_width;    /* LIST */
  const void *const *child_data;
  const uint64_t *const *child_validity;
  const uint64_t *child_sizes;
} duckdb_mock_column;

typedef struct mock_table {
  char *sql;
  int32_t ncols;
  duckdb_mock_column *cols;
  int64_t nchunks;
  uint32_t *counts;
  int64_t nrows;
  struct mock_table *next;
} mock_table;

static mock_table *g_tables = NULL;

typedef struct {
  int32_t type_id, dec_width, dec_scale, internal;
  const duckdb_mock_column *col;                   /* served columns */
  int32_t child_type_id, child_dec_width, child_dec_scale;  /* appender LIST columns */
} mock_ltype;
typedef struct { const mock_table *t; int64_t next_chunk; char error[128]; } mock_result;
typedef struct mock_vec {
  const duckdb_mock_column *col;  /* served vector */
  int64_t chunk;
  int is_child;
  struct mock_vec *child;         /* LIST: the chunk's child vector */
  /* created (appender side) vector */
  int created;
  mock_ltype ltype;
  uint8_t *buf;
  uint64_t *mask;
  char **strs;  /* owned copies of assigned strings */
  idx_t cap;    /* rows buf holds: MOCK_VECTOR_SIZE, or a LIST child's reserved size */
  idx_t list_size;
} mock_vec;
typedef struct { const mock_table *t; int64_t k; int32_t ncols; mock_vec *vecs; mock_vec *children; idx_t size; int created; } mock_chunk;

/* ---- registry (called by the tests through ctypes) */
int32_t duckdb_mock_register_table(const char *sql, int32_t ncols, const duckdb_mock_column *cols, int64_t nchunks, const uint32_t *counts) {
  mock_table *t = (mock_table *)calloc(1, sizeof(mock_table));
  t->sql = strdup(sql);
  t->ncols = ncols;
  t->cols = (duckdb_mock_column *)malloc(sizeof(duckdb_mock_column) * (size_t)(ncols > 0 ? ncols : 1));
  memcpy(t->cols, cols, sizeof(duckdb_mock_column) * (size_t)ncols);
  for (int32_t c = 0; c < ncols; c++) t->cols[c].name = strdup(cols[c].name ? cols[c].name : "");
  t->nchunks = nchunks;
  t->counts = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)(nchunks > 0 ? nchunks : 1));
  for (int64_t k = 0; k < nchunks; k++) { t->counts[k] = counts[k]; t->nrows += counts[k]; }
  t->next = g_tables;
  g_tables = t;
  return 1;
}

void duckdb_mock_reset(void) {
  while (g_tables) {
    mock_table *t = g_tables;
    g_tables = t->next;
    for (int32_t c = 0; c < t->ncols; c++) free((void *)t->cols[c].name);
    free(t->cols); free(t->counts); free(t->sql); free(t);
  }
}

static const mock_table *find_table(const char *sql) {
  for (const mock_table *t = g_tables; t; t = t->next)
    if (strcmp(t->sql, sql) == 0) return t;
  return NULL;
}

/* ---- query side */
duckdb_state duckdb_query(duckdb_connection connection, const char *query, duckdb_result *out_result) {
  (void)connection;
  memset(out_result, 0, sizeof(*out_result));
  mock_result *r = (mock_result *)calloc(1, sizeof(mock_result));
  out_result->internal_data = r;
  r->t = find_table(query);
  if (!r->t) {
    strcpy(r->error, "Parser Error: syntax error at or near \"");
    strncat(r->error, query, 40);
    strcat(r->error, "\"");
    return DuckDBError;
  }
  return DuckDBSuccess;
}
void duckdb_destroy_result(duckdb_result *result) { if (result) { free(result->internal_data); result->internal_data = NULL; } }
const char *duckdb_result_error(duckdb_result *result) {
  mock_result *r = result ? (mock_result *)result->internal_data : NULL;
  return (r && r->error[0]) ? r->error : NULL;
}
idx_t duckdb_column_count(duckdb_result *result) { mock_result *r = (mock_result *)result->internal_data; return r && r->t ? (idx_t)r->t->ncols : 0; }
idx_t duckdb_row_count(duckdb_result *result) { mock_result *r = (mock_result *)result->internal_data; return r && r->t ? (idx_t)r->t->nrows : 0; }
const char *duckdb_column_name(duckdb_result *result, idx_t col) {
  mock_result *r = (mock_result *)result->internal_data;
  return (r && r->t && col < (idx_t)r->t->ncols) ? r->t->cols[col].name : NULL;
}
duckdb_type duckdb_column_type(duckdb_result *result, idx_t col) {
  mock_result *r = (mock_result *)result->internal_data;
  return (r && r->t && col < (idx_t)r->t->ncols) ? (duckdb_type)r->t->cols[col].type_id : DUCKDB_TYPE_INVALID;
}
static duckdb_type internal_of_width(int w) { return w == 2 ? DUCKDB_TYPE_SMALLINT : w == 4 ? DUCKDB_TYPE_INTEGER : w == 8 ? DUCKDB_TYPE_BIGINT : DUCKDB_TYPE_HUGEINT; }
duckdb_logical_type duckdb_column_logical_type(duckdb_result *result, idx_t col) {
  mock_result *r = (mock_result *)result->internal_data;
  if (!r || !r->t || col >= (idx_t)r->t->ncols) return NULL;
  const duckdb_mock_column *c = &r->t->cols[col];
  mock_ltype *lt = (mock_ltype *)calloc(1, sizeof(mock_ltype));
  lt->type_id = c->type_id; lt->dec_width = c->dec_width; lt->dec_scale = c->dec_scale; lt->internal = internal_of_width(c->width); lt->col = c;
  return (duckdb_logical_type)lt;
}
duckdb_data_chunk duckdb_fetch_chunk(duckdb_result result) {
  mock_result *r = (mock_result *)result.internal_data;
  if (!r || !r->t || r->next_chunk >= r->t->nchunks) return NULL;
  mock_chunk *ch = (mock_chunk *)calloc(1, sizeof(mock_chunk));
  ch->t = r->t; ch->k = r->next_chunk++; ch->ncols = r->t->ncols; ch->size = r->t->counts[ch->k];
  ch->vecs = (mock_vec *)calloc((size_t)(ch->ncols > 0 ? ch->ncols : 1), sizeof(mock_vec));
  ch->children = (mock_vec *)calloc((size_t)(ch->ncols > 0 ? ch->ncols : 1), sizeof(mock_vec));
  for (int32_t c = 0; c < ch->ncols; c++) {
    ch->vecs[c].col = &r->t->cols[c]; ch->vecs[c].chunk = ch->k;
    ch->children[c].col = &r->t->cols[c]; ch->children[c].chunk = ch->k; ch->children[c].is_child = 1;
    ch->vecs[c].child = &ch->children[c];
  }
  return (duckdb_data_chunk)ch;
}
idx_t duckdb_data_chunk_get_size(duckdb_data_chunk chunk) { return chunk ? ((mock_chunk *)chunk)->size : 0; }
idx_t duckdb_data_chunk_get_column_count(duckdb_data_chunk chunk) { return chunk ? (idx_t)((mock_chunk *)chunk)->ncols : 0; }
duckdb_vector duckdb_data_chunk_get_vector(duckdb_data_chunk chunk, idx_t col_idx) {
  mock_chunk *ch = (mock_chunk *)chunk;
  return (ch && col_idx < (idx_t)ch->ncols) ? (duckdb_vector)&ch->vecs[col_idx] : NULL;
}
static void free_created_vec(mock_vec *v) {
  if (!v->created) return;
  free(v->buf); free(v->mask);
  if (v->strs) { for (idx_t i = 0; i < v->cap; i++) free(v->strs[i]); free(v->strs); }
  if (v->child) { free_created_vec(v->child); free(v->child); }
}
void duckdb_destroy_data_chunk(duckdb_data_chunk *chunk) {
  if (!chunk || !*chunk) return;
  mock_chunk *ch = (mock_chunk *)*chunk;
  for (int32_t c = 0; c < ch->ncols; c++) free_created_vec(&ch->vecs[c]);
  free(ch->vecs); free(ch->children); free(ch);
  *chunk = NULL;
}
void *duckdb_vector_get_data(duckdb_vector vector) {
  mock_vec *v = (mock_vec *)vector;
  if (v->created) return v->buf;
  return (void *)(v->is_child ? v->col->child_data[v->chunk] : v->col->data[v->chunk]);
}
uint64_t *duckdb_vector_get_validity(duckdb_vector vector) {
  mock_vec *v = (mock_vec *)vector;
  if (v->created) return v->mask;
  const uint64_t *const *m = v->is_child ? v->col->child_validity : v->col->validity;
  return m ? (uint64_t *)m[v->chunk] : NULL;
}
duckdb_vector duckdb_list_vector_get_child(duckdb_vector vector) {
  mock_vec *v = (mock_vec *)vector;
  if (v && v->created) return (duckdb_vector)v->child;
  return (v && !v->is_child && v->col->child_data) ? (duckdb_vector)v->child : NULL;
}
idx_t duckdb_list_vector_get_size(duckdb_vector vector) {
  mock_vec *v = (mock_vec *)vector;
  if (v->created) return v->list_size;
  return v->col->child_sizes ? v->col->child_sizes[v->chunk] : 0;
}

/* ---- logical types */
duckdb_type duckdb_get_type_id(duckdb_logical_type type) { return type ? (duckdb_type)((mock_ltype *)type)->type_id : DUCKDB_TYPE_INVALID; }
uint8_t duckdb_decimal_width(duckdb_logical_type type) { return (uint8_t)((mock_ltype *)type)->dec_width; }
uint8_t duckdb_decimal_scale(duckdb_logical_type type) { return (uint8_t)((mock_ltype *)type)->dec_scale; }
duckdb_type duckdb_decimal_internal_type(duckdb_logical_type type) { return (duckdb_type)((mock_ltype *)type)->internal; }
duckdb_type duckdb_enum_internal_type(duckdb_logical_type type) {
  const duckdb_mock_column *c = ((mock_ltype *)type)->col;
  return c->width == 1 ? DUCKDB_TYPE_UTINYINT : c->width == 2 ? DUCKDB_TYPE_USMALLINT : DUCKDB_TYPE_UINTEGER;
}
uint32_t duckdb_enum_dictionary_size(duckdb_logical_type type) { return ((mock_ltype *)type)->col->dict_size; }
char *duckdb_enum_dictionary_value(duckdb_logical_type type, idx_t index) { return strdup(((mock_ltype *)type)->col->dict_values[index]); }
duckdb_logical_type duckdb_list_type_child_type(duckdb_logical_type type) {
  const mock_ltype *t = (const mock_ltype *)type;
  if (!t->col) { /* an appender column's type */
    if (t->child_type_id == DUCKDB_TYPE_DECIMAL) return duckdb_create_decimal_type((uint8_t)t->child_dec_width, (uint8_t)t->child_dec_scale);
    return duckdb_create_logical_type((duckdb_type)t->child_type_id);
  }
  const duckdb_mock_column *c = t->col;
  mock_ltype *lt = (mock_ltype *)calloc(1, sizeof(mock_ltype));
  lt->type_id = c->child_type_id; lt->internal = internal_of_width(c->child_width); lt->col = c;
  return (duckdb_logical_type)lt;
}
duckdb_logical_type duckdb_create_logical_type(duckdb_type type) {
  mock_ltype *lt = (mock_ltype *)calloc(1, sizeof(mock_ltype));
  lt->type_id = (int32_t)type;
  return (duckdb_logical_type)lt;
}
duckdb_logical_type duckdb_create_decimal_type(uint8_t width, uint8_t scale) {
  mock_ltype *lt = (mock_ltype *)calloc(1, sizeof(mock_ltype));
  lt->type_id = DUCKDB_TYPE_DECIMAL; lt->dec_width = width; lt->dec_scale = scale;
  lt->internal = width <= 4 ? DUCKDB_TYPE_SMALLINT : width <= 9 ? DUCKDB_TYPE_INTEGER : width <= 18 ? DUCKDB_TYPE_BIGINT : DUCKDB_TYPE_HUGEINT;
  return (duckdb_logical_type)lt;
}
void duckdb_destroy_logical_type(duckdb_logical_type *type) { if (type && *type) { free(*type); *type = NULL; } }
void duckdb_free(void *ptr) { free(ptr); }

/* ---- appender side: a "table" = its column types + every chunk that was appended */
typedef struct { int32_t type_id, dec_width, dec_scale, child_type_id, child_dec_width, child_dec_scale; } mock_coltype;
typedef struct appended_chunk {
  idx_t size;
  uint8_t **data;
  uint64_t **mask;
  uint8_t **child_data;  /* LIST columns: the chunk's child vector */
  uint64_t **child_mask;
  idx_t *child_size;
  struct appended_chunk *next;
} appended_chunk;
typedef struct mock_append_table {
  char *schema, *table;
  int32_t ncols;
  mock_coltype *types;
  appended_chunk *head, *tail;
  int64_t nchunks, nrows, flushes;
  struct mock_append_table *next;
} mock_append_table;
static mock_append_table *g_append_tables = NULL;
typedef struct { mock_append_table *t; char error[128]; } mock_appender;

int32_t duckdb_mock_register_append_table(const char *schema, const char *table, int32_t ncols, const int32_t *type_ids,
                                          const int32_t *dec_widths, const int32_t *dec_scales) {
  mock_append_table *t = (mock_append_table *)calloc(1, sizeof(mock_append_table));
  t->schema = strdup(schema ? schema : ""); t->table = strdup(table);
  t->ncols = ncols;
  t->types = (mock_coltype *)calloc((size_t)ncols, sizeof(mock_coltype));
  for (int32_t c = 0; c < ncols; c++) { t->types[c].type_id = type_ids[c]; t->types[c].dec_width = dec_widths ? dec_widths[c] : 0; t->types[c].dec_scale = dec_scales ? dec_scales[c] : 0; }
  t->next = g_append_tables;
  g_append_tables = t;
  return 1;
}
static mock_append_table *find_append_table(const char *table) {
  for (mock_append_table *t = g_append_tables; t; t = t->next)
    if (strcmp(t->table, table) == 0) return t;
  return NULL;
}
/* the child type of a registered LIST column (what duckdb_list_type_child_type reports for it) */
int32_t duckdb_mock_set_append_list_child(const char *table, int32_t col, int32_t child_type, int32_t dec_width, int32_t dec_scale) {
  mock_append_table *t = find_append_table(table);
  if (!t || col < 0 || col >= t->ncols) return 0;
  t->types[col].child_type_id = child_type; t->types[col].child_dec_width = dec_width; t->types[col].child_dec_scale = dec_scale;
  return 1;
}
static int type_width(int32_t type_id, int32_t dec_width) {
  switch (type_id) {
    case DUCKDB_TYPE_BOOLEAN: case DUCKDB_TYPE_TINYINT: case DUCKDB_TYPE_UTINYINT: return 1;
    case DUCKDB_TYPE_SMALLINT: case DUCKDB_TYPE_USMALLINT: return 2;
    case DUCKDB_TYPE_INTEGER: case DUCKDB_TYPE_UINTEGER: case DUCKDB_TYPE_FLOAT: case DUCKDB_TYPE_DATE: return 4;
    case DUCKDB_TYPE_DECIMAL: return dec_width <= 4 ? 2 : dec_width <= 9 ? 4 : dec_width <= 18 ? 8 : 16;
    case DUCKDB_TYPE_VARCHAR: case DUCKDB_TYPE_BLOB: case DUCKDB_TYPE_INTERVAL: case DUCKDB_TYPE_HUGEINT: case DUCKDB_TYPE_UHUGEINT: case DUCKDB_TYPE_UUID:
    case DUCKDB_TYPE_LIST: return 16;
    default: return 8;
  }
}
duckdb_state duckdb_appender_create(duckdb_connection connection, const char *schema, const char *table, duckdb_appender *out_appender) {
  (void)connection; (void)schema;
  mock_appender *a = (mock_appender *)calloc(1, sizeof(mock_appender));
  *out_appender = (duckdb_appender)a;
  a->t = find_append_table(table);
  if (!a->t) { strcpy(a->error, "Catalog Error: Table does not exist!"); return DuckDBError; }
  return DuckDBSuccess;
}
idx_t duckdb_appender_column_count(duckdb_appender appender) { mock_appender *a = (mock_appender *)appender; return a && a->t ? (idx_t)a->t->ncols : 0; }
duckdb_logical_type duckdb_appender_column_type(duckdb_appender appender, idx_t col_idx) {
  mock_appender *a = (mock_appender *)appender;
  if (!a || !a->t || col_idx >= (idx_t)a->t->ncols) return NULL;
  const mock_coltype *ct = &a->t->types[col_idx];
  if (ct->type_id == DUCKDB_TYPE_DECIMAL) return duckdb_create_decimal_type((uint8_t)ct->dec_width, (uint8_t)ct->dec_scale);
  mock_ltype *lt = (mock_ltype *)duckdb_create_logical_type((duckdb_type)ct->type_id);
  lt->child_type_id = ct->child_type_id; lt->child_dec_width = ct->child_dec_width; lt->child_dec_scale = ct->child_dec_scale;
  return (duckdb_logical_type)lt;
}
const char *duckdb_appender_error(duckdb_appender appender) { mock_appender *a = (mock_appender *)appender; return a && a->error[0] ? a->error : NULL; }
duckdb_state duckdb_appender_flush(duckdb_appender appender) { mock_appender *a = (mock_appender *)appender; if (!a || !a->t) return DuckDBError; a->t->flushes++; return DuckDBSuccess; }
duckdb_state duckdb_appender_destroy(duckdb_appender *appender) { if (appender && *appender) { free(*appender); *appender = NULL; } return DuckDBSuccess; }

duckdb_data_chunk duckdb_create_data_chunk(duckdb_logical_type *types, idx_t column_count) {
  mock_chunk *ch = (mock_chunk *)calloc(1, sizeof(mock_chunk));
  ch->created = 1; ch->ncols = (int32_t)column_count;
  ch->vecs = (mock_vec *)calloc((size_t)(column_count ? column_count : 1), sizeof(mock_vec));
  for (idx_t c = 0; c < column_count; c++) {
    mock_vec *v = &ch->vecs[c];
    v->created = 1;
    v->ltype = *(mock_ltype *)types[c];
    v->cap = MOCK_VECTOR_SIZE;
    v->buf = (uint8_t *)calloc(MOCK_VECTOR_SIZE, (size_t)type_width(v->ltype.type_id, v->ltype.dec_width));
    if (v->ltype.type_id == DUCKDB_TYPE_LIST) { /* an empty child vector, grown by duckdb_list_vector_reserve */
      v->child = (mock_vec *)calloc(1, sizeof(mock_vec));
      v->child->created = 1;
      v->child->is_child = 1;
      v->child->ltype.type_id = v->ltype.child_type_id;
      v->child->ltype.dec_width = v->ltype.child_dec_width;
      v->child->ltype.dec_scale = v->ltype.child_dec_scale;
    }
  }
  return (duckdb_data_chunk)ch;
}
duckdb_state duckdb_list_vector_reserve(duckdb_vector vector, idx_t required_capacity) {
  mock_vec *v = (mock_vec *)vector;
  if (!v || !v->created || !v->child) return DuckDBError;
  mock_vec *c = v->child;
  if (required_capacity <= c->cap) return DuckDBSuccess;
  idx_t cap = c->cap * 2 > required_capacity ? c->cap * 2 : required_capacity;
  const size_t w = (size_t)type_width(c->ltype.type_id, c->ltype.dec_width);
  c->buf = (uint8_t *)realloc(c->buf, cap * w);
  memset(c->buf + c->cap * w, 0, (cap - c->cap) * w);
  if (c->mask) { /* new rows are valid */
    const size_t old_words = (c->cap + 63) / 64, words = (cap + 63) / 64;
    c->mask = (uint64_t *)realloc(c->mask, 8 * words);
    memset(c->mask + old_words, 0xff, 8 * (words - old_words));
    if (c->cap & 63) c->mask[old_words - 1] |= ~0ull << (c->cap & 63);
  }
  if (c->strs) { c->strs = (char **)realloc(c->strs, cap * sizeof(char *)); memset(c->strs + c->cap, 0, (cap - c->cap) * sizeof(char *)); }
  c->cap = cap;
  return DuckDBSuccess;
}
duckdb_state duckdb_list_vector_set_size(duckdb_vector vector, idx_t size) {
  mock_vec *v = (mock_vec *)vector;
  if (!v || !v->created || !v->child || size > v->child->cap) return DuckDBError;
  v->list_size = size;
  return DuckDBSuccess;
}
void duckdb_data_chunk_set_size(duckdb_data_chunk chunk, idx_t size) { ((mock_chunk *)chunk)->size = size; }
void duckdb_vector_ensure_validity_writable(duckdb_vector vector) {
  mock_vec *v = (mock_vec *)vector;
  if (v->created && !v->mask) {
    const size_t words = v->cap ? (v->cap + 63) / 64 : 1;
    v->mask = (uint64_t *)malloc(8 * words);
    memset(v->mask, 0xff, 8 * words);
  }
}
void duckdb_vector_assign_string_element_len(duckdb_vector vector, idx_t index, const char *str, idx_t str_len) {
  mock_vec *v = (mock_vec *)vector;
  if (!v->created || index >= v->cap) return;
  duckdb_string_t *e = (duckdb_string_t *)v->buf + index;
  memset(e, 0, sizeof(*e));
  e->value.inlined.length = (uint32_t)str_len;
  if (str_len <= 12) { memcpy(e->value.inlined.inlined, str, str_len); return; }
  if (!v->strs) v->strs = (char **)calloc(v->cap, sizeof(char *));
  free(v->strs[index]);
  v->strs[index] = (char *)malloc(str_len);
  memcpy(v->strs[index], str, str_len);
  memcpy(e->value.pointer.prefix, str, 4);
  e->value.pointer.ptr = v->strs[index];
}
duckdb_state duckdb_append_data_chunk(duckdb_appender appender, duckdb_data_chunk chunk) {
  mock_appender *a = (mock_appender *)appender;
  mock_chunk *ch = (mock_chunk *)chunk;
  if (!a || !a->t || !ch || ch->ncols != a->t->ncols) return DuckDBError;
  appended_chunk *ac = (appended_chunk *)calloc(1, sizeof(appended_chunk));
  ac->size = ch->size;
  ac->data = (uint8_t **)calloc((size_t)ch->ncols, sizeof(uint8_t *));
  ac->mask = (uint64_t **)calloc((size_t)ch->ncols, sizeof(uint64_t *));
  ac->child_data = (uint8_t **)calloc((size_t)ch->ncols, sizeof(uint8_t *));
  ac->child_mask = (uint64_t **)calloc((size_t)ch->ncols, sizeof(uint64_t *));
  ac->child_size = (idx_t *)calloc((size_t)ch->ncols, sizeof(idx_t));
  for (int32_t c = 0; c < ch->ncols; c++) {
    mock_vec *v = &ch->vecs[c];
    const int w = type_width(a->t->types[c].type_id, a->t->types[c].dec_width);
    const int is_str = a->t->types[c].type_id == DUCKDB_TYPE_VARCHAR || a->t->types[c].type_id == DUCKDB_TYPE_BLOB;
    ac->data[c] = (uint8_t *)malloc((size_t)MOCK_VECTOR_SIZE * (size_t)w);
    memcpy(ac->data[c], v->buf, (size_t)MOCK_VECTOR_SIZE * (size_t)w);
    if (v->mask) { ac->mask[c] = (uint64_t *)malloc(8 * (MOCK_VECTOR_SIZE / 64)); memcpy(ac->mask[c], v->mask, 8 * (MOCK_VECTOR_SIZE / 64)); }
    if (is_str) { /* the table owns its strings: copy what the pointers refer to */
      duckdb_string_t *e = (duckdb_string_t *)ac->data[c];
      for (idx_t i = 0; i < ch->size; i++) {
        if (ac->mask[c] && !((ac->mask[c][i >> 6] >> (i & 63)) & 1ull)) continue;
        if (e[i].value.inlined.length > 12) {
          char *copy = (char *)malloc(e[i].value.pointer.length);
          memcpy(copy, e[i].value.pointer.ptr, e[i].value.pointer.length);
          e[i].value.pointer.ptr = copy; /* (leaked with the table: test process) */
        }
      }
    }
    if (v->child) { /* LIST: the child vector, its first list_size rows */
      const mock_vec *cv = v->child;
      const idx_t size = v->list_size;
      const size_t cw = (size_t)type_width(cv->ltype.type_id, cv->ltype.dec_width), words = (size + 63) / 64;
      ac->child_size[c] = size;
      ac->child_data[c] = (uint8_t *)malloc(size * cw + 1);
      if (size) memcpy(ac->child_data[c], cv->buf, size * cw);
      if (cv->mask) { ac->child_mask[c] = (uint64_t *)malloc(8 * words + 8); memcpy(ac->child_mask[c], cv->mask, 8 * words); }
      if (cv->ltype.type_id == DUCKDB_TYPE_VARCHAR || cv->ltype.type_id == DUCKDB_TYPE_BLOB) {
        duckdb_string_t *e = (duckdb_string_t *)ac->child_data[c];
        for (idx_t i = 0; i < size; i++) {
          if (ac->child_mask[c] && !((ac->child_mask[c][i >> 6] >> (i & 63)) & 1ull)) continue;
          if (e[i].value.inlined.length > 12) {
            char *copy = (char *)malloc(e[i].value.pointer.length);
            memcpy(copy, e[i].value.pointer.ptr, e[i].value.pointer.length);
            e[i].value.pointer.ptr = copy;
          }
        }
      }
    }
  }
  if (a->t->tail) a->t->tail->next = ac; else a->t->head = ac;
  a->t->tail = ac;
  a->t->nchunks++;
  a->t->nrows += (int64_t)ch->size;
  return DuckDBSuccess;
}

/* ---- what reached the table (read back by the tests) */
int64_t duckdb_mock_appended_rows(const char *table) { mock_append_table *t = find_append_table(table); return t ? t->nrows : -1; }
int64_t duckdb_mock_appended_chunks(const char *table) { mock_append_table *t = find_append_table(table); return t ? t->nchunks : -1; }
int64_t duckdb_mock_append_flushes(const char *table) { mock_append_table *t = find_append_table(table); return t ? t->flushes : -1; }
/* chunk k: size, and per column the payload / mask pointers (mask NULL = all valid) */
int64_t duckdb_mock_appended_chunk(const char *table, int64_t k, int32_t col, const void **data, const uint64_t **mask) {
  mock_append_table *t = find_append_table(table);
  if (!t) return -1;
  appended_chunk *ac = t->head;
  for (int64_t i = 0; ac && i < k; i++) ac = ac->next;
  if (!ac || col < 0 || col >= t->ncols) return -1;
  *data = ac->data[col];
  *mask = ac->mask[col];
  return (int64_t)ac->size;
}
/* chunk k, LIST column col: the child vector's values / mask pointers (mask NULL = all valid); returns the child size */
int64_t duckdb_mock_appended_list_child(const char *table, int64_t k, int32_t col, const void **data, const uint64_t **mask) {
  mock_append_table *t = find_append_table(table);
  if (!t) return -1;
  appended_chunk *ac = t->head;
  for (int64_t i = 0; ac && i < k; i++) ac = ac->next;
  if (!ac || col < 0 || col >= t->ncols || !ac->child_data[col]) return -1;
  *data = ac->child_data[col];
  *mask = ac->child_mask[col];
  return (int64_t)ac->child_size[col];
}
