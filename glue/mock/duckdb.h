/*
 * duckdb.h (MOCK) — the subset of DuckDB's public C API that glue/duckdb_gpu_glue.c uses, declared from the API's
 * published documentation so that the glue COMPILES and RUNS in an image that has no libduckdb (SURVEY.md Appendix C).
 * glue/mock/libduckdb_mock.c implements these entry points over canned DataChunks that a test registers.
 * With a real DuckDB installation, point the include path at the real duckdb.h instead: the glue uses nothing else.
 */
#ifndef DUCKDB_MOCK_H
#define DUCKDB_MOCK_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef uint64_t idx_t;
typedef enum { DuckDBSuccess = 0, DuckDBError = 1 } duckdb_state;

typedef enum DUCKDB_TYPE {
  DUCKDB_TYPE_INVALID = 0, DUCKDB_TYPE_BOOLEAN = 1, DUCKDB_TYPE_TINYINT = 2, DUCKDB_TYPE_SMALLINT = 3, DUCKDB_TYPE_INTEGER = 4,
  DUCKDB_TYPE_BIGINT = 5, DUCKDB_TYPE_UTINYINT = 6, DUCKDB_TYPE_USMALLINT = 7, DUCKDB_TYPE_UINTEGER = 8, DUCKDB_TYPE_UBIGINT = 9,
  DUCKDB_TYPE_FLOAT = 10, DUCKDB_TYPE_DOUBLE = 11, DUCKDB_TYPE_TIMESTAMP = 12, DUCKDB_TYPE_DATE = 13, DUCKDB_TYPE_TIME = 14,
  DUCKDB_TYPE_INTERVAL = 15, DUCKDB_TYPE_HUGEINT = 16, DUCKDB_TYPE_VARCHAR = 17, DUCKDB_TYPE_BLOB = 18, DUCKDB_TYPE_DECIMAL = 19,
  DUCKDB_TYPE_TIMESTAMP_S = 20, DUCKDB_TYPE_TIMESTAMP_MS = 21, DUCKDB_TYPE_TIMESTAMP_NS = 22, DUCKDB_TYPE_ENUM = 23,
  DUCKDB_TYPE_LIST = 24, DUCKDB_TYPE_STRUCT = 25, DUCKDB_TYPE_MAP = 26, DUCKDB_TYPE_UUID = 27, DUCKDB_TYPE_UNION = 28,
  DUCKDB_TYPE_BIT = 29, DUCKDB_TYPE_TIME_TZ = 30, DUCKDB_TYPE_TIMESTAMP_TZ = 31, DUCKDB_TYPE_UHUGEINT = 32,
  DUCKDB_TYPE_ARRAY = 33, DUCKDB_TYPE_TIME_NS = 39
} duckdb_type;

typedef struct _duckdb_database { void *internal_ptr; } *duckdb_database;
typedef struct _duckdb_connection { void *internal_ptr; } *duckdb_connection;
typedef struct _duckdb_data_chunk { void *internal_ptr; } *duckdb_data_chunk;
typedef struct _duckdb_vector { void *internal_ptr; } *duckdb_vector;
typedef struct _duckdb_logical_type { void *internal_ptr; } *duckdb_logical_type;
typedef struct _duckdb_appender { void *internal_ptr; } *duckdb_appender;

typedef struct {
  idx_t deprecated_column_count;
  idx_t deprecated_row_count;
  idx_t deprecated_rows_changed;
  void *deprecated_columns;
  char *deprecated_error_message;
  void *internal_data;
} duckdb_result;

typedef struct {
  union {
    struct { uint32_t length; char prefix[4]; char *ptr; } pointer;
    struct { uint32_t length; char inlined[12]; } inlined;
  } value;
} duckdb_string_t;

typedef struct { uint64_t offset; uint64_t length; } duckdb_list_entry;

duckdb_state duckdb_query(duckdb_connection connection, const char *query, duckdb_result *out_result);
void duckdb_destroy_result(duckdb_result *result);
const char *duckdb_result_error(duckdb_result *result);
idx_t duckdb_column_count(duckdb_result *result);
idx_t duckdb_row_count(duckdb_result *result);
const char *duckdb_column_name(duckdb_result *result, idx_t col);
duckdb_type duckdb_column_type(duckdb_result *result, idx_t col);
duckdb_logical_type duckdb_column_logical_type(duckdb_result *result, idx_t col);
duckdb_data_chunk duckdb_fetch_chunk(duckdb_result result);

idx_t duckdb_data_chunk_get_size(duckdb_data_chunk chunk);
idx_t duckdb_data_chunk_get_column_count(duckdb_data_chunk chunk);
duckdb_vector duckdb_data_chunk_get_vector(duckdb_data_chunk chunk, idx_t col_idx);
void duckdb_destroy_data_chunk(duckdb_data_chunk *chunk);
void *duckdb_vector_get_data(duckdb_vector vector);
uint64_t *duckdb_vector_get_validity(duckdb_vector vector);
void duckdb_vector_ensure_validity_writable(duckdb_vector vector);
void duckdb_vector_assign_string_element_len(duckdb_vector vector, idx_t index, const char *str, idx_t str_len);
duckdb_vector duckdb_list_vector_get_child(duckdb_vector vector);
idx_t duckdb_list_vector_get_size(duckdb_vector vector);
duckdb_state duckdb_list_vector_reserve(duckdb_vector vector, idx_t required_capacity);
duckdb_state duckdb_list_vector_set_size(duckdb_vector vector, idx_t size);
duckdb_vector duckdb_struct_vector_get_child(duckdb_vector vector, idx_t index);

duckdb_type duckdb_get_type_id(duckdb_logical_type type);
uint8_t duckdb_decimal_width(duckdb_logical_type type);
uint8_t duckdb_decimal_scale(duckdb_logical_type type);
duckdb_type duckdb_decimal_internal_type(duckdb_logical_type type);
duckdb_type duckdb_enum_internal_type(duckdb_logical_type type);
uint32_t duckdb_enum_dictionary_size(duckdb_logical_type type);
char *duckdb_enum_dictionary_value(duckdb_logical_type type, idx_t index);
duckdb_logical_type duckdb_list_type_child_type(duckdb_logical_type type);
idx_t duckdb_struct_type_child_count(duckdb_logical_type type);
duckdb_logical_type duckdb_struct_type_child_type(duckdb_logical_type type, idx_t index);
duckdb_logical_type duckdb_create_logical_type(duckdb_type type);
duckdb_logical_type duckdb_create_decimal_type(uint8_t width, uint8_t scale);
void duckdb_destroy_logical_type(duckdb_logical_type *type);
void duckdb_free(void *ptr);

duckdb_data_chunk duckdb_create_data_chunk(duckdb_logical_type *types, idx_t column_count);
void duckdb_data_chunk_set_size(duckdb_data_chunk chunk, idx_t size);

duckdb_state duckdb_appender_create(duckdb_connection connection, const char *schema, const char *table, duckdb_appender *out_appender);
idx_t duckdb_appender_column_count(duckdb_appender appender);
duckdb_logical_type duckdb_appender_column_type(duckdb_appender appender, idx_t col_idx);
const char *duckdb_appender_error(duckdb_appender appender);
duckdb_state duckdb_appender_flush(duckdb_appender appender);
duckdb_state duckdb_appender_destroy(duckdb_appender *appender);
duckdb_state duckdb_append_data_chunk(duckdb_appender appender, duckdb_data_chunk chunk);

#ifdef __cplusplus
}
#endif
#endif
