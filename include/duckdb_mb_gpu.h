/*
 * duckdb_mb_gpu.h — C ABI of libduckdb_mb_gpu.so, the B200 (sm_100a) implementation of the
 * result/ingest boundary of the MoonBit DuckDB bindings f4ah6o/duckdb.mbt.
 *
 * Three layers, all `extern "C"`, plain pointers and sizes, no torch / C++ types:
 *
 *   L0  device API   dmb_dev_*        raw device pointers + a cudaStream_t (as void*); one launch
 *                                     converts a whole chunk batch.  bench.py `value`, ncu.
 *   L1  host API     duckdb_mb_gpu_*  HOST DuckDB-shaped chunk vectors in, Arrow C Data / typed
 *                                     columns / reference packed blobs out; pinned staging and
 *                                     cudaMemcpyAsync on streams inside.  bench.py `e2e`.
 *   L2  drop-in      duckdb_mb_arrow_* / duckdb_mb_bytes_to_double — the exact symbols the
 *                                     reference's MoonBit `extern "C"` declarations bind
 *                                     (src/duckdb_arrow_native.mbt:9-104), served from an L1 result.
 *
 * Every entry cites the reference interface (file:line under /root/reference) it replaces.
 */
#ifndef DUCKDB_MB_GPU_H
#define DUCKDB_MB_GPU_H

#include <stddef.h>
#include <stdint.h>

#include "moonbit_standin.h"

#ifdef __cplusplus
extern "C" {
#endif

#define DMB_VECTOR_SIZE 2048 /* DuckDB STANDARD_VECTOR_SIZE; chunks hold <= 2048 rows */
#define DMB_VALIDITY_WORDS 32 /* uint64 words per full vector */

/* ---- DuckDB type ids (duckdb.h DUCKDB_TYPE; the reference mirrors the numbering in
 *      src/duckdb_parsing.mbt:8-52 and switches on it in src/duckdb_native.c:271-303,553-662) */
enum dmb_type {
  DMB_TYPE_INVALID = 0,
  DMB_TYPE_BOOLEAN = 1,
  DMB_TYPE_TINYINT = 2,
  DMB_TYPE_SMALLINT = 3,
  DMB_TYPE_INTEGER = 4,
  DMB_TYPE_BIGINT = 5,
  DMB_TYPE_UTINYINT = 6,
  DMB_TYPE_USMALLINT = 7,
  DMB_TYPE_UINTEGER = 8,
  DMB_TYPE_UBIGINT = 9,
  DMB_TYPE_FLOAT = 10,
  DMB_TYPE_DOUBLE = 11,
  DMB_TYPE_TIMESTAMP = 12,
  DMB_TYPE_DATE = 13,
  DMB_TYPE_TIME = 14,
  DMB_TYPE_INTERVAL = 15,
  DMB_TYPE_HUGEINT = 16,
  DMB_TYPE_VARCHAR = 17,
  DMB_TYPE_BLOB = 18,
  DMB_TYPE_DECIMAL = 19,
  DMB_TYPE_TIMESTAMP_S = 20,
  DMB_TYPE_TIMESTAMP_MS = 21,
  DMB_TYPE_TIMESTAMP_NS = 22,
  DMB_TYPE_ENUM = 23,     /* uint8/16/32 indices into the type's dictionary (dmb_enum_dict) */
  DMB_TYPE_LIST = 24,     /* duckdb_list_entry vectors + one child vector per chunk (dmb_host_list) */
  DMB_TYPE_STRUCT = 25,   /* a validity mask per chunk + one vector per field and chunk (dmb_host_struct) */
  DMB_TYPE_MAP = 26,      /* LIST of STRUCT<key, value>: dmb_host_list whose child_col is a two-field STRUCT */
  DMB_TYPE_UUID = 27,
  DMB_TYPE_TIME_TZ = 30,
  DMB_TYPE_TIMESTAMP_TZ = 31,
  DMB_TYPE_UHUGEINT = 32,
  DMB_TYPE_TIME_NS = 39
};

/* ---- physical payload of a flat vector (duckdb_vector_get_data; reference reads them at
 *      src/duckdb_native.c:553-662) */
enum dmb_phys {
  DMB_PHYS_BOOL = 0, /* 1 B, 0/1 */
  DMB_PHYS_I8 = 1,
  DMB_PHYS_I16 = 2,
  DMB_PHYS_I32 = 3,
  DMB_PHYS_I64 = 4,
  DMB_PHYS_U8 = 5,
  DMB_PHYS_U16 = 6,
  DMB_PHYS_U32 = 7,
  DMB_PHYS_U64 = 8,
  DMB_PHYS_F32 = 9,
  DMB_PHYS_F64 = 10,
  DMB_PHYS_I128 = 11,     /* duckdb_hugeint {uint64 lower, int64 upper} */
  DMB_PHYS_U128 = 12,     /* duckdb_uhugeint / UUID */
  DMB_PHYS_INTERVAL = 13, /* {int32 months, int32 days, int64 micros} */
  DMB_PHYS_STRING = 14,   /* duckdb_string_t, 16 B */
  DMB_PHYS_COUNT = 15
};

/* ---- what a fixed-width column is converted to (kernels K2/K3/K4, SURVEY.md §2.2) */
enum dmb_dst {
  DMB_DST_SAME = 0,       /* Arrow primitive of the same width; NULL slots zeroed            */
  DMB_DST_I32_TRUNC = 1,  /* (int32_t)duckdb_value_int64      src/duckdb_native.c:2379-2387   */
  DMB_DST_I64 = 2,        /* duckdb_value_int64               src/duckdb_native.c:2413-2419   */
  DMB_DST_F64 = 3,        /* duckdb_value_double              src/duckdb_native.c:2445-2451   */
  DMB_DST_BOOL_BYTE = 4,  /* duckdb_value_boolean ? 1 : 0     src/duckdb_native.c:2537-2543   */
  DMB_DST_BOOL_BITS = 5,  /* Arrow bit-packed bool values                                     */
  DMB_DST_I128 = 6,       /* DECIMAL int16/32/64 -> Arrow decimal128 (sign-extend)            */
  DMB_DST_I32_SAT = 7,    /* typed Value::Int: Int32-saturating  src/duckdb_parsing.mbt:203-237 */
  DMB_DST_TS_US_FROM_S = 8,   /* typed Value::Timestamp micros   src/duckdb_parsing.mbt:375-398 */
  DMB_DST_TS_US_FROM_MS = 9,
  DMB_DST_TS_US_FROM_NS = 10, /* floor(ns/1000): fraction truncated to 6 digits :402-417      */
  DMB_DST_MONTH_DAY_NANO = 11, /* INTERVAL -> Arrow month_day_nano_interval                   */
  DMB_DST_DATE_REF = 12,  /* typed Value::Date through the reference's date_to_days, incl. its
                             pre-1970 leap-day defect      src/duckdb_parsing.mbt:318-338      */
  /* typed Value::Timestamp exactly as the reference computes it: text -> parse_timestamp =
     parse_date(date part) * 86400e6 + time of day (src/duckdb_parsing.mbt:375-398), so the
     date_to_days pre-1970 behaviour carries over; the source unit is converted to micros first
     (fraction truncated to 6 digits, :402-417) */
  DMB_DST_TS_REF = 13,
  DMB_DST_TS_REF_FROM_S = 14,
  DMB_DST_TS_REF_FROM_MS = 15,
  DMB_DST_TS_REF_FROM_NS = 16,
  /* DECIMAL columns through the reference getters: libduckdb's duckdb_value_int64 / _double / _boolean cast by the
     LOGICAL type (call sites src/duckdb_native.c:2384,2417,2449,2541), i.e. the stored integer is divided by
     10^scale -- round half away from zero for the integer targets (DuckDB TryCastFromDecimal), value / 10^scale for
     double.  dmb_fixed_job.param carries the scale.  UNPINNED: no reference test reads a DECIMAL through these getters. */
  DMB_DST_DEC_I64 = 17,
  DMB_DST_DEC_I32_TRUNC = 18, /* (int32_t) of the int64 cast, :2384-2385 */
  DMB_DST_DEC_F64 = 19,
  DMB_DST_DEC_BOOL_BYTE = 20, /* rounded integer != 0 */
  DMB_DST_COUNT = 21
};

#define DMB_OP(phys, dst) (((int32_t)(phys) << 8) | (int32_t)(dst))
#define DMB_OP_VALIDITY_ONLY 0x7f00 /* job writes only validity outputs (string columns) */

/* one flat vector of one chunk inside a device-resident column slab */
typedef struct dmb_vec_desc {
  uint64_t data_off; /* byte offset of the vector payload in the column slab (16-B aligned) */
  int64_t val_off;   /* offset in uint64 words of the validity mask in the validity slab,
                        or -1: duckdb_vector_get_validity returned NULL = all valid
                        (reference: src/duckdb_native.c:530-533) */
} dmb_vec_desc;

/* ---- one fixed-width output column of a batch (device pointers) */
typedef struct dmb_fixed_job {
  const void *in_data;         /* column slab */
  const uint64_t *in_validity; /* validity slab (may be NULL when every val_off is -1) */
  const dmb_vec_desc *vecs;    /* [nchunks] */
  void *out_values;            /* contiguous output values (256-B aligned)             */
  uint64_t *out_validity;      /* Arrow LSB bitmap, ceil(n/64) words, or NULL            */
  uint8_t *out_valid_bytes;    /* reference byte-per-row validity (1=valid), or NULL
                                  (src/duckdb_native.c:2594-2606)                        */
  unsigned long long *null_count; /* device counter, incremented; or NULL               */
  int32_t op;                  /* DMB_OP(phys, dst) */
  int32_t param;               /* DMB_DST_DEC_*: the DECIMAL's scale; otherwise 0 */
} dmb_fixed_job;

/* duckdb_string_t, 16 bytes (reference reads it at src/duckdb_native.c:597-603) */
typedef struct dmb_string_t {
  uint32_t length;
  char prefix[4];          /* first 4 bytes of the string (both forms) */
  union {
    char inlined_rest[8];  /* length <= 12: bytes 4..11, unused bytes zero */
    uint64_t ptr;          /* length  > 12: host heap pointer to the whole string */
  } tail;
} dmb_string_t;

enum dmb_string_mode {
  DMB_STR_ARROW_UTF8 = 0,  /* int32 offsets[n+1] + data; NULL rows have zero length          */
  DMB_STR_ARROW_LARGE = 1, /* int64 offsets                                                  */
  DMB_STR_REF_BLOB = 2     /* reference NUL-terminated concatenation, strlen semantics
                              (src/duckdb_native.c:2474-2510): int32 offsets[n+1] + data where
                              every row contributes strnlen(s)+1 bytes and a NULL row a lone \0 */
};

/* ---- one VARCHAR/BLOB output column of a batch (device pointers) */
typedef struct dmb_string_job {
  const dmb_string_t *in;      /* slab of string_t */
  const uint64_t *in_validity;
  const dmb_vec_desc *vecs;    /* data_off in bytes into `in` */
  const uint8_t *heap_dev;     /* device copy of the string heap                          */
  uint64_t heap_host_base;     /* host address the `ptr` fields are relative to: the kernel
                                  rebases dev = heap_dev + (ptr - heap_host_base)          */
  uint64_t heap_len;
  void *out_offsets;           /* int32[n+1] or int64[n+1]                                 */
  uint8_t *out_data;
  uint64_t *out_validity;      /* Arrow bitmap or NULL                                     */
  uint8_t *out_valid_bytes;    /* byte-per-row or NULL                                     */
  unsigned long long *null_count;
  unsigned long long *total_bytes; /* device: final data length                            */
  int32_t mode;
  int32_t reserved;
  uint64_t out_data_cap;       /* bytes `out_data` can hold, or 0: not checked.  string_t entries may ALIAS the same
                                  heap bytes (a flattened dictionary / constant vector does), so the summed lengths are
                                  not bounded by 12 n + heap_len: when the column's total exceeds the capacity no data
                                  byte is written past it, flag 8 is raised (dmb_dev_string_error) and *total_bytes still
                                  holds the exact total, so the caller can allocate and run again */
} dmb_string_job;

/* =====================================================================================
 * L0 — device API.  All pointers are device pointers unless said otherwise; `stream` is a
 * cudaStream_t.  Return 0 on success, negative on error (duckdb_mb_gpu_last_error()).
 * ===================================================================================== */

/* K1+K2+K3+K4 fused: every fixed-width column of a chunk batch in ONE launch.
 *   jobs_dev  device array [njobs]; jobs_host is the host mirror of the same array.  One launch
 *             covers each run of equal `op`, so sort jobs by op: a batch costs one launch per
 *             distinct conversion
 *   counts    device uint32[nchunks] rows per chunk (duckdb_data_chunk_get_size, <= 2048)
 *   row_off   device int64[nchunks+1] exclusive scan of counts
 * Replaces the per-cell loops src/duckdb_native.c:2379-2387,2413-2419,2445-2451,2537-2543,
 * 2597-2606 and the per-cell validity test :520-535. */
int32_t dmb_dev_fixed_batch(const dmb_fixed_job *jobs_dev, const dmb_fixed_job *jobs_host,
                            int32_t njobs, const uint32_t *counts, const int64_t *row_off,
                            int64_t nchunks, int64_t nrows, void *stream);

/* host-side op table: output bytes per value of DMB_OP(phys,dst) (0 = bit-packed), -1 if the
 * pair is not supported; bytes per value of a physical type */
int32_t dmb_op_out_width(int32_t op);
int32_t dmb_phys_width(int32_t phys);

/* K5: string_t -> utf8 offsets + data, single pass over the column (tile scan + decoupled look-back).
 * Arrow modes run string_pack_kernel: a persistent, warp-specialised pipeline whose byte movement in
 * and out of the SM is done by the copy engine (cp.async.bulk / mbarrier, sm_100 byte-masked bulk
 * stores); columns of long strings (> 29 heap bytes per row on average) and DMB_STR_REF_BLOB run the
 * run-gather string_batch_kernel.
 *   scratch   device, >= dmb_dev_string_scratch_bytes(nchunks) bytes, zeroed by the call
 *   layout    every chunk's string_t vector must have DMB_VECTOR_SIZE entries of storage (a DuckDB
 *             vector always has: rows past `count` are never interpreted, but whole tiles are fetched);
 *             `in`, `out_data`, `heap_dev` 16-byte aligned; the heap copy followed by >= 16 readable bytes
 * Replaces src/duckdb_native.c:597-603 (string_t read) and :2474-2510 / :2699-2755. */
size_t dmb_dev_string_scratch_bytes(int64_t nchunks);
/* How long a tile's look-back waits for its predecessors before it gives up with flag 16 (default 4 s; the launch then
 * ends normally, the host reports the error and the context stays usable).  Process-wide per device; a test knob. */
int32_t dmb_dev_set_lookback_limit_ns(unsigned long long ns);
/* error flags raised by the last string launch on `scratch` (0 = none); synchronises `stream`.
 * 1: a tile holds > 4 GiB  2: total exceeds int32 offsets  4: string_t pointer outside the heap
 * 8: total exceeds out_data_cap  16: a look-back gave up waiting (the outputs are not valid) */
int32_t dmb_dev_string_error(const void *scratch, void *stream);
int32_t dmb_dev_string_batch(const dmb_string_job *job, const uint32_t *counts,
                             const int64_t *row_off, int64_t nchunks, int64_t nrows,
                             void *scratch, void *stream);

/* K7: fixed-width cells -> their DuckDB VARCHAR rendering as duckdb_string_t (<= 12 bytes inlined,
 * else prefix + pointer into `out_heap`, one DMB_RENDER_SLOT_BYTES slot per row), so the rendered
 * column can be fed to dmb_dev_string_batch like a VARCHAR column.  Replaces libduckdb's
 * duckdb_value_varchar / duckdb_value_to_string at the reference's call sites
 * src/duckdb_native.c:224-238, :2478, :2715 and :305-318.  Rendered: BOOLEAN, the eight integer
 * types, HUGEINT, UHUGEINT, FLOAT, DOUBLE (shortest round trip), DATE, TIME, TIME_NS, TIMESTAMP / _TZ / _S / _MS / _NS, DECIMAL (any storage). */
#define DMB_RENDER_SLOT_BYTES 48
#define DMB_RENDER_SLOT_BYTES_WIDE 80 /* INTERVAL: up to 70 characters */
typedef struct dmb_render_job {
  const void *in_data;         /* column slab */
  const uint64_t *in_validity; /* validity slab or NULL */
  const dmb_vec_desc *vecs;    /* [nchunks], of the source column */
  dmb_string_t *out;           /* string_t slab: chunk k at k*2048 entries */
  uint8_t *out_heap;           /* nchunks*2048*dmb_render_slot_bytes(type_id) bytes */
  uint64_t heap_host_base;     /* the "host address" written into pointer entries (any value; the
                                  string kernel rebases against the same number) */
  int32_t type_id;             /* enum dmb_type */
  int32_t phys;                /* enum dmb_phys */
  int32_t dec_scale;
  int32_t reserved;
} dmb_render_job;
int32_t dmb_render_supported(int32_t type_id, int32_t phys);
int32_t dmb_render_slot_bytes(int32_t type_id); /* out_heap bytes per row for this type (48, INTERVAL: 80) */
int32_t dmb_dev_render_text(const dmb_render_job *job, const uint32_t *counts, int64_t nchunks, void *stream);

/* BLOB -> text: the VARCHAR cast of a BLOB cell (DuckDB Blob::ToString: printable ASCII except backslash and quotes as it
 * is, every other byte as \xHH).  Input: the dense utf8-style form of the column (int32 offsets[n+1] + data, as produced by
 * dmb_dev_string_batch); output: one string_t per row referring to out_heap (>= 4 * offsets[n] bytes; row i's text at
 * out_heap + 4 * offsets[i]), ready for dmb_dev_string_batch.  Replaces libduckdb's duckdb_value_varchar on a BLOB cell
 * (src/duckdb_native.c:224-238, :2478, :2715; chunk path :604-610).  UNPINNED. */
int32_t dmb_dev_blob_escape(const int32_t *offsets, const uint8_t *data, int64_t nrows, dmb_string_t *out, uint8_t *out_heap,
                            uint64_t heap_host_base, void *stream);

/* K8: ENUM index vectors -> string_t that refer to the dictionary's labels (<= 12 bytes inlined, else
 * prefix + dict_host_base + offset), one 2048-entry slot per chunk; feed the result to
 * dmb_dev_string_batch with the dictionary bytes as the heap.  Rows whose validity bit is clear get a
 * zero string_t; a valid row whose index is >= dict_size is counted in *bad_index and left empty. */
typedef struct dmb_enum_job {
  const void *in_data;            /* index slab                                     */
  const uint64_t *in_validity;    /* validity slab                                  */
  const dmb_vec_desc *vecs;       /* [nchunks]                                      */
  dmb_string_t *out;              /* chunk k at k*2048 entries                      */
  const uint32_t *dict_offsets;   /* device, [dict_size + 1]                        */
  const uint8_t *dict_data;       /* device                                         */
  uint64_t dict_host_base;        /* address the emitted pointers are relative to   */
  unsigned long long *bad_index;  /* device counter or NULL                         */
  uint32_t dict_size;
  int32_t phys;                   /* DMB_PHYS_U8 / U16 / U32                        */
} dmb_enum_job;

int32_t dmb_dev_enum_to_string_t(const dmb_enum_job *job, const uint32_t *counts, int64_t nchunks, void *stream);

/* K8 fused with K5 (Arrow modes): ENUM indices -> utf8 offsets + data in ONE launch, for dictionaries of up to
 * DMB_ENUM_FUSED_MAX_LABELS labels of <= 12 bytes each (every uint8 ENUM with short labels: flags, modes, codes).  The
 * labels become a string_t table in shared memory, so the string_t intermediate (16 B per row written and read back) of
 * the two-step form does not exist.  `ejob->out` and `sjob->in / vecs / in_validity / heap_*` are ignored: rows and validity come from
 * `ejob`, outputs from `sjob`.  A label longer than 12 bytes raises the heap-range flag (dmb_dev_string_error); a valid row whose
 * index is >= dict_size is counted in *bad_index and left empty.  `scratch` as for dmb_dev_string_batch.
 * Replaces, like the two-step form, libduckdb's duckdb_value_varchar on an ENUM cell at src/duckdb_native.c:224-238, :2478, :2715. */
#define DMB_ENUM_FUSED_MAX_LABELS 256
int32_t dmb_dev_enum_utf8(const dmb_enum_job *ejob, const dmb_string_job *sjob, const uint32_t *counts,
                          const int64_t *row_off, int64_t nchunks, int64_t nrows, void *scratch, void *stream);

/* K9: LIST vectors -> Arrow list<child> (fixed-width child; SURVEY.md 8f item 3).  The reference rejects
 * LIST on its chunk path (src/duckdb_native.c:271-303): the contract is the Arrow format.  Per chunk: a vector of
 * duckdb_list_entry {uint64 offset, uint64 length} (+ validity) indexing that chunk's child vector
 * (duckdb_list_vector_get_child / _get_size).  The child vectors of all chunks are staged back to back:
 * chunk k's elements start at element child_base[k], its validity mask (ceil(size/64) words) at word
 * child_val_off[k] of child_validity (-1: all valid).  Output: offsets[nrows+1] (running sum of the valid rows'
 * lengths), child values gathered in row order (payload under a NULL element zeroed), child bitmap. */
typedef struct dmb_list_job {
  const void *in_entries;           /* list_entry slab, chunk k at vecs[k].data_off             */
  const uint64_t *in_validity;      /* validity slab of the LIST column                         */
  const dmb_vec_desc *vecs;         /* [nchunks]                                                */
  const uint64_t *child_base;       /* [nchunks]                                                */
  const void *child_data;           /* staged child payload, child_width bytes per element      */
  const uint64_t *child_validity;   /* staged child masks or NULL                               */
  const int64_t *child_val_off;     /* [nchunks] or NULL                                        */
  void *out_offsets;                /* int32 (int64 when large) [nrows + 1]                     */
  void *out_child;                  /* child_width bytes per element, dense                     */
  uint64_t *out_child_validity;     /* LSB bitmap, ceil(capacity/64)+1 words, or NULL           */
  unsigned long long *total;        /* number of child elements written                         */
  unsigned long long *child_null_count;
  int32_t child_width;              /* 1 / 2 / 4 / 8 / 16                                       */
  int32_t large;                    /* bit 0: int64 offsets (large_list); bit 1 (DMB_LIST_DENSE_CHILD_BITS): child_validity
                                       is ONE bitmap over the whole staged child slab (bit i = element i; child_val_off is
                                       ignored) instead of one padded mask per chunk -- the form a second-level gather
                                       (nested lists: entries already rebased onto the slab) reads */
  const uint64_t *child_sizes;      /* [nchunks] elements in each chunk's child vector, or NULL: entries are only
                                       checked against 2^32 - 2 elements (the kernel keeps a row's offset and length
                                       as 32-bit values; a child vector larger than that raises flag 2).  A valid row
                                       whose offset + length reaches past its child vector raises flag 8 and
                                       contributes no elements (never read)                                     */
} dmb_list_job;

#define DMB_LIST_DENSE_CHILD_BITS 2
size_t dmb_dev_list_scratch_bytes(int64_t nchunks);
/* scratch[0] after the call: error flags (1: total exceeds int32 offsets, 2: a chunk with > 4 G child elements,
 * 4: a look-back gave up waiting, 8: a list entry outside its child vector) */
int32_t dmb_dev_list_batch(const dmb_list_job *job, const uint32_t *counts, const int64_t *row_off, int64_t nchunks,
                           int64_t nrows, int64_t child_capacity, void *scratch, void *stream);

/* K6 reverse (Arrow -> DataChunk vectors), the bulk door behind the appender
 * (reference row-at-a-time path: src/duckdb_native.c:1100-1235; chunk door :2029-2132). */
typedef struct dmb_rev_fixed_job {
  const void *in_values;        /* Arrow values buffer (already offset to the slice start) */
  const uint8_t *in_validity;   /* Arrow bitmap bytes or NULL                              */
  int64_t in_bit_offset;        /* Arrow array offset (bits into in_validity / bool values) */
  void *out_data;               /* vector slab: chunk k at k*2048*W bytes                  */
  uint64_t *out_validity;       /* validity slab: chunk k at k*32 words                    */
  unsigned long long *null_count;
  int32_t op;                   /* DMB_REV_* */
  int32_t reserved;
} dmb_rev_fixed_job;

enum dmb_rev_op {
  DMB_REV_COPY1 = 0, DMB_REV_COPY2 = 1, DMB_REV_COPY4 = 2, DMB_REV_COPY8 = 3, DMB_REV_COPY16 = 4,
  DMB_REV_BITS_TO_BOOL = 5,   /* Arrow bool bits -> DuckDB bool bytes                      */
  DMB_REV_I128_TO_I64 = 6,    /* decimal128 -> DECIMAL(<=18) int64                          */
  DMB_REV_I128_TO_I32 = 7,
  DMB_REV_I128_TO_I16 = 8,
  DMB_REV_COUNT = 9
};

/* jobs_dev: device array, jobs_host: its host mirror.  Device copies of Arrow bitmaps / data
 * buffers should carry >= 16 bytes of padding past their end. */
int32_t dmb_dev_rev_fixed_batch(const dmb_rev_fixed_job *jobs_dev, const dmb_rev_fixed_job *jobs_host,
                                int32_t njobs, int64_t nrows, void *stream);

typedef struct dmb_rev_string_job {
  const void *in_offsets;       /* int32 (or int64 when large) offsets, at the slice start */
  const uint8_t *in_data;       /* device copy of the Arrow data buffer                    */
  const uint8_t *in_validity;
  int64_t in_bit_offset;
  uint64_t data_host_base;      /* host address of the Arrow data buffer: pointer string_t
                                   reference it in place (SURVEY.md §8d)                   */
  dmb_string_t *out;            /* string_t slab: chunk k at k*2048 entries                */
  uint64_t *out_validity;
  unsigned long long *null_count;
  int32_t large_offsets;
  int32_t reserved;
} dmb_rev_string_job;

int32_t dmb_dev_rev_string_batch(const dmb_rev_string_job *job, int64_t nrows, void *stream);

/* Arrow list / large_list -> LIST vectors.  Row r of the slice gets duckdb_list_entry {off[r] - off[c0], off[r+1] - off[r]}
 * (c0: the first row of r's 2048-row chunk), so each chunk's entries index that chunk's own child vector; a NULL row gets
 * {off[r] - off[c0], 0}: DuckDB never sees a NULL row that owns elements.  The child values of the slice, Arrow elements
 * [off[0], off[nrows]), are converted as a dense column by dmb_dev_rev_fixed_batch / dmb_dev_rev_string_batch; this
 * kernel writes the entries, the list masks and each chunk's child mask, realigned to start at bit 0 of that chunk's
 * first element. */
typedef struct dmb_rev_list_job {
  const void *in_offsets;          /* int32 (or int64 when large) offsets at the slice start: nrows + 1 entries  */
  const uint8_t *in_validity;      /* list bitmap or NULL                                                       */
  int64_t in_bit_offset;
  const uint8_t *in_child_validity;  /* child bitmap or NULL                                                    */
  int64_t child_bit_offset;        /* bit of element off[0]: child array offset + off[0]                        */
  const int64_t *child_word;       /* [nchunks + 1]: chunk k's child mask starts at out_child_validity[child_word[k]] */
  void *out_entries;               /* duckdb_list_entry slab: chunk k at k*2048 entries                         */
  uint64_t *out_validity;          /* list mask slab: chunk k at k*32 words                                     */
  uint64_t *out_child_validity;    /* ceil(size_k / 64) words per chunk, bits past size_k are 0                 */
  unsigned long long *null_count;
  unsigned int *error;             /* |= 1: a row with off[r+1] < off[r]                                       */
  int32_t large_offsets;
  int32_t reserved;
} dmb_rev_list_job;

int32_t dmb_dev_rev_list_batch(const dmb_rev_list_job *job, int64_t nrows, void *stream);

/* STRUCT validity: out = in_a AND in_b over nrows rows (row r: bit a_bit_offset + r of in_a, bit b_bit_offset + r of in_b;
 * an absent bitmap is all valid), written from bit out_bit_offset (0..63) of `out` on as a dense bitmap of whole chunks:
 * ceil((out_bit_offset + nrows) / 2048) * 32 words, every bit outside [out_bit_offset, out_bit_offset + nrows) zero.
 * At bit offset 0 from a sub-batch's first row that is the DuckDB mask slab (chunk k at k*32 words): the appender writes a
 * STRUCT column's masks this way (its own bitmap AND its parent STRUCT's masks), and the combined bitmap that a field's
 * conversion reads as its validity (the parent's masks AND the field's own bitmap; for a BOOLEAN field at the bit phase
 * of its staged values).  jobs_dev: device array, jobs_host: its host mirror; grid.y = job. */
typedef struct dmb_rev_mask_job {
  const uint8_t *in_a;   /* bitmap bytes or NULL */
  int64_t a_bit_offset;
  const uint8_t *in_b;   /* bitmap bytes or NULL */
  int64_t b_bit_offset;
  uint64_t *out;
  int64_t out_bit_offset;
} dmb_rev_mask_job;

int32_t dmb_dev_rev_mask_batch(const dmb_rev_mask_job *jobs_dev, const dmb_rev_mask_job *jobs_host, int32_t njobs, int64_t nrows,
                               void *stream);
/* the appender's sub-batch cut (host only): the end chunk (exclusive) of the sub-batch that starts at chunk k0.  It takes
 * at most max_chunks chunks, and stops before the chunk that would give any of the nlists LIST columns more than
 * child_cap child elements; the first chunk is always taken, so one chunk's child range is never split.
 * bounds[l][k]: list l's Arrow offset at row 2048k (at the last row for k = nchunks). */
int64_t dmb_rev_list_cut(const int64_t *const *bounds, int32_t nlists, int64_t nchunks, int64_t k0, int64_t max_chunks,
                         int64_t child_cap);

/* Labels -> DuckDB ENUM positions.  Two conversions, one job:
 *   strings (index_width 0): utf8 / large_utf8 rows are looked up byte-exactly in an open-addressing table of the ENUM's
 *     labels (dmb_rev_enum_table); with out_width 0 ("remap" mode) the rows are an Arrow dictionary and each gets one
 *     uint32 code in `out` (a position, DMB_ENUM_CODE_NULL for a NULL entry, DMB_ENUM_CODE_MISSING for a label the ENUM
 *     lacks), no masks and no error;
 *   dictionary indices (index_width 1/2/4/8, signed or not): row r's position is remap[index] (remap: the codes of the
 *     Arrow dictionary, dict_len entries).
 * Otherwise the output is final vectors: positions of out_width (1/2/4) bytes, chunk k at k*2048*out_width bytes, masks
 * at k*32 words.  A NULL row, and a valid row whose dictionary entry is NULL, is NULL with payload 0.  A valid row whose
 * label is not in the ENUM, or whose index is outside [0, dict_len), is an error: *error takes the smallest such row
 * (atomicMin; the caller sets it to ~0 first) and the row is written as NULL. */
struct dmb_enum_dict;
#define DMB_ENUM_CODE_NULL 0xFFFFFFFEu
#define DMB_ENUM_CODE_MISSING 0xFFFFFFFFu
#define DMB_ENUM_SLOT_BYTES 32 /* one lookup-table slot: {position, length, hash, 0} {first 12 bytes, last 4 bytes} */
typedef struct dmb_rev_enum_job {
  const void *in_offsets;          /* strings: int32 (or int64 when large) offsets at the slice start: nrows + 1 entries */
  const uint8_t *in_data;          /* strings: device copy of the data buffer, indexed by the offsets                    */
  const void *in_indices;          /* indices: the first index of the slice                                              */
  const uint8_t *in_validity;      /* bitmap or NULL                                                                      */
  int64_t in_bit_offset;
  const uint32_t *remap;           /* indices: [dict_len] codes                                                           */
  int64_t dict_len;
  const void *table;               /* strings: table_size slots of DMB_ENUM_SLOT_BYTES                                    */
  const uint32_t *label_offsets;   /* strings: the ENUM's labels (dmb_enum_dict layout), read for labels > 16 bytes      */
  const uint8_t *label_data;
  void *out;
  uint64_t *out_validity;
  unsigned long long *null_count;
  unsigned long long *error;
  uint32_t table_size;             /* a power of two                                                                      */
  int32_t out_width;               /* 1 / 2 / 4; 0: remap mode (strings only)                                             */
  int32_t index_width;             /* 1 / 2 / 4 / 8; 0: strings                                                           */
  int32_t index_signed;
  int32_t large_offsets;
  int32_t reserved;
} dmb_rev_enum_job;

int32_t dmb_dev_rev_enum_batch(const dmb_rev_enum_job *job, int64_t nrows, void *stream);
/* host only: the lookup table of `dict` in table_size slots (a power of two above the label count), what
 * dmb_dev_rev_enum_batch probes.  Returns 0 with the last error set for a table that is too small or a duplicate label. */
int32_t dmb_rev_enum_table(const struct dmb_enum_dict *dict, uint32_t table_size, void *slots);
/* host only: the position of `bytes` in such a table, -1 when it is not a label (the device's probe, run on the host) */
int64_t dmb_rev_enum_lookup(const void *slots, uint32_t table_size, const struct dmb_enum_dict *dict, const uint8_t *bytes, uint32_t len);

/* Arrow string views (utf8_view / binary_view) -> string_t.  A view is 16 bytes, {int32 len, 12 inline bytes} when
 * len <= 12, else {int32 len, 4-byte prefix, int32 buffer index, int32 offset}; a string_t is the same 16 bytes inline and
 * {len, prefix, 8-byte pointer} otherwise.  So the kernel reads no string bytes: an inline view is copied with its bytes
 * past len zeroed, a pointer view takes its prefix from the view and points at buffers[index].host_base + offset, in
 * place in the caller's host buffer.  A NULL row is NULL with payload 0.  A valid row with a negative len, or a pointer view
 * whose index is >= nbuffers, whose offset is negative or whose offset + len passes that buffer's size is an error:
 * *error takes the smallest such row (atomicMin; the caller sets it to ~0 first).  out and out_validity are written for
 * whole 2048-row chunks (out_validity may be NULL, for a LIST child whose masks the list kernel writes). */
typedef struct dmb_view_buffer {
  uint64_t host_base;              /* host address of an Arrow data buffer */
  int64_t size;                    /* its size in bytes                    */
} dmb_view_buffer;

typedef struct dmb_rev_view_job {
  const void *in_views;            /* 16-byte views at the slice start, 16-byte aligned */
  const uint8_t *in_validity;      /* bitmap or NULL                                    */
  int64_t in_bit_offset;
  const dmb_view_buffer *buffers;  /* device table of the array's data buffers          */
  int64_t nbuffers;
  dmb_string_t *out;               /* string_t slab: chunk k at k*2048 entries          */
  uint64_t *out_validity;
  unsigned long long *null_count;
  unsigned long long *error;
} dmb_rev_view_job;

int32_t dmb_dev_rev_view_batch(const dmb_rev_view_job *job, int64_t nrows, void *stream);

/* Arrow dictionary indices (1/2/4/8 bytes, signed or not) -> string_t, gathered from `table`: the dictionary's dict_len
 * entries as string_t (converted once by dmb_dev_rev_string_batch or dmb_dev_rev_view_batch), a NULL entry marked by
 * len DMB_DICT_ENTRY_NULL (dmb_dev_rev_dict_mark).  A NULL row, and a valid row whose entry is NULL, is NULL with
 * payload 0.  A valid row whose index is outside [0, dict_len) is an error: *error takes the smallest such row
 * (atomicMin; the caller sets it to ~0 first).  out and out_validity are written for whole 2048-row chunks; out_validity
 * is required, and is a dense bitmap of the rows (bit r: row r). */
#define DMB_DICT_ENTRY_NULL 0xFFFFFFFFu
typedef struct dmb_rev_dict_job {
  const void *in_indices;          /* the first index of the slice */
  const uint8_t *in_validity;      /* bitmap or NULL               */
  int64_t in_bit_offset;
  const dmb_string_t *table;       /* [dict_len]                   */
  int64_t dict_len;
  dmb_string_t *out;
  uint64_t *out_validity;
  unsigned long long *null_count;
  unsigned long long *error;
  int32_t index_width;             /* 1 / 2 / 4 / 8                */
  int32_t index_signed;
} dmb_rev_dict_job;

int32_t dmb_dev_rev_dict_batch(const dmb_rev_dict_job *job, int64_t nrows, void *stream);
/* entry i of `table` whose bit i of `masks` (a dense bitmap) is 0 gets len DMB_DICT_ENTRY_NULL */
int32_t dmb_dev_rev_dict_mark(dmb_string_t *table, const uint64_t *masks, int64_t n, void *stream);

/* byte-per-row validity (MoonBit Array[Bool], src/duckdb_arrow_native.mbt:646-650) -> per-chunk
 * uint64 masks via warp ballots */
int32_t dmb_dev_valid_bytes_to_masks(const uint8_t *valid_bytes, uint64_t *out_validity,
                                     unsigned long long *null_count, int64_t nrows, void *stream);

/* bench/test helper: assemble DuckDB-shaped string_t on the device from lengths and heap
 * offsets (not part of the product path) */
int32_t dmb_dev_make_string_t(const uint32_t *lengths, const uint64_t *heap_off,
                              const uint8_t *heap_dev, uint64_t heap_host_base, dmb_string_t *out,
                              int64_t n, void *stream);

/* =====================================================================================
 * L1 — host API.
 * ===================================================================================== */

typedef struct duckdb_mb_gpu_ctx duckdb_mb_gpu_ctx;       /* one per GPU: streams, pinned ring   */
typedef struct duckdb_mb_arrow_result duckdb_mb_arrow_result; /* same handle name as the reference
                                                              (src/duckdb_native.c:2211-2217)    */

/* thread-local last error (the reference keeps one process-global string,
 * src/duckdb_native.c:22-40,240-246; SURVEY.md §5 asks for thread safety) */
const char *duckdb_mb_gpu_last_error(void);

int32_t duckdb_mb_gpu_device_count(void);
duckdb_mb_gpu_ctx *duckdb_mb_gpu_ctx_create(int32_t device);
void duckdb_mb_gpu_ctx_destroy(duckdb_mb_gpu_ctx *ctx);
int32_t duckdb_mb_gpu_ctx_sync(duckdb_mb_gpu_ctx *ctx);

/* Bind the calling thread (and the threads / page-locked allocations it makes afterwards) to the CPUs of the GPU's NUMA
 * node: call once per process before creating the context and allocating host buffers when one process drives one GPU
 * (SURVEY.md 8e).  Returns the node, or -1 when there is nothing to bind to; never fails. */
int32_t duckdb_mb_gpu_bind_numa(int32_t device);

/* pinned host memory for callers that can place chunk vectors / Arrow buffers in it
 * (staging then needs no bounce copy) */
void *duckdb_mb_gpu_host_alloc(size_t bytes);
void duckdb_mb_gpu_host_free(void *p);

/* ENUM: the type's dictionary, what duckdb_enum_dictionary_size / duckdb_enum_dictionary_value return,
 * packed: label i = data[offsets[i] .. offsets[i+1]).  The column's vectors hold the indices in the
 * width duckdb_enum_internal_type names (phys DMB_PHYS_U8 / U16 / U32).  The reference keeps an ENUM
 * cell as Value::String of its label (src/duckdb_parsing.mbt:119-122) and maps the column to "string"
 * in the Arrow schema (src/duckdb_native.c:2314-2339); the Arrow C Data export is dictionary-encoded. */
typedef struct dmb_enum_dict {
  uint32_t size;
  uint32_t reserved;
  const uint32_t *offsets; /* [size + 1], offsets[0] == 0 */
  const char *data;
} dmb_enum_dict;

/* LIST of a fixed-width child: the column's vectors hold duckdb_list_entry {uint64 offset, uint64 length} (phys
 * DMB_PHYS_U128: 16 bytes per row); per chunk, the child vector the entries index: duckdb_list_vector_get_child(v)
 * -> duckdb_vector_get_data / _get_validity, and duckdb_list_vector_get_size(v) elements of it.  Arrow export only
 * (list<child>; the child in the Arrow form of its type, as for a top-level column: BOOLEAN bit-packed, DECIMAL as
 * decimal128, INTERVAL as month_day_nano, the other fixed-width types as stored); the
 * reference rejects LIST on its chunk path (src/duckdb_native.c:271-303) and has no Arrow mapping for it. */
struct dmb_host_column;
typedef struct dmb_host_list {
  int32_t child_type_id;                  /* enum dmb_type */
  int32_t child_phys;                     /* enum dmb_phys */
  int32_t child_dec_width, child_dec_scale;
  const void *const *child_data;          /* [nchunks] */
  const uint64_t *const *child_validity;  /* [nchunks], entries may be NULL; the array may be NULL */
  const uint64_t *child_sizes;            /* [nchunks] elements in each chunk's child vector */
  /* Children that are not one fixed-width vector -- VARCHAR / BLOB (the child vectors' string heaps are gathered by the
   * stager), STRUCT (MAP = LIST<STRUCT<key, value>>), LIST (nested lists) -- are described as a full column: data[k] /
   * validity[k] / struct_ / list of child_col are those of chunk k's CHILD vector (child_sizes[k] elements of it:
   * duckdb_list_vector_get_child / _get_size).  When child_col is set it wins over the four child_* type fields and the two
   * pointer tables above.  NULL: the flat fixed-width form. */
  const struct dmb_host_column *child_col;
} dmb_host_list;

/* STRUCT: what duckdb_struct_vector_get_child(v, i) returns for every field, chunk by chunk; the struct's own validity
 * is the column's `validity` (its `data` is unused and may be NULL).  Arrow export only (struct<...>, fields exported like
 * top-level columns); the reference rejects STRUCT on its chunk path (src/duckdb_native.c:271-303). */
typedef struct dmb_host_struct {
  int32_t nfields;
  int32_t reserved;
  const struct dmb_host_column *fields;   /* [nfields]; name = the field's name */
} dmb_host_struct;

/* One column of a host chunk batch: the pointers duckdb_vector_get_data /
 * duckdb_vector_get_validity return for each chunk (src/duckdb_native.c:529-530,547). */
typedef struct dmb_host_column {
  const char *name;
  int32_t type_id;       /* enum dmb_type */
  int32_t phys;          /* enum dmb_phys (DECIMAL: by width) */
  int32_t dec_width;
  int32_t dec_scale;
  const void *const *data;          /* [nchunks] */
  const uint64_t *const *validity;  /* [nchunks], entries may be NULL; the array may be NULL */
  /* VARCHAR/BLOB: a contiguous host region containing every non-inlined string of the column
   * (copied wholesale, pointers rebased on the device), or heap_len == 0: the stager compacts
   * the pointed-to bytes into pinned memory itself. */
  const void *heap_base;
  uint64_t heap_len;
  const dmb_enum_dict *dict;        /* ENUM columns: the dictionary (copied by result_from_chunks); else NULL */
  const dmb_host_list *list;        /* LIST / MAP columns: the per-chunk child vectors (pointer tables copied); else NULL */
  const dmb_host_struct *struct_;   /* STRUCT columns: the per-field vectors; else NULL */
} dmb_host_column;

/* heap_base == DMB_HEAP_INLINE_ONLY (heap_len 0): the caller guarantees that every string of the
 * column is inlined in its string_t (<= 12 bytes: flags, codes, CHAR(n <= 12)), so there is no heap
 * to stage or compact and the heap-less kernel runs.  A pointer entry is then an error
 * ("string_t pointer outside the registered heap"), never a wild read. */
#define DMB_HEAP_INLINE_ONLY ((const void *)(uintptr_t)1)

typedef struct dmb_host_batch {
  int32_t ncols;
  int32_t flags;           /* DMB_BATCH_* */
  int64_t nchunks;
  const uint32_t *counts;  /* [nchunks] */
  const dmb_host_column *cols;
} dmb_host_batch;

#define DMB_BATCH_PINNED 1 /* all data/validity/heap pointers are in page-locked memory */

/* Build a result from host chunks: stages them to the device (async, on the ctx streams).
 * Conversion happens lazily per export call or eagerly with duckdb_mb_gpu_result_materialise.
 * Stands where the reference keeps the duckdb_result (src/duckdb_native.c:2219-2268). */
duckdb_mb_arrow_result *duckdb_mb_gpu_result_from_chunks(duckdb_mb_gpu_ctx *ctx,
                                                         const dmb_host_batch *batch);

/* Arrow C Data Interface structs (Arrow spec; 80 / 72 bytes) */
#ifndef ARROW_C_DATA_INTERFACE
#define ARROW_C_DATA_INTERFACE
struct ArrowSchema {
  const char *format;
  const char *name;
  const char *metadata;
  int64_t flags;
  int64_t n_children;
  struct ArrowSchema **children;
  struct ArrowSchema *dictionary;
  void (*release)(struct ArrowSchema *);
  void *private_data;
};
struct ArrowArray {
  int64_t length;
  int64_t null_count;
  int64_t offset;
  int64_t n_buffers;
  int64_t n_children;
  const void **buffers;
  struct ArrowArray **children;
  struct ArrowArray *dictionary;
  void (*release)(struct ArrowArray *);
  void *private_data;
};
#endif

#ifndef ARROW_C_STREAM_INTERFACE
#define ARROW_C_STREAM_INTERFACE
struct ArrowArrayStream { /* Arrow C stream interface */
  int (*get_schema)(struct ArrowArrayStream *, struct ArrowSchema *out);
  int (*get_next)(struct ArrowArrayStream *, struct ArrowArray *out); /* released array (release == NULL) = end of stream */
  const char *(*get_last_error)(struct ArrowArrayStream *);
  void (*release)(struct ArrowArrayStream *);
  void *private_data;
};
#endif

/* DataChunk -> Arrow for every column: H2D (if not yet staged), kernels, D2H into pinned
 * buffers owned by the result.  Blocking.  Returns 1/0 (reference mutator convention). */
int32_t duckdb_mb_gpu_result_materialise_arrow(duckdb_mb_arrow_result *r);
/* Export column `col` (or the whole batch as a struct array with col = -1). */
int32_t duckdb_mb_gpu_result_export_arrow(duckdb_mb_arrow_result *r, int32_t col,
                                          struct ArrowArray *out_array,
                                          struct ArrowSchema *out_schema);

/* typed columns (columnar to_typed; replaces the string round trip
 * src/duckdb_native.mbt:477-497 -> src/duckdb_typed_result.mbt:8-43) */
enum dmb_value_tag { /* order of `Value` in src/duckdb.mbt:183-193 */
  DMB_VALUE_INT = 0, DMB_VALUE_DOUBLE = 1, DMB_VALUE_BOOL = 2, DMB_VALUE_STRING = 3,
  DMB_VALUE_DATE = 4, DMB_VALUE_TIMESTAMP = 5, DMB_VALUE_DECIMAL = 6, DMB_VALUE_BLOB = 7,
  DMB_VALUE_NULL = 8
};
typedef struct dmb_typed_column {
  int32_t tag;            /* enum dmb_value_tag of the non-null cells                      */
  int32_t width;          /* bytes per value: Int 4, Double 8, Bool 1, Date 4, Timestamp 8 */
  int64_t length;
  int64_t null_count;
  const void *values;     /* host, pinned, owned by the result                            */
  const uint8_t *valid;   /* byte per row, 1 = non-null                                   */
  const int32_t *offsets; /* String: utf8 offsets[n+1]                                    */
  const uint8_t *data;    /* String: utf8 bytes                                           */
} dmb_typed_column;
int32_t duckdb_mb_gpu_result_typed_column(duckdb_mb_arrow_result *r, int32_t col,
                                          dmb_typed_column *out);
/* the string form of a column (tag = DMB_VALUE_STRING: utf8 offsets + data + byte validity): the
 * VARCHAR rendering of every cell, which the reference's Connection::query collects with two FFI
 * calls per cell, duckdb_mb_result_is_null + duckdb_mb_result_value -> duckdb_value_varchar
 * (src/duckdb_native.c:215-238, loop src/duckdb_native.mbt:477-497).  0 + last error for types
 * whose libduckdb rendering is not reproduced on the device (dmb_render_supported). */
int32_t duckdb_mb_gpu_result_text_column(duckdb_mb_arrow_result *r, int32_t col,
                                         dmb_typed_column *out);

/* ---- L2 drop-in, per-cell accessors of the materialised result (src/duckdb_native.c:174-254;
 * MoonBit externs src/duckdb_native.mbt:296-340).  The handle is the same result object: the
 * glue's duckdb_mb_query returns what duckdb_mb_gpu_result_from_chunks built.  `value` is the
 * cell's duckdb_value_varchar rendering (strlen-truncated, empty Bytes for NULL), produced for the
 * whole column by one GPU pass on the first call and sliced afterwards. */
void duckdb_mb_result_destroy(duckdb_mb_arrow_result *r);
int32_t duckdb_mb_is_null_result(duckdb_mb_arrow_result *r);
int32_t duckdb_mb_result_column_count(duckdb_mb_arrow_result *r);
int32_t duckdb_mb_result_row_count(duckdb_mb_arrow_result *r);
moonbit_bytes_t duckdb_mb_result_column_name(duckdb_mb_arrow_result *r, int32_t col);
int32_t duckdb_mb_result_column_type(duckdb_mb_arrow_result *r, int32_t col);
int32_t duckdb_mb_result_is_null(duckdb_mb_arrow_result *r, int32_t col, int32_t row);
moonbit_bytes_t duckdb_mb_result_value(duckdb_mb_arrow_result *r, int32_t col, int32_t row);

/* ---- L2 drop-in, streaming chunks (src/duckdb_native.c:260-667; externs src/duckdb_native.mbt:342-392).
 * duckdb_mb_gpu_stream_from_result is what the glue's duckdb_mb_query_stream calls after running
 * the SQL (reference: duckdb_mb_stream_from_result, :319-353, same type whitelist and error).
 * chunk_is_null is the validity-bit test of :520-535; chunk_value returns the VARCHAR cast of the
 * cell (the reference's duckdb_value_to_string format is pinned by no reference test: UNPINNED). */
typedef struct duckdb_mb_stream duckdb_mb_stream;
typedef struct duckdb_mb_chunk duckdb_mb_chunk;
duckdb_mb_stream *duckdb_mb_gpu_stream_from_result(duckdb_mb_arrow_result *r);
void duckdb_mb_stream_destroy(duckdb_mb_stream *s);
int32_t duckdb_mb_is_null_stream(duckdb_mb_stream *s);
int32_t duckdb_mb_stream_column_count(duckdb_mb_stream *s);
moonbit_bytes_t duckdb_mb_stream_column_name(duckdb_mb_stream *s, int32_t col);
duckdb_mb_chunk *duckdb_mb_stream_fetch_chunk(duckdb_mb_stream *s);
void duckdb_mb_chunk_destroy(duckdb_mb_chunk *c);
int32_t duckdb_mb_is_null_chunk(duckdb_mb_chunk *c);
int32_t duckdb_mb_chunk_row_count(duckdb_mb_chunk *c);
int32_t duckdb_mb_chunk_column_count(duckdb_mb_chunk *c);
int32_t duckdb_mb_chunk_is_null(duckdb_mb_chunk *c, int32_t col, int32_t row);
moonbit_bytes_t duckdb_mb_chunk_value(duckdb_mb_chunk *c, int32_t col, int32_t row);

/* What the glue hangs on a result: the duckdb_result and the data chunks the batch's pointers refer to.  `destroy(owner)`
 * runs when the result is destroyed (duckdb_mb_arrow_destroy / duckdb_mb_result_destroy, or the owning stream's destroy),
 * after the last use of the host pointers. */
void duckdb_mb_gpu_result_set_owner(duckdb_mb_arrow_result *r, void *owner, void (*destroy)(void *owner));
/* like duckdb_mb_gpu_stream_from_result, but duckdb_mb_stream_destroy also destroys the result (the reference's stream
 * owns its duckdb_result, src/duckdb_native.c:426-438); on failure the result is destroyed and NULL returned */
duckdb_mb_stream *duckdb_mb_gpu_stream_from_result_owned(duckdb_mb_arrow_result *r);

/* ---- one table over N GPUs, and record-batch streams (SURVEY.md §8e, §8f item 2).
 * The chunk list is cut into contiguous ranges of whole chunks ("parts"): GPU g gets chunks [g * ceil(C / G), ...), and
 * with max_rows_per_part > 0 a GPU's range is cut further into parts of at most that many rows.  Every part is a result
 * of its own on its context (duckdb_mb_gpu_sharded_part: borrowed, usable with every duckdb_mb_gpu_result_* /
 * duckdb_mb_arrow_* call); materialise runs one host thread per part.  The only cross-GPU datum is one byte total per
 * string column per part: duckdb_mb_gpu_sharded_string_bases is their host exclusive scan (the base each part's utf8
 * offsets are shifted by when one logical column is stitched; out has part_count + 1 entries).  No collective.
 * The reference has no counterpart (one duckdb_result, one thread, src/duckdb_native.c:2219-2268). */
typedef struct duckdb_mb_gpu_sharded duckdb_mb_gpu_sharded;
duckdb_mb_gpu_sharded *duckdb_mb_gpu_result_from_chunks_sharded(duckdb_mb_gpu_ctx *const *ctxs, int32_t nctx, const dmb_host_batch *batch);
duckdb_mb_gpu_sharded *duckdb_mb_gpu_result_shard(duckdb_mb_arrow_result *r, duckdb_mb_gpu_ctx *const *ctxs, int32_t nctx,
                                                 int64_t max_rows_per_part); /* ctxs NULL: the result's own context */
int32_t duckdb_mb_gpu_sharded_part_count(duckdb_mb_gpu_sharded *s);
duckdb_mb_arrow_result *duckdb_mb_gpu_sharded_part(duckdb_mb_gpu_sharded *s, int32_t i);
int64_t duckdb_mb_gpu_sharded_first_row(duckdb_mb_gpu_sharded *s, int32_t i); /* i = part_count: total rows */
int32_t duckdb_mb_gpu_sharded_materialise_arrow(duckdb_mb_gpu_sharded *s);
int32_t duckdb_mb_gpu_sharded_string_bases(duckdb_mb_gpu_sharded *s, int32_t col, uint64_t *out);
void duckdb_mb_gpu_sharded_destroy(duckdb_mb_gpu_sharded *s);
/* ArrowArrayStream (Arrow C stream interface): one record batch per part, in row order, converted one batch ahead of the
 * consumer.  _sharded_export_stream hands the handle over to the stream (do not destroy it afterwards);
 * _result_export_stream cuts a result into batches of at most max_batch_rows rows (<= 0: 16 M) on its own context, so a
 * column with more than 2^31 string bytes (BASELINE config C3) leaves as several utf8 batches instead of one large_utf8
 * array.  The host chunk vectors must stay alive until the stream is released (a glue owner is shared automatically). */
int32_t duckdb_mb_gpu_sharded_export_stream(duckdb_mb_gpu_sharded *s, struct ArrowArrayStream *out);
int32_t duckdb_mb_gpu_result_export_stream(duckdb_mb_arrow_result *r, int64_t max_batch_rows, struct ArrowArrayStream *out);

/* timings of the last materialise call, milliseconds: [0]=h2d [1]=kernels [2]=d2h [3]=total */
int32_t duckdb_mb_gpu_result_timings(duckdb_mb_arrow_result *r, double *out4);
/* bytes moved over the host link by the last materialise call: [0]=h2d [1]=d2h */
int32_t duckdb_mb_gpu_result_link_bytes(duckdb_mb_arrow_result *r, uint64_t *out2);

/* =====================================================================================
 * L2 — the reference's own symbols (src/duckdb_arrow_native.mbt:9-104), byte-compatible
 * results (src/duckdb_native.c:2357-2797), served by the GPU path.
 * duckdb_mb_query_arrow itself needs libduckdb to run SQL; INTEGRATION.md shows the glue that
 * turns its duckdb_result into a dmb_host_batch.
 * ===================================================================================== */
int32_t duckdb_mb_arrow_column_count(duckdb_mb_arrow_result *r); /* :2270-2275 */
int32_t duckdb_mb_arrow_row_count(duckdb_mb_arrow_result *r);    /* :2277-2282 */
moonbit_bytes_t duckdb_mb_arrow_schema(duckdb_mb_arrow_result *r); /* :2285-2355 */
moonbit_bytes_t duckdb_mb_arrow_get_column_int32(duckdb_mb_arrow_result *r, int32_t col);  /* :2359 */
moonbit_bytes_t duckdb_mb_arrow_get_column_int64(duckdb_mb_arrow_result *r, int32_t col);  /* :2392 */
moonbit_bytes_t duckdb_mb_arrow_get_column_double(duckdb_mb_arrow_result *r, int32_t col); /* :2424 */
moonbit_bytes_t duckdb_mb_arrow_get_column_string(duckdb_mb_arrow_result *r, int32_t col); /* :2456 */
moonbit_bytes_t duckdb_mb_arrow_get_column_bool(duckdb_mb_arrow_result *r, int32_t col);   /* :2516 */
moonbit_bytes_t duckdb_mb_arrow_get_column_int32_nullable(duckdb_mb_arrow_result *r, int32_t col);  /* :2572 */
moonbit_bytes_t duckdb_mb_arrow_get_column_int64_nullable(duckdb_mb_arrow_result *r, int32_t col);  /* :2611 */
moonbit_bytes_t duckdb_mb_arrow_get_column_double_nullable(duckdb_mb_arrow_result *r, int32_t col); /* :2649 */
moonbit_bytes_t duckdb_mb_arrow_get_column_string_nullable(duckdb_mb_arrow_result *r, int32_t col); /* :2687 */
moonbit_bytes_t duckdb_mb_arrow_get_column_bool_nullable(duckdb_mb_arrow_result *r, int32_t col);   /* :2761 */
void duckdb_mb_arrow_destroy(duckdb_mb_arrow_result *r);              /* :2548-2554 */
int32_t duckdb_mb_is_null_arrow_result(duckdb_mb_arrow_result *r);    /* :2556-2558 */
double duckdb_mb_bytes_to_double(const char *bytes, int32_t offset);  /* :2561-2565 */

/* =====================================================================================
 * Reverse path: Arrow record batch -> DataChunk vectors for duckdb_append_data_chunk, gated by
 * the appender protocol of src/duckdb_appender_state_machine.mbt:54-239.
 * ===================================================================================== */
typedef struct duckdb_mb_gpu_appender duckdb_mb_gpu_appender;

/* sink called once per finished 2048-row chunk: `vec_data[c]` / `vec_validity[c]` are host
 * pointers laid out exactly as duckdb_vector_get_data / _get_validity expect, so the glue
 * memcpy's (or, with pinned vectors, hands) them to duckdb_append_data_chunk
 * (src/duckdb_native.c:2109-2132).  Return 0 to abort. */
typedef int32_t (*dmb_chunk_sink)(void *user, int32_t ncols, uint32_t count,
                                  const void *const *vec_data,
                                  const uint64_t *const *vec_validity);

duckdb_mb_gpu_appender *duckdb_mb_gpu_appender_create(duckdb_mb_gpu_ctx *ctx, int32_t ncols,
                                                      const int32_t *type_ids,
                                                      dmb_chunk_sink sink, void *user);
void duckdb_mb_gpu_appender_destroy(duckdb_mb_gpu_appender *a);
moonbit_bytes_t duckdb_mb_gpu_appender_error(duckdb_mb_gpu_appender *a); /* cf. :1093-1098 */
/* state: 0 NotCreated 1 Ready 2 RowInProgress 3 Flushed 4 Closed 5 Error
 * (AppenderState, src/duckdb_appender_state_machine.mbt:7-14) */
int32_t duckdb_mb_gpu_appender_state(duckdb_mb_gpu_appender *a);
int64_t duckdb_mb_gpu_appender_row_count(duckdb_mb_gpu_appender *a);
/* bulk append of one Arrow record batch (struct array, one child per column); legal in
 * Ready / Flushed, like BeginRow; returns 1/0 with the per-handle error string set.
 * VARCHAR / BLOB columns (and fields and LIST children of that type) take utf8 / large_utf8 (binary / large_binary), string
 * views (vu / vz; the sizes buffer of the C data interface is required) and dictionary arrays of those (indices c C s S i I
 * l L); the table holds what the same array cast to utf8 / binary gives.  A malformed view or an out-of-range index on a
 * valid row fails the append before its sub-batch reaches the sink (a LIST child's element: one its own bitmap marks
 * valid, also under a NULL list row).  A dictionary of views is converted whole: a malformed view in it fails the append
 * whether or not a row refers to it. */
int32_t duckdb_mb_gpu_append_arrow_batch(duckdb_mb_gpu_appender *a, const struct ArrowArray *batch,
                                         const struct ArrowSchema *schema);
int32_t duckdb_mb_gpu_appender_flush(duckdb_mb_gpu_appender *a); /* cf. duckdb_mb_flush :1237 */
int32_t duckdb_mb_gpu_appender_close(duckdb_mb_gpu_appender *a);
int64_t duckdb_mb_gpu_appender_flushed_row_count(duckdb_mb_gpu_appender *a);
/* timings of the last conversion, ms: [0]=h2d [1]=kernels [2]=d2h [3]=total; link bytes [0]=h2d [1]=d2h */
int32_t duckdb_mb_gpu_appender_timings(duckdb_mb_gpu_appender *a, double *out4);
int32_t duckdb_mb_gpu_appender_link_bytes(duckdb_mb_gpu_appender *a, uint64_t *out2);

/* The reference's row-at-a-time protocol (duckdb_mb_begin_row / append_* / end_row,
 * src/duckdb_native.c:1100-1235, MoonBit wrappers src/duckdb_native.mbt:974-1058) on the same
 * handle: cells are buffered column-wise on the host and converted by the same kernels on
 * flush / close / every 2^20 rows.  Same 1/0 + per-handle error convention; an over- or
 * under-filled row, or a call outside a row, moves the handle to the Error state
 * (src/duckdb_appender_state_machine.mbt:96-177,228-238). */
int32_t duckdb_mb_gpu_begin_row(duckdb_mb_gpu_appender *a);                                   /* :1100 */
int32_t duckdb_mb_gpu_append_int(duckdb_mb_gpu_appender *a, int32_t v);                       /* :1116 */
int32_t duckdb_mb_gpu_append_bigint(duckdb_mb_gpu_appender *a, int64_t v);                    /* :1132 */
int32_t duckdb_mb_gpu_append_double(duckdb_mb_gpu_appender *a, double v);                     /* :1148 */
int32_t duckdb_mb_gpu_append_varchar(duckdb_mb_gpu_appender *a, const uint8_t *bytes, int32_t len); /* :1164 */
int32_t duckdb_mb_gpu_append_bool(duckdb_mb_gpu_appender *a, int32_t v);                      /* :1189 */
int32_t duckdb_mb_gpu_append_null(duckdb_mb_gpu_appender *a);                                 /* :1205 */
int32_t duckdb_mb_gpu_append_date(duckdb_mb_gpu_appender *a, int32_t days);   /* exact days, not the
                                      approximate string path of :1313-1331 (SURVEY.md B.10) */
int32_t duckdb_mb_gpu_append_timestamp(duckdb_mb_gpu_appender *a, int64_t micros);            /* :1350 */
int32_t duckdb_mb_gpu_append_blob(duckdb_mb_gpu_appender *a, const uint8_t *bytes, int32_t len);    /* :1397 */
/* DECIMAL from hugeint parts (:1447-1481).  The column's DECIMAL(width, scale) comes from
 * duckdb_mb_gpu_appender_set_decimal (what duckdb_appender_column_type reports) or, failing that, from the
 * first value; values of another scale are cast like DuckDB's decimal -> decimal cast, out-of-range is an error.
 * Arrow batches are narrowed to the declared width too: a decimal128 column must have the declared scale and a
 * precision <= the width (decimal32/64/256 and anything else are refused); an undeclared column takes both from its
 * first Arrow batch. */
int32_t duckdb_mb_gpu_appender_set_decimal(duckdb_mb_gpu_appender *a, int32_t col, int32_t width, int32_t scale);
int32_t duckdb_mb_gpu_append_decimal(duckdb_mb_gpu_appender *a, int32_t width, int32_t scale, int64_t lower, int64_t upper);
/* LIST columns take Arrow list / large_list arrays through duckdb_mb_gpu_append_arrow_batch.  The table's child type
 * (duckdb_list_type_child_type of duckdb_appender_column_type) is declared first: the Arrow child format alone does not
 * say it (`tsu:` is TIMESTAMP or TIMESTAMP_TZ, `L` UBIGINT or TIME_TZ).  Children: the types the reverse path converts
 * (not INTERVAL or ENUM), VARCHAR and BLOB; LIST, STRUCT and MAP children are refused.  The row protocol refuses a
 * table with a LIST column. */
int32_t duckdb_mb_gpu_appender_set_list(duckdb_mb_gpu_appender *a, int32_t col, int32_t child_type_id, int32_t child_dec_width,
                                        int32_t child_dec_scale);
/* Only inside a dmb_chunk_sink call, for the chunk being handed over: LIST column `col`'s child vector.  vec_data[col] /
 * vec_validity[col] of that call are the duckdb_list_entry vector and the list mask; the entries index this child.
 * `*data`: `*size` values in DuckDB vector layout (string_t for VARCHAR / BLOB, pointers into the Arrow data buffer),
 * `*validity`: ceil(size / 64) mask words.  Host memory of the appender, valid until the sink call returns. */
int32_t duckdb_mb_gpu_appender_list_child(duckdb_mb_gpu_appender *a, int32_t col, const void **data, const uint64_t **validity,
                                          uint64_t *size);
/* ENUM columns: the type's labels (duckdb_enum_dictionary_value, copied) and its internal type (duckdb_enum_internal_type:
 * UTINYINT / USMALLINT / UINTEGER), which is the width of the vector.  Refused: a column that is not ENUM, another
 * internal type, more labels than it can index, a duplicate label, malformed offsets, a second, different declaration.
 * A declared column then takes dictionary-encoded Arrow arrays (indices c C s S i I l L, dictionary u / U) and plain u / U
 * arrays, and append_varchar / append_null cells of the row protocol; each label is matched byte-exactly.  A valid row
 * whose label is not in the ENUM, or whose dictionary index is out of range, fails the append before its sub-batch reaches
 * the sink; a row whose dictionary entry is NULL is NULL. */
int32_t duckdb_mb_gpu_appender_set_enum(duckdb_mb_gpu_appender *a, int32_t col, int32_t internal_type_id, const dmb_enum_dict *dict);
/* STRUCT columns take Arrow struct arrays ('+s') through duckdb_mb_gpu_append_arrow_batch.  The table's field types
 * (duckdb_struct_type_child_type of duckdb_appender_column_type) are declared first.  The fields become "field columns",
 * numbered *first_field .. *first_field + nfields - 1: numbering starts at the table's column count and follows declaration
 * order across all STRUCT columns.  set_decimal, set_enum and set_struct take a field column as they take a table column,
 * which declares DECIMAL and ENUM fields and nested STRUCTs.  Fields: the types the reverse path converts at top level,
 * DECIMAL, VARCHAR, BLOB, ENUM and STRUCT.  Refused by name: a column that is not STRUCT, zero fields, LIST and MAP
 * fields, any other field type, and a second declaration that differs from the first.
 * Arrow fields match by position (names are not compared).  A NULL struct row makes every field NULL at that row,
 * recursively, with payload 0, as DuckDB stores it; a label missing from an ENUM field is an error only under a valid
 * struct row.  In the sink call, vec_data[col] of a STRUCT column is NULL and vec_validity[col] is the struct's mask (its
 * own NULLs AND those of its ancestors).  The row protocol refuses a table with a STRUCT column. */
int32_t duckdb_mb_gpu_appender_set_struct(duckdb_mb_gpu_appender *a, int32_t col, int32_t nfields, const int32_t *field_type_ids,
                                          int32_t *first_field);
/* Only inside a dmb_chunk_sink call, for the chunk being handed over: field `field` of STRUCT column `col` (a table column
 * or a field column).  `*data`: the chunk's count values in DuckDB vector layout (string_t for VARCHAR / BLOB, pointers
 * into the Arrow data buffer), NULL for a STRUCT field; `*validity`: 32 mask words with the ancestors' NULLs folded in.
 * Host memory of the appender, valid until the sink call returns. */
int32_t duckdb_mb_gpu_appender_struct_field(duckdb_mb_gpu_appender *a, int32_t col, int32_t field, const void **data,
                                            const uint64_t **validity);
int32_t duckdb_mb_gpu_append_interval(duckdb_mb_gpu_appender *a, int32_t months, int32_t days, int64_t micros); /* :1511 */
/* LIST / STRUCT / MAP cells: the reference serialises them as text -- `["a", "b"]` (:1735-1790), `{"k": "v", ...}`
 * (:1792-1858 struct, :1860-1926 map), items copied without escaping -- and appends the text as one VARCHAR cell
 * through duckdb_append_varchar, so the text ends at the first NUL byte.  values[i] / lens[i] stand for the
 * reference's Array[Bytes] (moonbit_bytes_t* + Moonbit_array_length). */
int32_t duckdb_mb_gpu_append_list_varchar(duckdb_mb_gpu_appender *a, const uint8_t *const *values, const int32_t *lens, int32_t count);
int32_t duckdb_mb_gpu_append_struct_varchar(duckdb_mb_gpu_appender *a, const uint8_t *const *names, const int32_t *name_lens,
                                            const uint8_t *const *values, const int32_t *value_lens, int32_t count);
int32_t duckdb_mb_gpu_append_map_varchar_varchar(duckdb_mb_gpu_appender *a, const uint8_t *const *keys, const int32_t *key_lens,
                                                 const uint8_t *const *values, const int32_t *value_lens, int32_t count);
int32_t duckdb_mb_gpu_end_row(duckdb_mb_gpu_appender *a);                                     /* :1221 */

/* hooks for a sink that owns a libduckdb appender (glue/duckdb_gpu_glue.c): on_flush runs after a flush has handed
 * every buffered chunk to the sink (-> duckdb_appender_flush; return 0 on failure), on_destroy when the handle dies
 * (-> duckdb_appender_destroy, free of `user`) */
typedef int32_t (*dmb_appender_flush_hook)(void *user);
typedef void (*dmb_appender_destroy_hook)(void *user);
void duckdb_mb_gpu_appender_set_hooks(duckdb_mb_gpu_appender *a, dmb_appender_flush_hook on_flush, dmb_appender_destroy_hook on_destroy);

/* ---- L2 drop-in, the appender set: the reference's own symbols and signatures (src/duckdb_native.c:1083-1251,
 * 1313-1533, 1735-1926; externs src/duckdb_native.mbt:44-110,134-144,165-217,266-288).  `duckdb_mb_appender` is this
 * library's handle; Bytes are moonbit_bytes_t (length from the object header), Array[Bytes] is moonbit_bytes_t*;
 * every parameter is #borrow.  Same 1/0 + duckdb_mb_appender_error convention, with the protocol of
 * src/duckdb_appender_state_machine.mbt enforced.  duckdb_mb_appender_create(conn, schema, table) needs libduckdb
 * (duckdb_appender_create, column types): glue/duckdb_gpu_glue.c. */
typedef struct duckdb_mb_gpu_appender duckdb_mb_appender;
void duckdb_mb_appender_destroy(duckdb_mb_appender *a);                                       /* :1083 */
moonbit_bytes_t duckdb_mb_appender_error(duckdb_mb_appender *a);                              /* :1093 */
int32_t duckdb_mb_is_null_appender(duckdb_mb_appender *a);                                    /* :1253 */
int32_t duckdb_mb_begin_row(duckdb_mb_appender *a);                                           /* :1100 */
int32_t duckdb_mb_append_int(duckdb_mb_appender *a, int32_t value);                           /* :1116 */
int32_t duckdb_mb_append_bigint(duckdb_mb_appender *a, int64_t value);                        /* :1132 */
int32_t duckdb_mb_append_double(duckdb_mb_appender *a, double value);                         /* :1148 */
int32_t duckdb_mb_append_varchar(duckdb_mb_appender *a, moonbit_bytes_t value);               /* :1164 */
#ifdef __cplusplus
int32_t duckdb_mb_append_bool(duckdb_mb_appender *a, bool value);                             /* :1189 */
#else
int32_t duckdb_mb_append_bool(duckdb_mb_appender *a, _Bool value);
#endif
int32_t duckdb_mb_append_null(duckdb_mb_appender *a);                                         /* :1205 */
int32_t duckdb_mb_end_row(duckdb_mb_appender *a);                                             /* :1221 */
int32_t duckdb_mb_flush(duckdb_mb_appender *a);                                               /* :1237 */
int32_t duckdb_mb_append_date(duckdb_mb_appender *a, int32_t days);                           /* :1313 (exact days) */
int32_t duckdb_mb_append_timestamp(duckdb_mb_appender *a, int64_t micros);                    /* :1350 (exact micros) */
int32_t duckdb_mb_append_blob(duckdb_mb_appender *a, moonbit_bytes_t data, int32_t length);   /* :1397 */
int32_t duckdb_mb_append_decimal(duckdb_mb_appender *a, uint8_t width, uint8_t scale, int64_t lower, int64_t upper); /* :1447 */
int32_t duckdb_mb_append_interval(duckdb_mb_appender *a, int32_t months, int32_t days, int64_t micros);             /* :1511 */
int32_t duckdb_mb_append_list_varchar(duckdb_mb_appender *a, moonbit_bytes_t *values, int32_t count);               /* :1735 */
int32_t duckdb_mb_append_struct_varchar(duckdb_mb_appender *a, moonbit_bytes_t *field_names, moonbit_bytes_t *field_values,
                                        int32_t field_count);                                                       /* :1792 */
int32_t duckdb_mb_append_map_varchar_varchar(duckdb_mb_appender *a, moonbit_bytes_t *keys, moonbit_bytes_t *values,
                                             int32_t entry_count);                                                  /* :1860 */

#ifdef __cplusplus
}
#endif
#endif /* DUCKDB_MB_GPU_H */
