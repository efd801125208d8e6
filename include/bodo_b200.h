/*
 * bodo_b200.h — C ABI of libbodo_b200.so: the B200-native replacement for Bodo's streaming
 * hash groupby / hash join / row->rank shuffle hot path.
 *
 * Every entry point mirrors one reference FFI symbol (cited per function, paths relative to the
 * reference checkout). Differences from the reference ABI, all deliberate:
 *   - tables cross the boundary as `b200_table` (plain column descriptors: data pointer, Arrow
 *     validity bitmap, Bodo_CTypes / bodo_array_type codes) instead of `table_info*`;
 *   - errors are reported by return code + b200_last_error() instead of the CPython error
 *     indicator (reference: PyErr_SetString, bodo/libs/streaming/_groupby.cpp:4669-4675);
 *   - input tables are BORROWED for the duration of the call (the reference steals them).
 * No torch / CUDA types appear in any signature: streams are passed as void* (cudaStream_t).
 *
 * This header is also parsed by cffi (bodo_b200/_lib.py): keep it plain C89 declarations;
 * lines starting with '#' are stripped before parsing.
 */
#ifndef BODO_B200_H
#define BODO_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* ---- data model (reference: bodo/libs/_bodo_common.h:331-359 Bodo_CTypes, :515-532 bodo_array_type,
 *      :927 array_info, :1819 table_info) ---- */

/* b200_column.c_type uses Bodo_CTypes codes: INT8=0 UINT8=1 INT32=2 UINT32=3 INT64=4 FLOAT32=5
 * FLOAT64=6 UINT64=7 INT16=8 UINT16=9 _BOOL=11 DATE=13 DATETIME=15 TIMEDELTA=16.
 * b200_column.arr_type uses bodo_array_type codes: NUMPY=0, NULLABLE_INT_BOOL=2. */
typedef struct b200_column {
    void* data;        /* contiguous values, length * itemsize bytes (host or device, see b200_table.device) */
    uint8_t* validity; /* Arrow validity bitmap (bit i%8 of byte i/8, 1 = valid) or NULL = all valid */
    int64_t length;
    int32_t c_type;
    int32_t arr_type;
} b200_column;

typedef struct b200_table {
    int64_t n_rows;
    int32_t n_cols;
    int32_t device; /* -1: pointers are host memory; >= 0: CUDA device ordinal owning the pointers */
    b200_column* cols;
} b200_table;

/* Last error message of the calling thread ("" if none). Every int-returning entry point returns
 * a negative value on error; pointer-returning ones return NULL. */
const char* b200_last_error(void);

/* Library/runtime probes (used by tests and __graft_entry__). b200_device_count() returns 0 without
 * a GPU and never raises; all compute entry points fail with an error instead of falling back. */
int b200_abi_version(void);
int b200_device_count(void);

/* ---- streaming hash groupby (reference door 1: bodo/libs/streaming/_groupby.cpp) ---- */

/* groupby_state_init_py_entry (_groupby.cpp:4917-4970). Keys are the first n_keys (1..4, integer/date typed;
 * multi-column keys on the non-sharded path only) columns of every build batch; n_funcs may be 0 (select
 * distinct / drop_duplicates, reference: physical/aggregate.h:198-227); ftypes are Bodo_FTypes (groupby/_groupby_ftypes.h:17-110: size=4 sum=6 count=7 mean=14
 * min=15 max=16); f_in_offsets/f_in_cols is the CSR map function -> physical input column
 * (streaming/_groupby.h:1059-1070). Arguments of the reference that only concern window functions,
 * MRNF, sort keys and the host operator pool are dropped. `pandas_drop_na`: drop rows with NA keys
 * (filter_na_keys, _groupby.cpp:4278-4309). `parallel`: state is one shard of n_pes; ownership
 * is hash_to_rank(key) (bodo/libs/_shuffle.h:5-7). `expected_groups` is a sizing hint (0 = unknown).
 * `stream` is a cudaStream_t all work is enqueued on (NULL = legacy default stream). */
void* b200_groupby_state_init(int64_t operator_id, const int8_t* build_arr_c_types,
                              const int8_t* build_arr_array_types, int32_t n_build_arrs,
                              const int32_t* ftypes, const int32_t* f_in_offsets,
                              const int32_t* f_in_cols, int32_t n_funcs, uint64_t n_keys,
                              int64_t output_batch_size, int32_t parallel, int32_t pandas_drop_na,
                              int32_t device, int32_t n_pes, int32_t myrank,
                              int64_t expected_groups, void* stream);

/* groupby_build_consume_batch_py_entry (_groupby.cpp:4663-4676). Returns 1 when the build is globally
 * finished (is_last was passed), 0 otherwise, <0 on error. *request_input is always set to 1 (the GPU
 * state sizes its table up front and never back-pressures). */
int b200_groupby_build_consume_batch(void* state, const b200_table* in_table, int32_t is_last,
                                     int32_t is_final_pipeline, int32_t* request_input);

/* Multi-rank exchange step, replacing GroupbyIncrementalShuffleState (streaming/_groupby.cpp:1558-1873)
 * + shuffle_issend/irecv (streaming/_shuffle.cpp:567-652): after the last local batch,
 *   1. b200_groupby_shuffle_prepare: compacts the local partial aggregates and radix-partitions them by
 *      hash_to_rank into one packed send buffer (layout: see DESIGN.md "partial-aggregate wire format");
 *      writes n_pes send row counts (host) and returns the packed row width in bytes;
 *   2. the host exchanges counts and bytes (ncclSend/Recv all-to-all-v; torch.distributed plumbing);
 *   3. b200_groupby_shuffle_combine merges the received partial rows (combine functions of
 *      groupby/_groupby_update.cpp:41-57: count/size/mean -> sum, min -> min, max -> max).
 * send_buf must hold b200_groupby_shuffle_send_bytes(state) bytes on the state's device. */
int64_t b200_groupby_shuffle_prepare(void* state, int64_t* send_row_counts);
int64_t b200_groupby_shuffle_send_bytes(void* state);
int b200_groupby_shuffle_pack(void* state, void* send_buf);
int b200_groupby_shuffle_combine(void* state, const void* recv_buf, int64_t n_recv_rows);

/* Fused form of the same exchange (pack + all-to-all in one kernel over NVLink peer memory; what
 * shuffle_issend/irecv + the combine step do in the reference, streaming/_shuffle.cpp:567-652):
 * every rank owns a receive slab in memory mapped into all peers (CUDA IPC / symmetric memory, set up once per
 * process group by the host layer): 256 header bytes + n_pes segments of cap_rows rows of
 * b200_groupby_exchange_row_bytes(state) bytes.
 *   1. b200_groupby_exchange_fused_pack: one pass over the local table stores every partial row another rank
 *      owns straight into that rank's slab (peer_slabs_dev = device array of the n_pes slab addresses) and
 *      posts the per-source row counts into the peers' headers;
 *   2. a barrier across the ranks on the same stream (host layer);
 *   3. b200_groupby_exchange_fused_combine merges the rows received in my_slab.
 * Nothing here synchronises with the host.  If some rank's share for one destination exceeded cap_rows no
 * rank combines and b200_groupby_finalize returns -2: run the prepare/pack/combine exchange above and
 * finalize again (the local tables are intact). */
int64_t b200_groupby_exchange_row_bytes(void* state);
int b200_groupby_exchange_fused_pack(void* state, void* const* peer_slabs_dev, int64_t cap_rows);
int b200_groupby_exchange_fused_combine(void* state, const void* my_slab, int64_t cap_rows);

/* FinalizeBuild (_groupby.cpp:4062-4256): evaluates the output columns (mean_eval etc.). Called
 * implicitly by the first produce call; exposed so the exchange step can be timed separately.
 * Returns the number of output rows (groups owned by this shard), or -2 (see the fused exchange). */
int64_t b200_groupby_finalize(void* state);

/* groupby_produce_output_batch_py_entry (_groupby.cpp:4772-4783). Fills `out` (caller provides
 * out->cols with room for n_keys + n_funcs descriptors) with pointers to library-owned device
 * columns holding the next <= output_batch_size groups; they stay valid until the next produce call
 * or delete. Sets *out_is_last. Output order of groups is unspecified (as in the reference). */
int b200_groupby_produce_output_batch(void* state, b200_table* out, int32_t* out_is_last,
                                      int32_t produce_output);

/* delete_groupby_state (_groupby.cpp:5246). */
void b200_delete_groupby_state(void* state);

/* Metrics (subset of GroupbyMetrics, streaming/_groupby.h:106-223): 0 n_groups, 1 table capacity,
 * 2 rows consumed, 3 table rebuilds, 4 kernel launches so far, 5 rows replayed from the fail list,
 * 6 accumulated device time of the consume kernel in microseconds (CUDA events on the state's stream;
 * only when profiling was enabled by querying metric 100 first), 7 consume-kernel launches, 8 SM-partitioned
 * (SPG) launches, 9 rows/partials replayed from the SPG retry lists, 10 low-cardinality (LC) launches, 11 small batches
 * that were coalesced on the device before a fast-path launch, 12 SPG launches of the generic signature (SPG-G: nullable /
 * 4-byte keys or values, mean / min / max; included in 8), 13 groups in the table right now (exact: reads the device counter,
 * synchronises the state's stream), 14 SPG launches with narrow (int32 key, int32 value) bucket rows (SPG-N; included in 8). */
/* nunique keeps one nested distinct state over (key, value) per value column (owned by `state`).  A sharded caller exchanges every
 * nested state (b200_groupby_exchange_fused_pack / _combine + b200_groupby_finalize on the handle returned here — a key's pairs are
 * owned where the key is owned) BEFORE it exchanges and finalizes the outer state; single-GPU callers never need these. */
int32_t b200_groupby_num_inner_states(void* state);
void* b200_groupby_inner_state(void* state, int32_t i);

int64_t b200_groupby_get_metric(void* state, int32_t which);

/* ---- streaming hash join (reference: bodo/libs/streaming/_join.cpp) ---- */

/* join_state_init_py_entry (_join.cpp:4087-4136). Equi-join on the first n_keys (1..4) columns of each side:
 * key column j of the build side is compared with key column j of the probe side, on the values widened to
 * int64; key columns are integer / date / datetime / timedelta / bool typed, and both sides have the same byte
 * width at every key position. build_table_outer / probe_table_outer select right/left/full-outer semantics.
 * `is_na_equal` is the HashJoinState option of the same name: 0 (what join_state_init_py_entry constructs:
 * a row with an NA in ANY key column matches nothing, _join.cpp:3180) or 1 (what bodo/pandas/physical/join.h:267
 * passes, pandas merge semantics: NA equals NA at the same key position and never equals a value).
 * n_probe_arrs may be 0: the probe schema is then taken from the first probe batch. */
void* b200_join_state_init(int64_t operator_id, const int8_t* build_arr_c_types,
                           const int8_t* build_arr_array_types, int32_t n_build_arrs,
                           const int8_t* probe_arr_c_types, const int8_t* probe_arr_array_types,
                           int32_t n_probe_arrs, uint64_t n_keys, int32_t build_table_outer,
                           int32_t probe_table_outer, int32_t is_na_equal, int64_t output_batch_size,
                           int32_t device, int64_t expected_build_rows, void* stream);

/* join_build_consume_batch_py_entry (_join.cpp:4149-4185): appends a build batch; on is_last builds the
 * hash table + CSR groups (JoinPartition::BuildHashTable / FinalizeGroups, _join.cpp:381-512). */
int b200_join_build_consume_batch(void* state, const b200_table* in_table, int32_t is_last,
                                  int32_t* request_input);

/* join_probe_consume_batch_py_entry (_join.cpp:4205-4260): probes one batch and materialises the joined
 * rows (kept build columns then kept probe columns, reference order: build table first) into
 * library-owned device columns described by `out` (valid until the next probe call). *total_rows
 * receives the number of output rows of this call. */
int b200_join_probe_consume_batch(void* state, const b200_table* in_table,
                                  const uint64_t* kept_build_cols, int64_t n_kept_build,
                                  const uint64_t* kept_probe_cols, int64_t n_kept_probe,
                                  b200_table* out, int64_t* total_rows, int32_t is_last,
                                  int32_t* out_is_last);

/* delete_join_state (_join.cpp:4429). */
void b200_delete_join_state(void* state);
/* Join kind, to be called between init and the first build batch: mark join (HashJoinState::is_mark_join, _join.h:402 — every
 * probe row goes out once, no build columns, plus one trailing BOOL column "has a match": `out->cols` needs n_kept_probe + 1
 * descriptors) or probe-side anti join (the is_anti_join template argument of the reference's probe, _join.cpp:763-767 — a probe
 * row goes out, with NULL build columns, iff no build row matches).  build_table_outer must be false for both. */
int b200_join_set_kind(void* state, int32_t is_mark_join, int32_t is_anti_join);

/* Runtime join filter (HashJoinState::RuntimeFilter, _join.h:1060-1095; bloom filter bodo/libs/gpu_bloom_filter.cu:60-201; key
 * min / max _join.cpp:3199-3238), available once the build side is complete, for single-column keys only: the three calls return
 * an error for a state with n_keys > 1.
 * b200_join_build_filter builds a split-block bloom filter over the build keys (n_bloom_blocks 32-byte blocks, 0 = one per 32 build
 * rows) and their min / max; it returns the device address of the filter words (n_blocks * 8 uint32) so that the ranks of a sharded
 * join can OR their filters together in place (all ranks pass the same n_bloom_blocks; b200_join_set_key_bounds installs the
 * reduced bounds).  b200_join_runtime_filter writes keep_out[i] = 1 for the rows of a DEVICE-resident table that can still find a
 * partner (key not NA, inside the bounds, bloom hit): the rows a probe-side scan may drop before they are shuffled or probed
 * (inner and build-outer joins only — an outer probe side must keep its rows). */
int b200_join_build_filter(void* state, int64_t n_bloom_blocks, void** bloom_words_dev, int64_t* n_blocks_out, int64_t* key_min_max);
int b200_join_set_key_bounds(void* state, int64_t key_min, int64_t key_max);
int b200_join_runtime_filter(void* state, const b200_table* in_table, int32_t key_col, int32_t use_min_max, int32_t use_bloom,
                             uint8_t* keep_out);

/* Operator metrics (the reference's JoinMetrics, bodo/libs/streaming/_join.h): 0 build rows, 1 hash-table slots, 2 probe rows,
 * 3 output rows, 4 kernel launches, 5 probe batches through a fused (unique-build-key) probe kernel, 6 of those through the
 * inline-payload kernel (key + payload in one 32-byte slot), 7 inline-payload table builds. */
int64_t b200_join_get_metric(void* state, int32_t which);

/* ---- row -> rank shuffle (reference: bodo/libs/_shuffle.cpp) ---- */

/* hash_keys_table(SEED_HASH_PARTITION) + hash_to_rank (bodo/libs/_array_hash.cpp:76-109,
 * _shuffle.h:5-7): dest[i] = (uint32)XXH3_64bits_withSeed(&key[i], 8, 0xb0d01289) % n_pes. Writes
 * per-row destinations (device int32) — exposed for placement-parity tests. */
int b200_hash_to_rank(const b200_table* in_table, int32_t n_pes, int32_t* dest_out, void* stream);
/* hash_keys_table(table, n_keys, SEED_HASH_PARTITION) (bodo/libs/_array_hash.cpp:1599-1621) over the first n_keys (1..4)
 * columns: integer / date columns hash their sizeof(T) raw bytes, float columns go through _Py_HashDouble first
 * (:119-170), NA -> hash_na_val, further columns are folded in with hash_combine_boost (:41-56).  Writes the 32-bit row
 * hashes (hash_out, device uint32, may be NULL) and / or hash % n_pes (dest_out, device int32, may be NULL). */
int b200_hash_keys_table(const b200_table* in_table, int64_t n_keys, int32_t n_pes, int32_t* dest_out,
                         uint32_t* hash_out, void* stream);

/* mpi_comm_info::set_send_count + fill_send_array (bodo/libs/_shuffle.cpp:94-163,345-368,477+) as one
 * radix-partition pass: histogram of destinations, exclusive scan, stable scatter of every column
 * into per-destination contiguous segments. `out` columns (device, same schema/length as the input,
 * provided by the caller) receive the rows grouped by destination; send_counts (host, n_pes) the
 * rows per destination. Validity bitmaps are re-packed per destination segment at byte granularity
 * (segment d starts at byte offset of a fresh bitmap: see DESIGN.md). */
int b200_shuffle_partition(const b200_table* in_table, int64_t n_keys, int32_t n_pes,
                           b200_table* out, int64_t* send_counts, void* stream);
/* Same, and also writes the source row of every output row to perm_out_dev (device int64[n_rows]);
 * used by the parity tests to compare the placement with the oracle row by row. */
int b200_shuffle_partition_perm(const b200_table* in_table, int64_t n_keys, int32_t n_pes,
                                b200_table* out, int64_t* send_counts, int64_t* perm_out_dev,
                                void* stream);

/* Receive side of shuffle_table: turns the n_src per-source validity segments (each ceil(counts[j]/8) bytes, back to
 * back, in source-rank order — what the all-to-all-v of the per-destination bitmaps delivers) into one contiguous Arrow
 * bitmap of sum(counts) rows.  out_bitmap must hold 4 * ceil(sum(counts) / 32) bytes on `device`. */
int b200_merge_segment_bitmaps(const uint8_t* segments, const int64_t* counts, int32_t n_src,
                               uint8_t* out_bitmap, int32_t device, void* stream);

/* ---- fused filter + projection front end (reference: bodo/pandas/physical/filter.h, project.h, expression.{h,cpp};
 *      GPU twins gpu_expression.cpp:601+ / gpu_filter.h:143 built on cudf::ast + apply_boolean_mask) ---- */

/* One postfix instruction: op (EX_* below) + 64-bit argument (column index, or the bits of an int64 / double constant).
 * EX_COL=0 CONST_I64=1 CONST_F64=2 ADD=3 SUB=4 MUL=5 DIV=6 LT=7 LE=8 GT=9 GE=10 EQ=11 NE=12 AND=13 OR=14 NOT=15
 * TO_F64=16 TO_I64=17 IS_NULL=18 NEG=19 END=20.  A program is a sequence of expressions, each terminated by END and
 * leaving one value; arithmetic / comparisons propagate NA, AND / OR are Kleene, a NA predicate drops the row. */
typedef struct b200_expr_instr { int32_t op; int32_t pad; int64_t arg; } b200_expr_instr;

/* Evaluates the predicate (expression starting at instruction pred_start; -1 = keep every row) and the n_out output
 * expressions (starting at out_starts[j]) of every row of a device-resident table in ONE kernel, compacting the surviving
 * rows: out->cols[j] (device buffers of in_table->n_rows items provided by the caller, c_type = storage type, validity =
 * bitmap buffer or NULL) receive the rows that pass.  Returns the number of output rows (< 0 on error). */
int64_t b200_filter_project(const b200_table* in_table, const void* program, int32_t n_instr, int32_t pred_start,
                            const int32_t* out_starts, int32_t n_out, b200_table* out, void* stream);

/* out[i] = map[in[i]] (0 where invalid): the transpose step of dictionary unification
 * (DictionaryBuilder::UnifyDictionaryArray, bodo/libs/_dict_builder.cpp): batch-local dictionary indices -> global ids. */
int b200_remap_i32(const int32_t* in_dev, const uint8_t* valid_dev, int64_t n, const int32_t* map_dev, int32_t map_len,
                   int32_t* out_dev, int32_t device, void* stream);

/* ---- helpers for host code that does not link CUDA ---- */
void* b200_device_malloc(int32_t device, int64_t nbytes);
void b200_device_free(int32_t device, void* p);
/* Scratch memory (owner buckets, retry lists, staging) comes from a process-wide, stream-ordered per-device pool that
 * keeps freed blocks for the next operator state; this returns pooled blocks beyond keep_bytes to the driver. */
int64_t b200_pool_trim(int32_t device, int64_t keep_bytes);
int b200_memcpy_d2h(void* dst_host, const void* src_dev, int64_t nbytes, void* stream);
int b200_memcpy_h2d(void* dst_dev, const void* src_host, int64_t nbytes, void* stream);
int b200_stream_synchronize(void* stream);

/* Synthetic table generator used by bench.py (counter-based, seeded; mirrored by the numpy generator
 * in bodo_b200/synth.py so the oracle sees the same rows): key = mix64(seed_k, row) % n_groups,
 * val = (int64)(mix64(seed_v, row) % 1000) - 500 (INT64) or u01 (FLOAT64). */
int b200_synth_fill(void* key_out, void* val_out, int64_t row_start, int64_t n_rows, int64_t n_groups,
                    uint64_t seed, int32_t val_c_type, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BODO_B200_H */
