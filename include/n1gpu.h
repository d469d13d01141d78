/*
 * n1gpu.h — C ABI of libn1gpu.so: the B200-native replacement for the N1QL data-parallel chain
 *
 *     PrimaryScan / Fetch -> Filter -> InitialGroup -> IntermediateGroup -> FinalGroup
 *
 * of pavel-paulau/query.  The reference has no FFI for this path (it is 100 % Go); the boundary it
 * offers is a set of Go interfaces.  Each entry point below names the reference interface it stands
 * in for (file:line under the reference tree); INTEGRATION.md shows the cgo binding a maintainer
 * would add in package `execution`.
 *
 * Conventions: plain C types only; every function returns 0 (N1GPU_OK) or a negative status;
 * the message for the last failure on the calling thread is n1gpu_last_error().  Handles are opaque.
 * Output buffers are caller-owned.  Host pointers unless the name says `dev`.  Thread-safe per
 * handle (one goroutine / OS thread drives one handle at a time).  No caller pointer is retained
 * after a call returns, except where stated.
 */
#ifndef N1GPU_H
#define N1GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes ------------------------------------------------------------------------------ */
#define N1GPU_OK 0
#define N1GPU_E_INVALID (-1)      /* bad argument / handle */
#define N1GPU_E_PARSE (-2)        /* expression / plan / JSON text could not be parsed */
#define N1GPU_E_INELIGIBLE (-3)   /* plan is outside the substituted subset: caller keeps its own operators */
#define N1GPU_E_CUDA (-4)         /* CUDA runtime / driver / NVRTC failure (there is NO CPU fallback) */
#define N1GPU_E_IO (-5)           /* keyspace directory could not be read */
#define N1GPU_E_CANCELLED (-6)    /* n1gpu_query_cancel() was called (execution.Operator.SendStop) */
#define N1GPU_E_NOMEM (-7)

/* ---- value classes (the per-row tag byte of a column; N1QL type order value/value.go:69-79) ------ */
#define N1GPU_C_MISSING 0
#define N1GPU_C_NULL 1
#define N1GPU_C_FALSE 2
#define N1GPU_C_TRUE 3
#define N1GPU_C_INT 4    /* payload = int64 */
#define N1GPU_C_FLOAT 5  /* payload = float64 bits (never integral when it came from a document) */
#define N1GPU_C_STRING 6 /* payload = rank in the column's bytewise-sorted dictionary */
#define N1GPU_C_OTHER 7  /* array / object / binary: referencing such a column makes a plan ineligible */

typedef struct n1gpu_table n1gpu_table;   /* a shredded keyspace (columns + dictionaries), resident in HBM */
typedef struct n1gpu_query n1gpu_query;   /* a compiled Filter + Group chain (one specialised sm_100a kernel) */
typedef struct n1gpu_result n1gpu_result; /* finalised groups (what FinalGroup emits) or a partial state */

/* ---- library ----------------------------------------------------------------------------------- */
/* Selects the CUDA device of this process (one process per GPU).  device < 0: current device.
 * Stands in for nothing in the reference; called from the shim's init().                           */
int n1gpu_init(int device);
int n1gpu_shutdown(void);
const char* n1gpu_last_error(void);
const char* n1gpu_version(void);
/* number of kernel launches issued by this library since load (bench.py's gpu_launches evidence) */
uint64_t n1gpu_launch_count(void);

/* ---- columnar shredder: replaces PrimaryScan + Fetch over datastore/file ---------------------------
 * Reference: execution/scan_primary.go:61-118, execution/fetch.go:54-153,
 * datastore/file/file.go:312-353,711-743 (sorted ReadDir, one ReadFile per key),
 * value/parsed.go:38-98,159-207 (type sniffing, lazy field find), value/value.go:367-430.          */
int n1gpu_table_create(n1gpu_table** out);
/* Declares a column for a field path below the document root; components separated by '\x1f'
 * (e.g. "pricing\x1flist" for `pricing`.`list`).  Must precede any append.  Returns the index.      */
int n1gpu_table_add_column(n1gpu_table* t, const char* path);
int n1gpu_table_find_column(const n1gpu_table* t, const char* path); /* index or -1 */
/* Appends ndocs documents: doc i is bytes [offsets[i], offsets[i+1]) of buf, in primary-key order.
 * threads >= 0: shreds with that many host threads (0 = all cores).
 * threads == -1: the device shredder - the raw JSON is copied to HBM once and parsed there, one thread per
 * document (shred.cu); only documents it cannot decide exactly (escapes in a wanted name/value, numbers
 * outside the exactly-rounded fast path) are re-shredded on the host.  Takes the whole keyspace in one call.
 * Both produce identical columns.                                                                    */
int n1gpu_table_append_json(n1gpu_table* t, const char* buf, const int64_t* offsets, int64_t ndocs, int threads);
/* Reads a file-datastore keyspace directory <root>/<namespace>/<keyspace>: every non-directory entry,
 * sorted by file name, is one document (file.go:711-730).                                           */
int n1gpu_table_load_dir(n1gpu_table* t, const char* dir, int threads);
/* Pre-shredded column (the "columns already resident" metric): nrows payload words of `width` bytes
 * (8: int64 / float64 bits / string rank; 4: string rank) and nrows class bytes (NULL = all C_INT for
 * width 8 / all C_STRING for width 4).  dict_blob/dict_offsets: the column's sorted dictionary
 * (ndict strings, string i = blob[off[i], off[i+1])), or NULL.  Buffers are copied.                 */
int n1gpu_table_set_column(n1gpu_table* t, int col, int width, const void* payload, const uint8_t* tags,
                           int64_t nrows, const char* dict_blob, const int64_t* dict_offsets, int64_t ndict);
/* The same for a column that already lives in DEVICE memory (dev_payload / dev_tags are device pointers of the
 * current device; copied device-to-device into the table's padded arrays).  Integral floats are canonicalised
 * and the column statistics computed by kernels; there is no host staging.  All columns of a table must be set
 * the same way (host or device).  The dictionary still comes from host memory.                        */
int n1gpu_table_set_column_device(n1gpu_table* t, int col, int width, const void* dev_payload, const uint8_t* dev_tags,
                                  int64_t nrows, const char* dict_blob, const int64_t* dict_offsets, int64_t ndict);
/* Builds dictionaries and column statistics, uploads the columns to HBM.  After seal the table is
 * immutable and may be shared by any number of queries.                                             */
int n1gpu_table_seal(n1gpu_table* t);
int64_t n1gpu_table_num_rows(const n1gpu_table* t);
int n1gpu_table_num_columns(const n1gpu_table* t);
/* HBM bytes per row of column `col` that a scan reads: payload width (+1 when its tag bytes vary). */
int n1gpu_table_column_scan_bytes(const n1gpu_table* t, int col);
/* Dictionary exchange for multi-GPU tables (one process per GPU; the dictionary must be global so
 * that string ranks are comparable across ranks).  Before seal: export this rank's distinct strings
 * of a column, then import the merged sorted global dictionary.                                      */
int n1gpu_table_dict_export(n1gpu_table* t, int col, char* blob, int64_t blob_cap, int64_t* offsets,
                            int64_t offsets_cap, int64_t* ndict, int64_t* blob_bytes);
int n1gpu_table_dict_import(n1gpu_table* t, int col, const char* blob, const int64_t* offsets, int64_t ndict);
/* The same in one call: merges nparts sorted, unique dictionaries (e.g. every rank's export, gathered by the caller) with
 * the column's own into the global sorted dictionary and remaps the column's ranks - on the host while the column is
 * staged, by a kernel when its rows already live in HBM (device shredder, set_column_device).                          */
int n1gpu_table_dict_merge(n1gpu_table* t, int col, int nparts, const char* const* blobs, const int64_t* const* offsets, const int64_t* ndicts);
/* Column statistics exchange (int range / class mask) so that every rank compiles the same kernel. */
int n1gpu_table_stats_get(n1gpu_table* t, int col, int64_t stats[8]);
int n1gpu_table_stats_set(n1gpu_table* t, int col, const int64_t stats[8]);
/* A packed document source: `path` holds one JSON document per line (NDJSON) in primary-key order - what a keyspace of
 * more than a few million documents is kept as when one file per document (datastore/file/file.go:312-353) stops being
 * practical.  Same shredding and `threads` meaning as n1gpu_table_load_dir (-1: device shredder); blank lines skipped. */
int n1gpu_table_load_ndjson(n1gpu_table* t, const char* path, int threads);
/* Persistent columnar segments (SURVEY.md 8f row 3): the shredded form of a keyspace for this table's columns - typed
 * columns, class bytes, sorted dictionaries - written once and loaded instead of reading and parsing every document.
 * set_segment_output: n1gpu_table_seal also writes the (host-shredded) columns to `path` under `source_tag`.
 * load_segment: fills the empty table from `path` when it was written for the same columns under the very same tag
 * (*loaded = 1; the caller seals); absent, foreign, truncated or stale files give *loaded = 0 and an untouched table.
 * The tag is the caller's change detector for the keyspace (the plan-level operator uses directory mtime, document
 * count, newest document mtime and total bytes); it plays the part of the reference's invalidation on
 * performOp / Delete (datastore/file/file.go:375-471).  Never place segments inside a keyspace directory: every plain
 * file there is a document (file.go:715-729).                                                                     */
int n1gpu_table_set_segment_output(n1gpu_table* t, const char* path, const char* source_tag);
int n1gpu_table_load_segment(n1gpu_table* t, const char* path, const char* source_tag, int* loaded);
/* Directory in which n1gpu_plan_build keeps one segment per (keyspace, column set); NULL or "" = none (the default,
 * or the N1GPU_SEGMENT_DIR environment variable).                                                                  */
int n1gpu_set_segment_dir(const char* dir);
/* Declares how many rows the whole keyspace holds over ALL partitions (ranks) whose partial group states will be
 * merged with this table's (>= this partition's rows; a single-partition keyspace declares its own row count).
 * Queries compiled afterwards size their overflow proofs with it: exact one-word integer sums, and two row counters
 * sharing one 64-bit table word (needs < 2^32 rows).  Undeclared, a query assumes up to 16 partitions of this size.
 * The reference has no counterpart: its counters are boxed int64 values (algebra/agg_count.go:95-149).             */
int n1gpu_table_set_global_rows(n1gpu_table* t, int64_t rows);
/* Copies a column's staged rows (before seal): payload[nrows] (int64 / float64 bits / dictionary rank)
 * and tags[nrows].  For shredder parity tests; either pointer may be NULL.                           */
int n1gpu_table_column_peek(n1gpu_table* t, int col, int64_t* payload, uint8_t* tags, int64_t nrows);
int n1gpu_table_free(n1gpu_table* t);

/* ---- query: replaces Filter + InitialGroup + IntermediateGroup + FinalGroup -------------------------
 * Reference: execution/filter.go:49-61, group_util.go:18-35, group_initial.go:56-108,
 * group_intermediate.go:56-104, group_final.go:55-118, algebra/agg_*.go.
 * Expressions arrive in the reference's own serialised form: the Stringer text that plan JSON carries
 * (plan/filter.go "condition", plan/group.go "group_keys"/"aggregates"; expression/stringer.go), e.g.
 *   where      "((`d`.`n`) between 10 and 20)"          (NULL/"" = no Filter)
 *   group key  "(`d`.`type`)"
 *   aggregate  "sum((`d`.`n`))"  "count(*)"  "count(distinct (`d`.`x`))"
 * alias = the keyspace term's alias (plan/fetch.go).  N1GPU_E_INELIGIBLE when the chain uses anything
 * outside the subset of SURVEY.md section 8b; the caller then runs its own operators.                */
int n1gpu_query_compile(n1gpu_table* t, const char* alias, const char* where, const char* const* group_keys,
                        int nkeys, const char* const* aggregates, int naggs, n1gpu_query** out);
/* The same for a prepared statement: `$name` / `$1` in the expressions (algebra/param_named.go:63, param_positional.go;
 * Stringer text expression/stringer.go:611-620) take the values of the request (execution.Context.NamedArg /
 * PositionalArg, execution/context.go): param_names[i] ("name", "$name", "1") is bound to the JSON scalar text
 * param_values[i] ("10", "2.5", "\"abc\"", "true", "null"), or to a JSON array of such scalars ("[1, 2.5, \"a\", null]").
 * An array is legal only as the right operand of IN / NOT IN (`x IN $ids`); anywhere else, nested in an array, or an
 * object, it is N1GPU_E_INELIGIBLE.  The list is probed as a device-resident set whose contents are kernel data, so
 * every binding of the statement, whatever its length, shares one compiled kernel.  A parameter without a value fails
 * like the reference's Evaluate ("No value for named parameter $x.").  Constants and parameter values reach the kernel as ARGUMENTS - the
 * generated source only fixes their class - so every binding of a statement, and statements that differ in a bound,
 * share one compiled kernel (n1gpu_jit_stats counts compilations and reuses).                                       */
int n1gpu_query_compile_params(n1gpu_table* t, const char* alias, const char* where, const char* const* group_keys,
                               int nkeys, const char* const* aggregates, int naggs, const char* const* param_names,
                               const char* const* param_values, int nparams, n1gpu_query** out);
int n1gpu_jit_stats(uint64_t* compiled, uint64_t* reused);
/* Runs the chain over the whole table and finalises (FinalGroup).  Blocking.                        */
int n1gpu_query_execute(n1gpu_query* q, n1gpu_result** out);
/* Asynchronous pair for pipelined use: launch enqueues the scan on the query's stream and returns;
 * collect waits and finalises.  One launch may be outstanding per query handle.                    */
int n1gpu_query_launch(n1gpu_query* q);
int n1gpu_query_collect(n1gpu_query* q, n1gpu_result** out);
/* execution.Operator.SendStop (execution/base.go:313-338): makes a running execute return CANCELLED. */
int n1gpu_query_cancel(n1gpu_query* q);
/* The generated CUDA source / kernel facts, for EXPLAIN-style inspection and tests.                 */
const char* n1gpu_query_kernel_source(const n1gpu_query* q);
/* The partitioning kernel of a chain that runs as a partitioned DISTINCT aggregation ("" otherwise): many groups, one
 * DISTINCT operand of few bits, no other per-row accumulator than COUNT(*) - BASELINE config 4's shape.                */
const char* n1gpu_query_part_source(const n1gpu_query* q);
/* info[0]=mode (0 ungrouped, 1 dense shared-memory table, 2 HBM hash 64-bit keys, 3 HBM hash 128-bit)
 * info[1]=accumulator words per group  info[2]=registers/thread  info[3]=grid  info[4]=block
 * info[5]=scan bytes per row  info[6]=static shared bytes  info[7]=dense slots / hash capacity      */
int n1gpu_query_info(const n1gpu_query* q, int64_t info[8]);
/* Device time of the last scan (kernel(s) between CUDA events on the query's stream), nanoseconds.  */
int64_t n1gpu_query_last_scan_ns(const n1gpu_query* q);
/* Rebinds a compiled query to another sealed table with the same schema/dictionaries/statistics
 * (bench.py rotates table copies so that no step finds its input in L2).                            */
int n1gpu_query_rebind(n1gpu_query* q, n1gpu_table* t);
/* Makes the query enqueue its work on a caller-owned CUDA stream (cudaStream_t as void*; NULL = the legacy
 * default stream; (void*)-1 = back to the query's own stream), so that callers can bracket scans with their
 * own CUDA events (bench.py).                                                                              */
int n1gpu_query_set_stream(n1gpu_query* q, void* cuda_stream);
/* The scan is bracketed by two CUDA events (n1gpu_query_last_scan_ns, "#stats" execTime).  Each record costs the
 * GPU front-end a few microseconds - as much as a third of a 10 M-row scan - so throughput-critical callers that
 * time whole regions themselves switch it off.  Default: on.                                                    */
int n1gpu_query_set_timing(n1gpu_query* q, int enable);
int n1gpu_query_free(n1gpu_query* q);

/* ---- multi-GPU: InitialGroup per GPU, IntermediateGroup merge across GPUs ----------------------------
 * Reference: execution/group_intermediate.go:56-104 + the CumulateIntermediate methods of algebra/agg_count.go ... agg_avg_distinct.go.
 * One process per GPU.  Each rank scans its row range and exports its partial groups as fixed-size
 * records in DEVICE memory; the caller moves records between ranks (NCCL all-to-all / all-gather over
 * NVLink - torch.distributed in this repo, ncclSend/Recv from Go); the owner imports and finalises.
 * Record layout: record_words 64-bit words = [key_lo, key_hi, acc words...]; DISTINCT entries travel
 * as 2-word records [lo, hi].  owner(record) = mix(key) % nranks, computed by partial_partition.     */
int n1gpu_query_scan_partial(n1gpu_query* q);                       /* scan only, state stays on device */
int n1gpu_query_partial_counts(n1gpu_query* q, int64_t* ngroups, int64_t* ndistinct, int* record_words);
/* Writes the partial groups, bucketed by owner rank, into dev_records (capacity in records) and the
 * per-owner record counts into counts[nranks] (host).  Same for DISTINCT entries.                   */
int n1gpu_query_partial_export(n1gpu_query* q, int nranks, void* dev_records, int64_t cap_records,
                               int64_t* counts, void* dev_distinct, int64_t cap_distinct, int64_t* dcounts);
/* Clears the local state, then merges n records (from any ranks) into it.                           */
int n1gpu_query_partial_reset(n1gpu_query* q);
int n1gpu_query_partial_import(n1gpu_query* q, const void* dev_records, int64_t n, const void* dev_distinct, int64_t nd);
int n1gpu_query_finalize(n1gpu_query* q, n1gpu_result** out);
/* Small-state chains (no GROUP BY, or a dense shared-memory table; no DISTINCT): the whole partial state is
 * nwords 64-bit accumulator words at *dev_words.  Pipelined multi-GPU step without host round trips:
 *   n1gpu_query_launch(q);                       enqueue the scan on the query's stream
 *   ncclAllGather(*dev_words -> all, nwords)      on the same stream (every rank's words, in rank order)
 *   n1gpu_query_merge_words(q, all, nranks);      enqueue the fold over ranks (result also lands, zero-copy, in
 *                                                 pinned host memory)
 *   n1gpu_query_collect(q, &res);                 wait + FinalGroup
 * n1gpu_query_state_words fails with N1GPU_E_INVALID for hash-table / DISTINCT chains (use partial_export).  */
int n1gpu_query_state_words(n1gpu_query* q, void** dev_words, int64_t* nwords);
int n1gpu_query_merge_words(n1gpu_query* q, const void* dev_all_words, int nranks);
/* The combine operation of every accumulator word (N1GPU_OP_*: 0 add u64, 1 add f64, 2 min i64, 3 max i64, 4 min u64,
 * 5 max u64, 6 or u64), word w occupying dev_words[w * slots, (w + 1) * slots).  Returns the number of words (also
 * when ops is NULL or cap is too small).  A caller whose collective library reduces with these operations (NCCL:
 * sum / min / max) can merge a direct-indexed table in place with one all-reduce per run of equal operations
 * instead of all-gather + merge_words.                                                                  */
int n1gpu_query_word_ops(const n1gpu_query* q, int* ops, int cap);

/* Fused merge for small-state chains: instead of a collective, the scan kernel's last block stores this rank's
 * accumulator words straight into every peer's mailbox over NVLink (peer stores + a release flag), and a 1-block
 * kernel on each rank folds its own mailbox once all flags arrived.  A step is then launch + collect, no NCCL.
 * Setup, once per process: create (HBM buffer of 64 slots x nranks cells of max_words+1 words), exchange the
 * 64-byte CUDA IPC handles between the ranks (any transport), open_peers(handles of all ranks, rank-major),
 * then n1gpu_query_set_mailbox on every query that should use it.  All ranks must launch the same sequence of
 * steps on a mailbox.  A peer that never delivers makes collect fail with N1GPU_E_CUDA after ~10 s.           */
typedef struct n1gpu_mailbox n1gpu_mailbox;
int n1gpu_mailbox_create(int nranks, int rank, int64_t max_words, n1gpu_mailbox** out);
/* The same with an ARENA of arena_bytes behind the mailbox cells, mapped into every rank like the cells.  A query whose
 * group table is direct-indexed in HBM (slot == packed key on every rank; no DISTINCT) places its table there when the
 * mailbox is set on it (double-buffered: 2 x slots x words x 8 bytes; every rank must set its queries in the same order),
 * and the Intermediate -> Final merge becomes owner-sharded and collective-free: each rank raises a flag in every peer's
 * flag row when its scan is complete, and n1gpu_query_collect on rank r waits for all flags, then folds slot range r of
 * EVERY rank's table with plain loads over NVLink while it finalises (ComputeFinal) exactly those groups - rank r's result
 * holds its 1/nranks of the groups.  Replaces execution/group_intermediate.go:56-104 + group_final.go:55-118 across ranks. */
int n1gpu_mailbox_create_arena(int nranks, int rank, int64_t max_words, int64_t arena_bytes, n1gpu_mailbox** out);
int n1gpu_mailbox_ipc_handle(n1gpu_mailbox* mb, uint8_t handle[64]);
/* In-process wiring (several ranks driven by one process, peer access enabled by the caller - or one device in tests):
 * the device base pointer of rank `rank`'s mailbox buffer, instead of an IPC handle.                                   */
int n1gpu_mailbox_set_peer(n1gpu_mailbox* mb, int rank, void* dev_base);
void* n1gpu_mailbox_base(n1gpu_mailbox* mb);
int n1gpu_mailbox_open_peers(n1gpu_mailbox* mb, const uint8_t* handles);
int n1gpu_mailbox_free(n1gpu_mailbox* mb);
int n1gpu_query_set_mailbox(n1gpu_query* q, n1gpu_mailbox* mb);
/* How the query merges across the ranks of its mailbox: 0 = not through the arena (small states are pushed through the
 * mailbox cells, hash tables / DISTINCT sets are exported as records for the caller to exchange), 1 = its direct-indexed
 * table lives in the arena and collect() folds + finalises this rank's slot range of every rank's table, 2 = partitioned
 * DISTINCT aggregation whose records live in the arena: this rank aggregates and finalises its range of partitions.
 * With 1 and 2 a step is launch() + collect() on every rank, and each rank's result holds its share of the groups.      */
int n1gpu_query_peer_mode(const n1gpu_query* q);

/* ---- result: what FinalGroup sends downstream ---------------------------------------------------------
 * Per group: the group-key values and, per aggregate (in the order given to compile), the final value
 * (algebra ComputeFinal).  A value is a class byte + 64-bit payload; string payloads index the result's
 * string table.  Downstream contract: algebra/aggregate.go:97-118, execution/project_initial.go:98-144. */
int64_t n1gpu_result_num_groups(const n1gpu_result* r);
int n1gpu_result_num_keys(const n1gpu_result* r);
int n1gpu_result_num_aggregates(const n1gpu_result* r);
/* key_cls/key_val: [ngroups][nkeys]; agg_cls/agg_val: [ngroups][naggs] (row-major).                 */
int n1gpu_result_fetch(const n1gpu_result* r, uint8_t* key_cls, int64_t* key_val, uint8_t* agg_cls, int64_t* agg_val);
int n1gpu_result_string(const n1gpu_result* r, int64_t index, const char** ptr, int64_t* len);
/* stats[0]=rows scanned (#itemsIn) stats[1]=groups (#itemsOut) stats[2]=scan ns (execTime)
 * stats[3]=shred+upload ns (servTime) stats[4]=HBM bytes scanned stats[5]=kernel launches          */
int n1gpu_result_stats(const n1gpu_result* r, int64_t stats[8]);
int n1gpu_result_free(n1gpu_result* r);

/* ---- plan level: the reference's plan.Visitor / execution.Operator contract ----------------------------
 * Reference: plan/visitor.go:12-123, plan/op_registry.go:18-29 (plans round-trip through JSON),
 * execution/build.go:22-45,473-491, execution/execution.go:26-64.
 * n1gpu_plan_build takes the reference's own plan JSON (what EXPLAIN prints / PREPARE stores), looks for
 *   Sequence[ PrimaryScan, Fetch, (Parallel(Sequence[Filter?, InitialGroup]) | Filter?, InitialGroup),
 *             IntermediateGroup, FinalGroup, ...rest ]
 * and, when eligible, returns an operator handle that replaces that prefix; `rest_index` receives the
 * index of the first child the caller must still run.  datastore_root is cbq-engine's -datastore dir.  */
typedef struct n1gpu_operator n1gpu_operator;
int n1gpu_plan_build(const char* plan_json, const char* datastore_root, n1gpu_operator** out, int* rest_index);
/* The same, also taking over the operators BEHIND FinalGroup when every one of them up to FinalProject is within the
 * subset (SURVEY.md 8f rows 1-2): Let (LETTING, plan/let.go), Filter (HAVING, plan/filter.go), InitialProject and
 * FinalProject (plan/project.go; no star, raw or DISTINCT projection), Order / Offset / Limit (plan/order.go,
 * plan/offset.go, plan/limit.go) of the enclosing Sequence.  Their expressions may use group keys, the aggregates of
 * the group operators, LETTING variables, explicit projection aliases (ORDER BY), the operators of Filter and ROUND
 * (expression/func_num.go:1304-1336).
 * `rest_index` then points behind the consumed children of the chain's Sequence, `outer_rest_index` behind those
 * consumed from the enclosing Sequence (0: none).  A plan whose tail is not eligible builds like n1gpu_plan_build
 * (n1gpu_operator_tail_operators reports an empty list) and the caller keeps its own operators after FinalGroup.
 * Replaces: execution/let.go:50-62, filter.go:49-61, project_initial.go:52-144, project_final.go:51-59,
 * order.go:50-170 (ties: the reference's sort.Sort is not stable, here they keep group order), offset.go:53-83,
 * limit.go:53-85.                                                                                                  */
int n1gpu_plan_build_tail(const char* plan_json, const char* datastore_root, n1gpu_operator** out, int* rest_index,
                          int* outer_rest_index);
/* Comma-separated names of the consumed tail operators, in execution order ("" = none).              */
int n1gpu_operator_tail_operators(const n1gpu_operator* op, char* buf, int64_t cap, int64_t* len);
/* Runs the tail over the result of run_once: the rows FinalProject sends, as a JSON array of objects
 * (field names sorted, MISSING values left out: value/object.go:246-255); *rows = number of rows.    */
int n1gpu_operator_run_tail(n1gpu_operator* op, const n1gpu_result* r, char* buf, int64_t cap, int64_t* len, int64_t* rows);
/* Builds a result for this operator from flat arrays in n1gpu_result_fetch layout (string payloads index the
 * nstrings strings blob[offsets[i] .. offsets[i+1])): the groups of several ranks gathered in one place - each
 * owner finalises its share of the groups (SURVEY.md 8e) and ORDER BY / LIMIT need all of them - or groups that a
 * caller's own operators produced.  The tail runs over it like over the result of run_once.          */
int n1gpu_operator_import_result(const n1gpu_operator* op, int64_t ngroups, const uint8_t* key_cls, const int64_t* key_val,
                                 const uint8_t* agg_cls, const int64_t* agg_val, const char* blob, const int64_t* offsets,
                                 int64_t nstrings, n1gpu_result** out);
/* Group keys / aggregates of the operator's group operators (the row widths of import_result).       */
int n1gpu_operator_num_keys(const n1gpu_operator* op);
int n1gpu_operator_num_aggregates(const n1gpu_operator* op);
/* execution.Operator.RunOnce: scans, filters, groups; the result is what FinalGroup would have sent. */
int n1gpu_operator_run_once(n1gpu_operator* op, n1gpu_result** out);
int n1gpu_operator_send_stop(n1gpu_operator* op);
/* The operator as plan JSON with "#stats" (execution/base.go:896-949 marshalTimes).                  */
int n1gpu_operator_marshal_json(n1gpu_operator* op, char* buf, int64_t cap, int64_t* len);
/* Rows as the JSON the downstream InitialProject would see: one object per group
 * {"<alias>": {<key paths>}, "aggregates": {"<agg text>": value}}                                    */
int n1gpu_result_to_json(const n1gpu_result* r, char* buf, int64_t cap, int64_t* len);
int n1gpu_operator_free(n1gpu_operator* op);

#ifdef __cplusplus
}
#endif
#endif /* N1GPU_H */
