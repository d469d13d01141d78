// abi.cpp — the extern "C" surface declared in include/n1gpu.h.  Exceptions never cross it.
#include <cstring>
#include <mutex>

#include "execution.hpp"
#include "query.hpp"
#include "table.hpp"

using namespace n1;

// the public class codes are the value classes of n1ql_value.cuh
static_assert(N1GPU_C_MISSING == C_MISSING && N1GPU_C_NULL == C_NULL && N1GPU_C_FALSE == C_FALSE && N1GPU_C_TRUE == C_TRUE &&
                  N1GPU_C_INT == C_INT && N1GPU_C_FLOAT == C_FLOAT && N1GPU_C_STRING == C_STRING && N1GPU_C_OTHER == C_OTHER,
              "N1GPU_C_* differ from the value classes");

struct n1gpu_table { Table t; };
struct n1gpu_query { std::unique_ptr<Query> q; };
struct n1gpu_result { std::unique_ptr<Result> r; };
struct n1gpu_operator {
    std::unique_ptr<execution::GpuGroupAggregate> op;
    // the rows of the last run_tail, kept between the size query and the call that fills the caller's buffer
    const void* tail_of = nullptr;
    std::string tail_rows;
    int64_t tail_count = 0;
};

static thread_local std::string g_last_error;

template <class F> static int guard(F&& f) {
    try {
        f();
        return N1GPU_OK;
    } catch (const Error& e) {
        g_last_error = e.what();
        return e.code;
    } catch (const std::bad_alloc&) {
        g_last_error = "out of host memory";
        return N1GPU_E_NOMEM;
    } catch (const std::exception& e) {
        g_last_error = e.what();
        return N1GPU_E_INVALID;
    }
}
#define REQUIRE(p) do { if (!(p)) N1_THROW(N1GPU_E_INVALID, "null argument: %s", #p); } while (0)

extern "C" {

int n1gpu_init(int device) {
    return guard([&] {
        int n = 0;
        CK(cudaGetDeviceCount(&n));
        if (n == 0) N1_THROW(N1GPU_E_CUDA, "no CUDA device: libn1gpu has no CPU fallback");
        if (device >= 0) CK(cudaSetDevice(device));
        CK(cudaFree(0));
    });
}
int n1gpu_shutdown(void) { return N1GPU_OK; }
const char* n1gpu_last_error(void) { return g_last_error.c_str(); }
const char* n1gpu_version(void) { return "n1gpu 0.1 (sm_100a)"; }
uint64_t n1gpu_launch_count(void) { return (uint64_t)g_launches.load(); }

// ---- table ----------------------------------------------------------------------------------------------
int n1gpu_table_create(n1gpu_table** out) {
    return guard([&] { REQUIRE(out); *out = new n1gpu_table(); });
}
int n1gpu_table_add_column(n1gpu_table* t, const char* path) {
    int idx = -1;
    int rc = guard([&] { REQUIRE(t); REQUIRE(path); idx = t->t.add_column(path); });
    return rc == N1GPU_OK ? idx : rc;
}
int n1gpu_table_find_column(const n1gpu_table* t, const char* path) {
    if (!t || !path) return -1;
    return t->t.find_column(path);
}
int n1gpu_table_append_json(n1gpu_table* t, const char* buf, const int64_t* offsets, int64_t ndocs, int threads) {
    return guard([&] { REQUIRE(t); REQUIRE(offsets); t->t.append_json(buf, (const i64*)offsets, ndocs, threads); });
}
int n1gpu_table_load_dir(n1gpu_table* t, const char* dir, int threads) {
    return guard([&] { REQUIRE(t); REQUIRE(dir); t->t.load_dir(dir, threads); });
}
int n1gpu_table_set_column(n1gpu_table* t, int col, int width, const void* payload, const uint8_t* tags, int64_t nrows,
                           const char* dict_blob, const int64_t* dict_offsets, int64_t ndict) {
    return guard([&] { REQUIRE(t); REQUIRE(payload || nrows == 0); t->t.set_column(col, width, payload, tags, nrows, dict_blob, (const i64*)dict_offsets, ndict); });
}
int n1gpu_table_set_column_device(n1gpu_table* t, int col, int width, const void* dev_payload, const uint8_t* dev_tags, int64_t nrows,
                                  const char* dict_blob, const int64_t* dict_offsets, int64_t ndict) {
    return guard([&] {
        REQUIRE(t); REQUIRE(dev_payload || nrows == 0);
        t->t.set_column_device(col, width, dev_payload, dev_tags, nrows, dict_blob, (const i64*)dict_offsets, ndict);
    });
}
int n1gpu_table_seal(n1gpu_table* t) {
    return guard([&] { REQUIRE(t); t->t.seal(); });
}
int64_t n1gpu_table_num_rows(const n1gpu_table* t) { return t ? t->t.nrows : -1; }
int n1gpu_table_num_columns(const n1gpu_table* t) { return t ? (int)t->t.cols.size() : -1; }
int n1gpu_table_column_scan_bytes(const n1gpu_table* t, int col) {
    if (!t || col < 0 || col >= (int)t->t.cols.size() || !t->t.sealed) return -1;
    return t->t.scan_bytes(col);
}
int n1gpu_table_dict_export(n1gpu_table* t, int col, char* blob, int64_t blob_cap, int64_t* offsets, int64_t offsets_cap,
                            int64_t* ndict, int64_t* blob_bytes) {
    return guard([&] {
        REQUIRE(t); REQUIRE(ndict); REQUIRE(blob_bytes);
        const auto& d = t->t.exchange_column(col).dict;
        i64 bytes = 0;
        for (auto& s : d) bytes += (i64)s.size();
        *ndict = (int64_t)d.size();
        *blob_bytes = bytes;
        if (!blob || !offsets) return;
        if (blob_cap < bytes || offsets_cap < (i64)d.size() + 1) N1_THROW(N1GPU_E_INVALID, "dictionary export buffers too small");
        i64 at = 0;
        for (size_t i = 0; i < d.size(); ++i) { offsets[i] = at; memcpy(blob + at, d[i].data(), d[i].size()); at += (i64)d[i].size(); }
        offsets[d.size()] = at;
    });
}
int n1gpu_table_dict_import(n1gpu_table* t, int col, const char* blob, const int64_t* offsets, int64_t ndict) {
    return guard([&] { REQUIRE(t); REQUIRE(offsets); t->t.import_dictionary(col, blob, (const i64*)offsets, ndict); });
}
int n1gpu_table_dict_merge(n1gpu_table* t, int col, int nparts, const char* const* blobs, const int64_t* const* offsets, const int64_t* ndicts) {
    return guard([&] {
        REQUIRE(t); REQUIRE(blobs); REQUIRE(offsets); REQUIRE(ndicts);
        if (nparts < 1) N1_THROW(N1GPU_E_INVALID, "no dictionaries to merge");
        t->t.merge_dictionaries(col, nparts, blobs, (const i64* const*)offsets, (const i64*)ndicts);
    });
}
int n1gpu_table_stats_get(n1gpu_table* t, int col, int64_t stats[8]) {
    return guard([&] {
        REQUIRE(t); REQUIRE(stats);
        if (col < 0 || col >= (int)t->t.cols.size()) N1_THROW(N1GPU_E_INVALID, "no such column");
        Column& c = t->t.cols[col];
        ColumnStats st = c.stats;
        if (!t->t.sealed && !c.stats_forced && !t->t.rows_in_hbm()) {  // compute from staging
            st = host_stats(c.tags, c.payload);
            st.set_dictionary(c.dict);
        }
        stats[0] = st.class_mask; stats[1] = st.has_int; stats[2] = st.int_min; stats[3] = st.int_max;
        stats[4] = st.has_float; stats[5] = st.ndict; stats[6] = st.empty_rank; stats[7] = st.absent_rows;
    });
}
int n1gpu_table_stats_set(n1gpu_table* t, int col, const int64_t stats[8]) {
    return guard([&] {
        REQUIRE(t); REQUIRE(stats);
        if (col < 0 || col >= (int)t->t.cols.size()) N1_THROW(N1GPU_E_INVALID, "no such column");
        if (t->t.sealed) N1_THROW(N1GPU_E_INVALID, "statistics exchange happens before seal");
        Column& c = t->t.cols[col];
        c.stats.set_dictionary(c.dict);  // empty_rank: the exchanged word 6 is ignored
        c.stats.class_mask = (u32)stats[0]; c.stats.has_int = stats[1] != 0; c.stats.int_min = stats[2]; c.stats.int_max = stats[3];
        c.stats.has_float = stats[4] != 0; c.stats.ndict = stats[5]; c.stats.absent_rows = stats[7];
        c.stats_forced = true;
    });
}
int n1gpu_table_load_ndjson(n1gpu_table* t, const char* path, int threads) {
    return guard([&] { REQUIRE(t); REQUIRE(path); t->t.load_ndjson(path, threads); });
}
int n1gpu_table_set_segment_output(n1gpu_table* t, const char* path, const char* source_tag) {
    return guard([&] {
        REQUIRE(t);
        if (t->t.sealed) N1_THROW(N1GPU_E_INVALID, "the segment is written by seal");
        t->t.segment_out = path ? path : "";
        t->t.segment_source = source_tag ? source_tag : "";
    });
}
int n1gpu_table_load_segment(n1gpu_table* t, const char* path, const char* source_tag, int* loaded) {
    return guard([&] {
        REQUIRE(t); REQUIRE(path); REQUIRE(loaded);
        *loaded = t->t.load_segment(path, source_tag ? source_tag : "") ? 1 : 0;
    });
}
int n1gpu_set_segment_dir(const char* dir) {
    return guard([&] { execution::set_segment_dir(dir ? dir : ""); });
}
int n1gpu_table_set_global_rows(n1gpu_table* t, int64_t rows) {
    return guard([&] {
        REQUIRE(t);
        if (rows < 0) N1_THROW(N1GPU_E_INVALID, "negative row count");
        t->t.global_rows = rows;
    });
}
int n1gpu_table_column_peek(n1gpu_table* t, int col, int64_t* payload, uint8_t* tags, int64_t nrows) {
    return guard([&] {
        REQUIRE(t);
        if (col < 0 || col >= (int)t->t.cols.size()) N1_THROW(N1GPU_E_INVALID, "no such column");
        if (t->t.sealed) N1_THROW(N1GPU_E_INVALID, "staged rows are released at seal");
        t->t.build_dictionary(col);
        Column& c = t->t.cols[col];
        if (nrows != (i64)c.tags.size()) N1_THROW(N1GPU_E_INVALID, "column has %lld rows", (long long)c.tags.size());
        if (payload) memcpy(payload, c.payload.data(), (size_t)nrows * 8);
        if (tags) memcpy(tags, c.tags.data(), (size_t)nrows);
    });
}
int n1gpu_table_free(n1gpu_table* t) { delete t; return N1GPU_OK; }

// ---- query ------------------------------------------------------------------------------------------------
int n1gpu_query_compile(n1gpu_table* t, const char* alias, const char* where, const char* const* group_keys, int nkeys,
                        const char* const* aggregates, int naggs, n1gpu_query** out) {
    return guard([&] {
        REQUIRE(t); REQUIRE(alias); REQUIRE(out);
        if (nkeys < 0 || naggs < 0) N1_THROW(N1GPU_E_INVALID, "negative count");
        std::vector<std::string> keys, aggs;
        for (int i = 0; i < nkeys; ++i) { REQUIRE(group_keys && group_keys[i]); keys.push_back(group_keys[i]); }
        for (int i = 0; i < naggs; ++i) { REQUIRE(aggregates && aggregates[i]); aggs.push_back(aggregates[i]); }
        auto q = Query::compile(&t->t, alias, where, keys, aggs);
        *out = new n1gpu_query{std::move(q)};
    });
}
int n1gpu_query_compile_params(n1gpu_table* t, const char* alias, const char* where, const char* const* group_keys, int nkeys,
                               const char* const* aggregates, int naggs, const char* const* param_names, const char* const* param_values,
                               int nparams, n1gpu_query** out) {
    return guard([&] {
        REQUIRE(t); REQUIRE(alias); REQUIRE(out);
        if (nkeys < 0 || naggs < 0 || nparams < 0) N1_THROW(N1GPU_E_INVALID, "negative count");
        std::vector<std::string> keys, aggs;
        for (int i = 0; i < nkeys; ++i) { REQUIRE(group_keys && group_keys[i]); keys.push_back(group_keys[i]); }
        for (int i = 0; i < naggs; ++i) { REQUIRE(aggregates && aggregates[i]); aggs.push_back(aggregates[i]); }
        std::vector<ParamValue> params;
        for (int i = 0; i < nparams; ++i) {
            REQUIRE(param_names && param_names[i] && param_values && param_values[i]);
            const char* n = param_names[i];
            ParamValue pv = parse_param_value(param_values[i]);
            pv.name = n[0] == '$' ? n + 1 : n;
            params.push_back(std::move(pv));
        }
        auto q = Query::compile(&t->t, alias, where, keys, aggs, params);
        *out = new n1gpu_query{std::move(q)};
    });
}
int n1gpu_jit_stats(uint64_t* compiled, uint64_t* reused) {
    if (!compiled || !reused) return N1GPU_E_INVALID;
    unsigned long long c = 0, r = 0;
    jit_stats(&c, &r);
    *compiled = c; *reused = r;
    return N1GPU_OK;
}
int n1gpu_query_execute(n1gpu_query* q, n1gpu_result** out) {
    return guard([&] {
        REQUIRE(q); REQUIRE(out);
        q->q->scan_blocking();
        *out = new n1gpu_result{q->q->finalize()};
    });
}
int n1gpu_query_launch(n1gpu_query* q) {
    return guard([&] { REQUIRE(q); q->q->launch_scan(); });
}
int n1gpu_query_collect(n1gpu_query* q, n1gpu_result** out) {
    return guard([&] {
        REQUIRE(q); REQUIRE(out);
        if (!q->q->wait_scan()) q->q->scan_blocking();  // a table was grown: rerun
        *out = new n1gpu_result{q->q->finalize()};
    });
}
int n1gpu_query_cancel(n1gpu_query* q) {
    if (!q) return N1GPU_E_INVALID;
    q->q->cancel();
    return N1GPU_OK;
}
const char* n1gpu_query_kernel_source(const n1gpu_query* q) { return q ? q->q->kp.source.c_str() : ""; }
const char* n1gpu_query_part_source(const n1gpu_query* q) { return q ? q->q->kp.part_source.c_str() : ""; }
int n1gpu_query_info(const n1gpu_query* q, int64_t info[8]) {
    return guard([&] {
        REQUIRE(q); REQUIRE(info);
        const Query& Q = *q->q;
        info[0] = Q.kp.dense_global ? 4 : Q.kp.mode; info[1] = Q.ops.n; info[2] = Q.kernel ? Q.kernel->regs : 0; info[3] = Q.grid; info[4] = Q.kp.block;
        info[5] = Q.kp.scan_bytes_per_row; info[6] = Q.kernel ? Q.kernel->static_smem : 0;
        info[7] = Q.kp.mode == MODE_DENSE ? Q.kp.dense_slots : (i64)Q.cap;
    });
}
int64_t n1gpu_query_last_scan_ns(const n1gpu_query* q) { return q ? (int64_t)(q->q->last_scan_ms * 1e6) : -1; }
int n1gpu_query_rebind(n1gpu_query* q, n1gpu_table* t) {
    return guard([&] { REQUIRE(q); REQUIRE(t); q->q->rebind(&t->t); });
}
int n1gpu_query_set_stream(n1gpu_query* q, void* cuda_stream) {
    return guard([&] {
        REQUIRE(q);
        if (q->q->launched) N1_THROW(N1GPU_E_INVALID, "a scan is outstanding");
        // NULL is a real stream (the legacy default stream, which is what torch.cuda.current_stream() is
        // unless the caller changed it); (void*)-1 restores the query's own non-blocking stream
        q->q->stream = (cuda_stream == (void*)-1) ? q->q->own_stream : (cudaStream_t)cuda_stream;
    });
}
int n1gpu_query_set_timing(n1gpu_query* q, int enable) {
    if (!q) return N1GPU_E_INVALID;
    q->q->timing = enable != 0;
    return N1GPU_OK;
}
int n1gpu_query_free(n1gpu_query* q) { delete q; return N1GPU_OK; }

// ---- peer mailbox (fused small-state all-gather over NVLink) ----------------------------------------------------
struct n1gpu_mailbox { Mailbox m; };
int n1gpu_mailbox_create(int nranks, int rank, int64_t max_words, n1gpu_mailbox** out) {
    return n1gpu_mailbox_create_arena(nranks, rank, max_words, 0, out);
}
int n1gpu_mailbox_create_arena(int nranks, int rank, int64_t max_words, int64_t arena_bytes, n1gpu_mailbox** out) {
    return guard([&] {
        REQUIRE(out);
        if (nranks < 1 || nranks > 16 || rank < 0 || rank >= nranks || max_words < 1 || arena_bytes < 0) N1_THROW(N1GPU_E_INVALID, "bad mailbox geometry");
        if (!have_device()) N1_THROW(N1GPU_E_CUDA, "no CUDA device");
        std::unique_ptr<n1gpu_mailbox> mb(new n1gpu_mailbox());
        Mailbox& m = mb->m;
        m.nranks = nranks; m.rank = rank; m.stride = (u64)max_words + 1;
        m.flags_off = ((size_t)m.slots * nranks * m.stride * 8 + 255) & ~(size_t)255;
        m.arena_off = (m.flags_off + (size_t)2 * 64 * nranks * 8 + 255) & ~(size_t)255;  // rows 0-63: table complete, 64-127: records consumed
        m.arena_bytes = (size_t)arena_bytes;
        m.bytes = m.arena_off + m.arena_bytes;
        CK(cudaMalloc(&m.base, m.bytes));
        CK(cudaMemset(m.base, 0, m.bytes));
        CK(cudaDeviceSynchronize());
        m.peers.assign((size_t)nranks, nullptr);
        m.peers[(size_t)rank] = m.base;
        *out = mb.release();
    });
}
int n1gpu_mailbox_ipc_handle(n1gpu_mailbox* mb, uint8_t handle[64]) {
    return guard([&] {
        REQUIRE(mb); REQUIRE(handle);
        static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
        cudaIpcMemHandle_t h;
        CK(cudaIpcGetMemHandle(&h, mb->m.base));
        memcpy(handle, &h, 64);
    });
}
int n1gpu_mailbox_open_peers(n1gpu_mailbox* mb, const uint8_t* handles) {
    return guard([&] {
        REQUIRE(mb); REQUIRE(handles);
        Mailbox& m = mb->m;
        for (int r = 0; r < m.nranks; ++r) {
            if (r == m.rank) continue;
            cudaIpcMemHandle_t h;
            memcpy(&h, handles + (size_t)r * 64, 64);
            void* p = nullptr;
            CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
            m.peers[(size_t)r] = p;
        }
        m.d_peers.alloc((size_t)m.nranks * 8);
        CK(cudaMemcpy(m.d_peers.p, m.peers.data(), (size_t)m.nranks * 8, cudaMemcpyHostToDevice));
    });
}
int n1gpu_mailbox_set_peer(n1gpu_mailbox* mb, int rank, void* dev_base) {
    return guard([&] {
        REQUIRE(mb);
        Mailbox& m = mb->m;
        if (rank < 0 || rank >= m.nranks || !dev_base) N1_THROW(N1GPU_E_INVALID, "bad peer");
        if (rank != m.rank) m.peers[(size_t)rank] = dev_base;
        bool all = true;
        for (void* p : m.peers) all = all && p;
        if (all) {
            m.d_peers.alloc((size_t)m.nranks * 8);
            CK(cudaMemcpy(m.d_peers.p, m.peers.data(), (size_t)m.nranks * 8, cudaMemcpyHostToDevice));
        }
    });
}
void* n1gpu_mailbox_base(n1gpu_mailbox* mb) { return mb ? mb->m.base : nullptr; }
int n1gpu_mailbox_free(n1gpu_mailbox* mb) { delete mb; return N1GPU_OK; }
int n1gpu_query_set_mailbox(n1gpu_query* q, n1gpu_mailbox* mb) {
    return guard([&] {
        REQUIRE(q);
        if (q->q->launched) N1_THROW(N1GPU_E_INVALID, "a scan is outstanding");
        if (mb && mb->m.nranks > 1 && !mb->m.d_peers.p) N1_THROW(N1GPU_E_INVALID, "mailbox peers are not opened");
        q->q->attach_mailbox(mb ? &mb->m : nullptr);
    });
}

int n1gpu_query_peer_mode(const n1gpu_query* q) {
    if (!q) return N1GPU_E_INVALID;
    const Query& Q = *q->q;
    if (!Q.mailbox || Q.mailbox->nranks < 2) return 0;
    if (Q.peer_part && Q.use_part()) return 2;
    if (Q.peer_table) return 1;
    return 0;
}

// ---- multi-GPU partial state ----------------------------------------------------------------------------------
int n1gpu_query_scan_partial(n1gpu_query* q) {
    return guard([&] {
        REQUIRE(q);
        // the record / DISTINCT-entry exchange that follows reads the general scan's tables and sets: the partitioned
        // DISTINCT aggregation (which leaves finished words instead) is for handles whose groups are finalised in place
        q->q->part_disabled = true;
        q->q->scan_blocking();
    });
}
int n1gpu_query_partial_counts(n1gpu_query* q, int64_t* ngroups, int64_t* ndistinct, int* record_words) {
    return guard([&] {
        REQUIRE(q); REQUIRE(ngroups); REQUIRE(ndistinct); REQUIRE(record_words);
        i64 g = 0, d = 0;
        q->q->partial_counts(&g, &d);
        *ngroups = g; *ndistinct = d; *record_words = 2 + q->q->ops.n;
    });
}
int n1gpu_query_partial_export(n1gpu_query* q, int nranks, void* dev_records, int64_t cap_records, int64_t* counts,
                               void* dev_distinct, int64_t cap_distinct, int64_t* dcounts) {
    return guard([&] {
        REQUIRE(q); REQUIRE(counts); REQUIRE(dcounts);
        if (nranks < 1) N1_THROW(N1GPU_E_INVALID, "nranks must be >= 1");
        q->q->partial_export(nranks, dev_records, cap_records, (i64*)counts, dev_distinct, cap_distinct, (i64*)dcounts);
    });
}
int n1gpu_query_partial_reset(n1gpu_query* q) {
    return guard([&] { REQUIRE(q); q->q->partial_reset(); });
}
int n1gpu_query_partial_import(n1gpu_query* q, const void* dev_records, int64_t n, const void* dev_distinct, int64_t nd) {
    return guard([&] { REQUIRE(q); q->q->partial_import(dev_records, n, dev_distinct, nd); });
}
int n1gpu_query_state_words(n1gpu_query* q, void** dev_words, int64_t* nwords) {
    return guard([&] {
        REQUIRE(q); REQUIRE(dev_words); REQUIRE(nwords);
        Query& Q = *q->q;
        if (!Q.kernel) N1_THROW(N1GPU_E_CUDA, "no CUDA device");
        if (!(Q.kp.mode == MODE_UNGROUPED || Q.kp.mode == MODE_DENSE) || Q.kp.ndistinct)
            N1_THROW(N1GPU_E_INVALID, "state_words is for ungrouped / dense chains without DISTINCT; use partial_export");
        *dev_words = Q.acc();
        *nwords = (int64_t)(Q.cap * (u64)Q.ops.n);
    });
}
int n1gpu_query_merge_words(n1gpu_query* q, const void* dev_all_words, int nranks) {
    return guard([&] {
        REQUIRE(q); REQUIRE(dev_all_words);
        Query& Q = *q->q;
        if (!Q.kernel) N1_THROW(N1GPU_E_CUDA, "no CUDA device");
        if (!(Q.kp.mode == MODE_UNGROUPED || Q.kp.mode == MODE_DENSE) || Q.kp.ndistinct) N1_THROW(N1GPU_E_INVALID, "not a small-state chain");
        if (nranks < 1) N1_THROW(N1GPU_E_INVALID, "nranks must be >= 1");
        launch_merge_words((const u64*)dev_all_words, nranks, Q.cap, Q.ops, Q.acc(), Q.h_records.as<u64>(), Q.stream);
    });
}
int n1gpu_query_word_ops(const n1gpu_query* q, int* ops, int cap) {
    if (!q) return -1;
    const Query& Q = *q->q;
    for (int w = 0; ops && w < Q.ops.n && w < cap; ++w) ops[w] = Q.ops.op[w];
    return Q.ops.n;
}
int n1gpu_query_finalize(n1gpu_query* q, n1gpu_result** out) {
    return guard([&] { REQUIRE(q); REQUIRE(out); *out = new n1gpu_result{q->q->finalize()}; });
}

// ---- result ------------------------------------------------------------------------------------------------------
int64_t n1gpu_result_num_groups(const n1gpu_result* r) { return r ? r->r->ngroups : -1; }
int n1gpu_result_num_keys(const n1gpu_result* r) { return r ? r->r->nkeys : -1; }
int n1gpu_result_num_aggregates(const n1gpu_result* r) { return r ? r->r->naggs : -1; }
int n1gpu_result_fetch(const n1gpu_result* r, uint8_t* key_cls, int64_t* key_val, uint8_t* agg_cls, int64_t* agg_val) {
    return guard([&] {
        REQUIRE(r);
        const Result& R = *r->r;
        if (key_cls && !R.key_cls.empty()) memcpy(key_cls, R.key_cls.data(), R.key_cls.size());
        if (key_val && !R.key_val.empty()) memcpy(key_val, R.key_val.data(), R.key_val.size() * 8);
        if (agg_cls && !R.agg_cls.empty()) memcpy(agg_cls, R.agg_cls.data(), R.agg_cls.size());
        if (agg_val && !R.agg_val.empty()) memcpy(agg_val, R.agg_val.data(), R.agg_val.size() * 8);
    });
}
int n1gpu_result_string(const n1gpu_result* r, int64_t index, const char** ptr, int64_t* len) {
    return guard([&] {
        REQUIRE(r); REQUIRE(ptr); REQUIRE(len);
        if (!r->r->string_ok(index)) N1_THROW(N1GPU_E_INVALID, "string index out of range");
        const std::string& str = r->r->string_at(index);
        *ptr = str.data();
        *len = (int64_t)str.size();
    });
}
int n1gpu_result_stats(const n1gpu_result* r, int64_t stats[8]) {
    return guard([&] { REQUIRE(r); REQUIRE(stats); for (int i = 0; i < 8; ++i) stats[i] = r->r->stats[i]; });
}
int n1gpu_result_free(n1gpu_result* r) { delete r; return N1GPU_OK; }

static int copy_out(const std::string& s, char* buf, int64_t cap, int64_t* len) {
    if (len) *len = (int64_t)s.size();
    if (buf && cap > 0) {
        size_t n = std::min<size_t>(s.size(), (size_t)cap - 1);
        memcpy(buf, s.data(), n);
        buf[n] = '\0';
    }
    return N1GPU_OK;
}
// ---- plan level -----------------------------------------------------------------------------------------------------
int n1gpu_plan_build(const char* plan_json, const char* datastore_root, n1gpu_operator** out, int* rest_index) {
    return guard([&] {
        REQUIRE(plan_json); REQUIRE(datastore_root); REQUIRE(out);
        int rest = 0;
        auto op = execution::Build(plan_json, datastore_root, &rest);
        if (rest_index) *rest_index = rest;
        *out = new n1gpu_operator{std::move(op)};
    });
}
int n1gpu_plan_build_tail(const char* plan_json, const char* datastore_root, n1gpu_operator** out, int* rest_index, int* outer_rest_index) {
    return guard([&] {
        REQUIRE(plan_json); REQUIRE(datastore_root); REQUIRE(out);
        int rest = 0, outer = 0;
        auto op = execution::BuildWithTail(plan_json, datastore_root, true, &rest, &outer);
        if (rest_index) *rest_index = rest;
        if (outer_rest_index) *outer_rest_index = outer;
        *out = new n1gpu_operator{std::move(op)};
    });
}
int n1gpu_operator_tail_operators(const n1gpu_operator* op, char* buf, int64_t cap, int64_t* len) {
    std::string s;
    int rc = guard([&] {
        REQUIRE(op);
        for (auto& n : op->op->tail.operators) { if (!s.empty()) s += ","; s += n; }
    });
    return rc == N1GPU_OK ? copy_out(s, buf, cap, len) : rc;
}
int n1gpu_operator_run_tail(n1gpu_operator* op, const n1gpu_result* r, char* buf, int64_t cap, int64_t* len, int64_t* rows) {
    std::string s;
    int rc = guard([&] {
        REQUIRE(op); REQUIRE(r);
        if (op->op->tail.empty()) N1_THROW(N1GPU_E_INVALID, "the operator was built without a tail (n1gpu_plan_build_tail, eligible plan)");
        if (op->tail_of != (const void*)r->r.get()) {
            i64 n = 0;
            op->tail_rows = op->op->tail.Run(*r->r, &n);
            op->tail_count = n;
            op->tail_of = (const void*)r->r.get();
        }
        if (rows) *rows = op->tail_count;
    });
    if (rc != N1GPU_OK) return rc;
    rc = copy_out(op->tail_rows, buf, cap, len);
    if (buf && cap > (int64_t)op->tail_rows.size()) { op->tail_of = nullptr; std::string().swap(op->tail_rows); }  // delivered in full
    return rc;
}
int n1gpu_operator_import_result(const n1gpu_operator* op, int64_t ngroups, const uint8_t* key_cls, const int64_t* key_val,
                                 const uint8_t* agg_cls, const int64_t* agg_val, const char* blob, const int64_t* offsets,
                                 int64_t nstrings, n1gpu_result** out) {
    return guard([&] {
        REQUIRE(op); REQUIRE(out);
        if (ngroups < 0 || nstrings < 0) N1_THROW(N1GPU_E_INVALID, "negative count");
        const Query& Q = *op->op->query;
        std::unique_ptr<Result> r(new Result());
        r->nkeys = (int)Q.keys.size();
        r->naggs = (int)Q.aggs.size();
        r->ngroups = ngroups;
        r->agg_texts = Q.agg_texts;
        r->key_texts = Q.key_texts;
        r->alias = Q.alias;
        for (auto& k : Q.keys) {
            std::vector<std::string> path;
            if (k->kind == EK::FIELD && k->col >= 0) path = Q.table->cols[k->col].path;
            r->key_paths.push_back(path);
        }
        const size_t nk = (size_t)ngroups * r->nkeys, na = (size_t)ngroups * r->naggs;
        if ((nk && (!key_cls || !key_val)) || (na && (!agg_cls || !agg_val))) N1_THROW(N1GPU_E_INVALID, "missing value arrays");
        r->key_cls.assign(key_cls, key_cls + nk); r->key_val.assign(key_val, key_val + nk);
        r->agg_cls.assign(agg_cls, agg_cls + na); r->agg_val.assign(agg_val, agg_val + na);
        for (int64_t i = 0; i < nstrings; ++i) r->strings.emplace_back(blob + offsets[i], (size_t)(offsets[i + 1] - offsets[i]));
        auto check = [&](const FlatArr<u8>& cls, const FlatArr<i64>& val) {
            for (size_t i = 0; i < cls.size(); ++i) {
                if (cls[i] > C_STRING) N1_THROW(N1GPU_E_INVALID, "value class %d is not a scalar class", (int)cls[i]);
                if (cls[i] == C_STRING && (val[i] < 0 || val[i] >= nstrings)) N1_THROW(N1GPU_E_INVALID, "string index out of range");
            }
        };
        check(r->key_cls, r->key_val);
        check(r->agg_cls, r->agg_val);
        r->stats[1] = ngroups;
        *out = new n1gpu_result{std::move(r)};
    });
}
int n1gpu_operator_num_keys(const n1gpu_operator* op) { return op && op->op->query ? (int)op->op->query->keys.size() : N1GPU_E_INVALID; }
int n1gpu_operator_num_aggregates(const n1gpu_operator* op) { return op && op->op->query ? (int)op->op->query->aggs.size() : N1GPU_E_INVALID; }
int n1gpu_operator_run_once(n1gpu_operator* op, n1gpu_result** out) {
    return guard([&] { REQUIRE(op); REQUIRE(out); *out = new n1gpu_result{op->op->RunOnce()}; });
}
int n1gpu_operator_send_stop(n1gpu_operator* op) {
    if (!op) return N1GPU_E_INVALID;
    op->op->SendStop();
    return N1GPU_OK;
}
int n1gpu_operator_marshal_json(n1gpu_operator* op, char* buf, int64_t cap, int64_t* len) {
    std::string s;
    int rc = guard([&] { REQUIRE(op); s = op->op->MarshalJSON(); });
    return rc == N1GPU_OK ? copy_out(s, buf, cap, len) : rc;
}
int n1gpu_result_to_json(const n1gpu_result* r, char* buf, int64_t cap, int64_t* len) {
    std::string s;
    int rc = guard([&] { REQUIRE(r); s = execution::ResultToJSON(*r->r); });
    return rc == N1GPU_OK ? copy_out(s, buf, cap, len) : rc;
}
int n1gpu_operator_free(n1gpu_operator* op) { delete op; return N1GPU_OK; }

}  // extern "C"
