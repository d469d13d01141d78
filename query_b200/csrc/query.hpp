// query.hpp — a compiled Filter + InitialGroup/IntermediateGroup/FinalGroup chain bound to a table.
#pragma once
#include <atomic>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "codegen.hpp"
#include "jit.hpp"
#include "kernels.hpp"

namespace n1 {

// A flat result array: owns its storage, or views a region of the result's pinned buffer (the device finalisation lands
// there with one copy per array and nothing is copied again until n1gpu_result_fetch).
template <class T> struct FlatArr {
    std::vector<T> own;
    T* p = nullptr;
    size_t n = 0;
    void resize(size_t k) { own.resize(k); p = own.data(); n = k; }
    template <class U> void assign(const U* a, const U* b) { own.assign(a, b); p = own.data(); n = own.size(); }
    void view(T* ptr, size_t k) { std::vector<T>().swap(own); p = ptr; n = k; }
    T* data() { return p; }
    const T* data() const { return p; }
    size_t size() const { return n; }
    bool empty() const { return n == 0; }
    T& operator[](size_t i) { return p[i]; }
    const T& operator[](size_t i) const { return p[i]; }
};

struct Result {
    int nkeys = 0, naggs = 0;
    i64 ngroups = 0;
    // [ngroups][nkeys] / [ngroups][naggs] as class byte + 64-bit payload (int / float bits / index into `strings`):
    // flat arrays, so that a million-group result costs two allocations, not four million string-carrying objects
    FlatArr<u8> key_cls, agg_cls;
    FlatArr<i64> key_val, agg_val;
    PinnedBuf pinned;  // backing store of the arrays when the groups were finalised on the device
    std::vector<std::string> strings;
    // Strings of groups finalised here are REFERENCES (dictionary column << 40 | rank) into the table's dictionaries, which
    // the result keeps alive; nothing is copied until a string is asked for.  Imported results own `strings` instead.
    bool string_refs = false;
    std::vector<std::shared_ptr<const std::vector<std::string>>> dicts;  // [column]
    const std::string& string_at(i64 val) const {
        static const std::string empty;
        if (!string_refs) return strings[(size_t)val];
        const size_t col = (size_t)((u64)val >> 40), rank = (size_t)((u64)val & 0xffffffffffULL);
        if (col >= dicts.size() || !dicts[col] || rank >= dicts[col]->size()) return empty;
        return (*dicts[col])[rank];
    }
    bool string_ok(i64 val) const { return string_refs ? val >= 0 : (val >= 0 && (size_t)val < strings.size()); }
    HValue value(u8 cls, i64 val) const {
        HValue v;
        v.cls = cls;
        if (cls == C_STRING) v.s = string_at(val); else v.bits = val;
        return v;
    }
    HValue key(i64 g, int k) const { const size_t i = (size_t)g * nkeys + k; return value(key_cls[i], key_val[i]); }
    HValue agg(i64 g, int a) const { const size_t i = (size_t)g * naggs + a; return value(agg_cls[i], agg_val[i]); }
    std::vector<std::string> agg_texts, key_texts;
    std::vector<std::vector<std::string>> key_paths;  // field path of each key (empty: computed key)
    std::string alias;
    i64 stats[8] = {0, 0, 0, 0, 0, 0, 0, 0};
};

// Peer mailbox for the fused small-state all-gather: every rank owns slots x nranks cells of (stride) words in
// HBM, exported to the other ranks' processes through CUDA IPC; scan kernels store into the peers' cells over
// NVLink, k_merge_mailbox folds the own mailbox.
//
// The same IPC-mapped buffer can carry an ARENA behind the mailbox cells: direct-indexed HBM group tables are placed
// there (double-buffered), so that every rank can read every other rank's partial table with plain loads over NVLink.
// The owner-sharded merge + finalisation (k_finalize_groups over PeerTables) then replaces the collective: a rank raises
// a flag in every peer's flag row when its scan is complete (k_peer_signal), and rank r's finalisation kernel waits for
// all flags of the step before it folds slot range r of all tables.  Layout: [cells | flags 64 x nranks | arena].
struct Mailbox {
    int nranks = 1, rank = 0, slots = 64;
    u64 stride = 0;              // words per cell = max_words + 1 (sequence flag)
    void* base = nullptr;        // own buffer (plain cudaMalloc: IPC-exported, never pooled)
    size_t bytes = 0;
    size_t flags_off = 0;        // byte offset of the step flags (64 slots x nranks u64)
    size_t arena_off = 0, arena_bytes = 0, arena_used = 0;
    // bump allocation with exact-size recycling; every rank must set / free its peer-table queries in the same order
    // (same sizes -> same offsets on every rank)
    std::map<size_t, std::vector<size_t>> arena_bins;
    void arena_free(size_t at, size_t n) { arena_bins[(n + 255) & ~(size_t)255].push_back(at); }
    size_t arena_alloc(size_t n) {
        n = (n + 255) & ~(size_t)255;
        auto it = arena_bins.find(n);
        if (it != arena_bins.end() && !it->second.empty()) { const size_t at = it->second.back(); it->second.pop_back(); return at; }
        if (arena_used + n > arena_bytes) N1_THROW(N1GPU_E_NOMEM, "peer arena of %zu bytes is exhausted (%zu used, %zu wanted)", arena_bytes, arena_used, n);
        const size_t at = arena_off + arena_used;
        arena_used += n;
        return at;
    }
    std::vector<void*> peers;    // [nranks], own entry = base
    DevBuf d_peers;              // the same pointers in device memory
    u64 seq = 0;
    ~Mailbox();
};

struct Query {
    Table* table = nullptr;
    Mailbox* mailbox = nullptr;
    std::string alias, where_text;
    std::vector<std::string> key_texts, agg_texts;
    ExprP where;
    std::vector<ExprP> keys, aggs;
    KernelPlan kp;
    std::shared_ptr<JitKernel> kernel;
    std::shared_ptr<JitKernel> part_kernel;  // KernelPlan::part: the partitioning kernel (null: not this shape)
    bool part_disabled = false;              // a partition overflowed its share (skewed keys): this handle scans the general way
    bool part_done = false;                  // the last scan left finished DISTINCT words in the table (no k_distinct_finalize)
    u64 part_cap = 0;                        // records a partition holds
    DevBuf d_part_recs, d_part_cur;
    bool use_part() const { return part_kernel && !part_disabled; }
    // multi-GPU: the partitioned records live in the mailbox arena; rank r aggregates partition range r reading every
    // rank's records of those partitions over NVLink, and finalises the groups of that range
    bool peer_part = false;
    size_t peer_recs_off = 0, peer_cur_off = 0, peer_recs_bytes = 0, peer_cur_bytes = 0;
    u64 part_seq = 0;   // step whose records this rank last published (its consumption is awaited before they are overwritten)
    bool peer_part_merge() const { return peer_part && mailbox && mailbox->nranks > 1 && use_part(); }
    void part_range(int* p0, int* p1) const {
        const int np = 1 << kp.part_bits;
        if (!peer_part_merge()) { *p0 = 0; *p1 = np; return; }
        *p0 = (int)((i64)np * mailbox->rank / mailbox->nranks);
        *p1 = (int)((i64)np * (mailbox->rank + 1) / mailbox->nranks);
    }
    DistinctDescs distinct_descs() const;
    DevBuf d_in_sets;                  // every IN set of the chain (KernelPlan::in_sets), copied once at compile time
    std::vector<NqInSet> in_descs;     // NqParams::inset
    void upload_in_sets();
    OpsArr ops{};

    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    int grid = 0;
    u64 cap = 1;      // group slots (1 / dense slots / hash capacity)
    u64 set_cap = 0;  // DISTINCT entry set capacity: hash slots, or bits when the set is a bitmap
    size_t set_bytes() const { return kp.set_bitmap ? (size_t)(set_cap >> 3) : (size_t)set_cap * (kp.set128 ? 16 : 8); }
    int set_kw() const { return kp.set_bitmap ? 4 : (kp.set128 ? 2 : 1); }  // how kernels.cu enumerates the set
    DevBuf d_partials, d_acc, d_accum, d_keys, d_set, d_status, d_counts, d_records, d_drecords, d_ticket, d_final;
    PinnedBuf h_status, h_counts, h_records, h_drecords;
    std::atomic<bool> cancelled{false};
    // The word a running kernel polls lives in HBM (polling host memory over PCIe cost 40x the scan); cancel() sets it with
    // an asynchronous copy on a stream of its own, which the copy engine executes while the scan runs.
    DevBuf d_cancel;
    PinnedBuf h_cancel;          // the value 1, in pinned memory (source of that copy)
    cudaStream_t cancel_stream = nullptr;
    int device = 0;
    void cancel();
    bool launched = false;
    bool timing = true;        // record CUDA events around the scan (each record costs GPU front-end time)
    bool timed_launch = false;
    bool ungrouped_live = true;
    bool host_acc_valid = false;  // h_records holds the table words of the last scan (small-state modes)
    bool import_dirty() const { return !host_acc_valid; }
    // direct-indexed table kept in the mailbox arena (peer-readable), double-buffered by step parity
    bool peer_table = false;
    size_t peer_off[2] = {0, 0}, peer_bytes = 0;
    u64 peer_seq = 0;            // step whose table the next finalisation folds (0: none outstanding)
    u64 peer_steps = 0;          // steps THIS query launched: their parity selects the buffer (the mailbox-wide seq numbers the
                                 // flags; with several queries in flight on one mailbox its parity would not alternate per query,
                                 // and a step could overwrite the table a slower peer is still folding)
    u64* acc() const {           // the group table of the current step
        if (peer_table) return (u64*)((char*)mailbox->base + peer_off[peer_steps & 1]);
        return d_acc.as<u64>();
    }
    bool peer_merge() const { return peer_table && mailbox && mailbox->nranks > 1; }
    void attach_mailbox(Mailbox* mb);
    double last_scan_ms = 0;
    u64 launches_at_start = 0;

    ~Query();
    static std::unique_ptr<Query> compile(Table* t, const std::string& alias, const char* where,
                                          const std::vector<std::string>& keys, const std::vector<std::string>& aggs,
                                          const std::vector<ParamValue>& params = {});
    // the scan publishes the whole table to pinned host memory (and may push it through the peer mailbox)
    bool small_state() const { return kp.mode == MODE_UNGROUPED || (kp.mode == MODE_DENSE && !kp.dense_global); }
    int kw() const {
        if (kp.mode == MODE_HASHW) return KW_WIDE + kp.key_words;
        return kp.mode == MODE_UNGROUPED ? 3 : (kp.mode == MODE_DENSE ? 0 : (kp.mode == MODE_HASH64 ? 1 : 2));
    }
    bool hashed() const { return kp.mode == MODE_HASH64 || kp.mode == MODE_HASH128 || kp.mode == MODE_HASHW; }
    size_t key_bytes() const {  // the key array of a hash table
        return (size_t)cap * 8 * (kp.mode == MODE_HASHW ? 1 + kp.key_words : (kp.mode == MODE_HASH128 ? 2 : 1));
    }
    int record_words() const { return (kp.mode == MODE_HASHW ? kp.key_words : 2) + ops.n; }  // n1gpu_query_partial_counts
    void alloc_state();
    bool uses_status() const;         // hash tables / DISTINCT sets can overflow and report it
    void reset_state();               // clears tables (async on stream)
    void launch_scan();               // enqueue reset + scan (+ partial reduction)
    bool wait_scan();                 // sync; returns false when a table overflowed and was grown (caller relaunches)
    void scan_blocking();             // launch + wait, growing tables as needed
    void partial_counts(i64* ngroups, i64* ndistinct);
    void partial_export(int nranks, void* dev_records, i64 cap_records, i64* counts, void* dev_distinct, i64 cap_distinct, i64* dcounts);
    void partial_reset();
    void partial_import(const void* dev_records, i64 n, const void* dev_distinct, i64 nd);
    std::unique_ptr<Result> finalize();
    // FinalGroup on the device over slots [slot0, slot1) of `tables` (this rank's table, or every rank's, peer-mapped):
    // fills res' flat arrays; returns the number of groups
    i64 finalize_device(Result& res, const PeerTables& tables, u64 slot0, u64 slot1);
    FinalDesc final_desc() const;
    bool device_final_ok() const { return keys.size() <= 16 && aggs.size() <= 24 && kp.word_ops.size() <= 64; }
    u64 dense_key(u64 slot) const;
    void rebind(Table* t);
};

}  // namespace n1
