// query.cpp — compile / scan / merge / finalise of one Filter + Group chain.
//
// finalize() finalises the groups on the host or on the device (k_finalize_groups); both run the one restatement of
// ComputeFinal in final_group.hpp.  Reference behaviour the host side adds:
//   execution/group_final.go:108-117   no keys and no input -> one row of Default() values
#include "query.hpp"

#include <algorithm>
#include <cmath>
#include <thread>
#include <unordered_map>

namespace n1 {

namespace {

u64 pow2_at_least(u64 n) { u64 p = 1; while (p < n) p <<= 1; return p; }

}  // namespace

bool have_device() {
    static int n = -1;
    if (n < 0) { int c = 0; if (cudaGetDeviceCount(&c) != cudaSuccess) c = 0; n = c; cudaGetLastError(); }
    return n > 0;
}

Query::~Query() {
    if (launched && stream) cudaStreamSynchronize(stream);  // nothing of this query may still be running when its buffers are recycled
    if (peer_table && mailbox) { mailbox->arena_free(peer_off[1], peer_bytes); mailbox->arena_free(peer_off[0], peer_bytes); }
    if (peer_part && mailbox) { mailbox->arena_free(peer_cur_off, peer_cur_bytes); mailbox->arena_free(peer_recs_off, peer_recs_bytes); }
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    if (own_stream) cudaStreamDestroy(own_stream);
    if (cancel_stream) cudaStreamDestroy(cancel_stream);
}

void Query::cancel() {
    cancelled.store(true);
    if (!d_cancel.p) return;
    int prev = 0;  // SendStop may come from any thread: the copy must be issued on this query's device
    if (cudaGetDevice(&prev) != cudaSuccess) prev = device;
    if (prev != device) cudaSetDevice(device);
    cudaMemcpyAsync(d_cancel.p, h_cancel.p, 4, cudaMemcpyHostToDevice, cancel_stream);
    if (prev != device) cudaSetDevice(prev);
}

std::unique_ptr<Query> Query::compile(Table* t, const std::string& alias, const char* where,
                                      const std::vector<std::string>& key_texts, const std::vector<std::string>& agg_texts,
                                      const std::vector<ParamValue>& params) {
    if (!t || !t->sealed) N1_THROW(N1GPU_E_INVALID, "table must be sealed before a query is compiled");
    std::unique_ptr<Query> q(new Query());
    q->table = t;
    q->alias = alias;
    q->key_texts = key_texts;
    q->agg_texts = agg_texts;
    if (where && *where) { q->where_text = where; q->where = parse_expr(where); }
    for (auto& k : key_texts) q->keys.push_back(parse_expr(k));
    for (auto& a : agg_texts) q->aggs.push_back(parse_expr(a));
    // named / positional parameters take their values now (execution.Context.NamedArg / PositionalArg); the kernel text only
    // depends on their classes, the payloads are kernel arguments: re-binding a prepared statement reuses the cubin
    if (q->where) bind_params(*q->where, params);
    for (auto& k : q->keys) bind_params(*k, params);
    for (auto& a : q->aggs) bind_params(*a, params);
    if (q->where) bind_and_analyze(*q->where, alias, *t);
    for (auto& k : q->keys) {
        if (k->kind == EK::AGG) N1_THROW(N1GPU_E_INELIGIBLE, "aggregate as a group key");
        bind_and_analyze(*k, alias, *t);
    }
    for (auto& a : q->aggs) bind_and_analyze(*a, alias, *t);
    if (q->aggs.size() > 24) N1_THROW(N1GPU_E_INELIGIBLE, "more than 24 aggregates");
    // rows any one accumulator can see over all partitions: declared (n1gpu_table_set_global_rows), else room for 16 ranks
    const double rows_bound = t->global_rows > 0 ? (double)std::max<i64>(t->global_rows, t->nrows) : (double)std::max<i64>(t->nrows, 1) * 16.0;
    q->kp = generate_kernel(*t, q->where.get(), q->keys, q->aggs, agg_texts, rows_bound);
    q->ops.n = (int)q->kp.phys_ops.size();  // physical words: what the table holds and every merge moves
    for (int w = 0; w < q->ops.n; ++w) q->ops.op[w] = q->kp.phys_ops[w];
    if (have_device()) {
        q->kernel = jit_load(q->kp.source, q->kp.dyn_smem, q->kp.block);
        if (q->kp.part) q->part_kernel = jit_load(q->kp.part_source, q->kp.part_smem, PART_THREADS);
        CK(cudaStreamCreateWithFlags(&q->own_stream, cudaStreamNonBlocking));
        q->stream = q->own_stream;
        CK(cudaEventCreate(&q->ev0));
        CK(cudaEventCreate(&q->ev1));
        q->alloc_state();
        q->upload_in_sets();
    } else {
        // no GPU in this process (build / CPU test container): still prove the kernel compiles for sm_100a
        std::string log;
        jit_compile_cubin(q->kp.source, &log);
        if (q->kp.part) jit_compile_cubin(q->kp.part_source, &log);
    }
    return q;
}

// One device buffer holds every set of the chain: [bitmap | INT table | FLOAT table] per set, 8-byte aligned.
void Query::upload_in_sets() {
    const auto& S = kp.in_sets;
    if (S.empty()) return;
    std::vector<size_t> at;
    size_t words = 0;  // u64 words
    for (auto& s : S) { at.push_back(words); words += (s.bits.size() + 1) / 2 + s.ikeys.size() + s.fkeys.size(); }
    std::vector<u64> host(std::max<size_t>(words, 1), 0);
    for (size_t k = 0; k < S.size(); ++k) {
        u64* w = host.data() + at[k];
        memcpy(w, S[k].bits.data(), S[k].bits.size() * 4);
        w += (S[k].bits.size() + 1) / 2;
        std::copy(S[k].ikeys.begin(), S[k].ikeys.end(), w);
        std::copy(S[k].fkeys.begin(), S[k].fkeys.end(), w + S[k].ikeys.size());
    }
    d_in_sets.alloc(host.size() * 8);
    CK(cudaMemcpyAsync(d_in_sets.p, host.data(), host.size() * 8, cudaMemcpyHostToDevice, stream));
    CK(cudaStreamSynchronize(stream));  // a later scan may run on another stream (n1gpu_query_set_stream)
    const u64* base = d_in_sets.as<u64>();
    in_descs.clear();
    for (size_t k = 0; k < S.size(); ++k) {
        NqInSet d{};
        d.bits = S[k].bits.empty() ? nullptr : (const u32*)(base + at[k]);
        d.keys = base + at[k] + (S[k].bits.size() + 1) / 2;
        d.icap = (u32)S[k].ikeys.size();
        d.fcap = (u32)S[k].fkeys.size();
        d.flags = S[k].flags;
        in_descs.push_back(d);
    }
}

void Query::rebind(Table* t) {
    if (!t || !t->sealed) N1_THROW(N1GPU_E_INVALID, "rebind needs a sealed table");
    if (t->cols.size() != table->cols.size() || t->nrows != table->nrows) N1_THROW(N1GPU_E_INVALID, "rebind: schema mismatch");
    for (size_t c = 0; c < t->cols.size(); ++c) {
        const Column &a = t->cols[c], &b = table->cols[c];
        if (a.path != b.path || a.width != b.width || a.stats.class_mask != b.stats.class_mask || a.stats.int_min != b.stats.int_min ||
            a.stats.int_max != b.stats.int_max || a.dict != b.dict)
            N1_THROW(N1GPU_E_INVALID, "rebind: column %zu differs in layout, statistics or dictionary", c);
    }
    table = t;
}

void Query::alloc_state() {
    const int W = ops.n;
    const i64 tile = (i64)kp.block * 4;
    i64 blocks_needed = std::max<i64>(1, (table->nrows + tile - 1) / tile);
    grid = (int)std::min<i64>(blocks_needed, (i64)device_sm_count() * kernel->max_blocks_per_sm);
    if (grid > 1280) grid = 1280;  // the last block folds at most 5 x 256 float partials per word
    if (kp.mode == MODE_UNGROUPED) {
        cap = 1;
        d_partials.ensure((size_t)grid * W * 8);
        if (!d_accum.p) {  // persistent order-independent accumulators, re-armed by the kernel's last block
            d_accum.alloc((size_t)W * 8);
            launch_init_words(d_accum.as<u64>(), 1, ops, nullptr);
            CK(cudaDeviceSynchronize());
        }
    }
    else if (kp.mode == MODE_DENSE) cap = (u64)kp.dense_slots;
    else {
        if (cap <= 1) {
            double want = 2.0 * std::min((double)std::max<i64>(table->nrows, 1), (double)std::max<i64>(kp.est_groups, 1));
            cap = pow2_at_least((u64)std::min(std::max(want, 1024.0), 67108864.0));
        }
        d_keys.ensure((size_t)cap * (kp.mode == MODE_HASH128 ? 16 : 8));
    }
    d_acc.ensure((size_t)cap * W * 8);
    if (kp.ndistinct) {
        if (kp.set_bitmap) set_cap = std::max<u64>(64, (u64)1 << kp.entry_bits);  // bits
        else if (set_cap == 0) {
            // every row can add one entry per set: at least twice as many slots (load <= 0.5 keeps linear probing to
            // ~1.5 slots per insert; at 0.7 it is over 5, each a DRAM sector) - HBM is plentiful, probes are not
            double want = 2.0 * (double)std::max<i64>(table->nrows, 1) * kp.ndistinct;
            set_cap = pow2_at_least((u64)std::min(std::max(want, 1024.0), 4294967296.0));
        }
        d_set.ensure(set_bytes());
    }
    if (part_kernel) {
        // every partition gets its expected share of this table's rows plus a quarter and a constant: uniform keys never
        // come near it, skewed ones overflow it and the handle falls back to the general scan (status 4)
        const u64 np = (u64)1 << kp.part_bits;
        part_cap = ((u64)std::max<i64>(table->nrows, 1) / np) * 5 / 4 + 4096;
        d_part_recs.ensure((size_t)(np * part_cap) * 4);
        d_part_cur.ensure((size_t)np * 4);
    }
    if (!d_cancel.p) {
        CK(cudaGetDevice(&device));
        d_cancel.alloc(64);
        CK(cudaMemset(d_cancel.p, 0, 64));
        h_cancel.ensure(64);
        *h_cancel.as<int>() = 1;
        CK(cudaStreamCreateWithFlags(&cancel_stream, cudaStreamNonBlocking));
    }
    d_status.ensure(64);
    h_status.ensure(64);
    memset(h_status.p, 0, 64);
    if (!d_ticket.p) { d_ticket.alloc(64); CK(cudaMemset(d_ticket.p, 0, 64)); }
    d_counts.ensure(4096);
    h_counts.ensure(4096);
    if (small_state()) h_records.ensure((size_t)cap * W * 8);
}

bool Query::uses_status() const { return kp.mode == MODE_HASH64 || kp.mode == MODE_HASH128 || kp.ndistinct > 0 || mailbox != nullptr; }

void Query::attach_mailbox(Mailbox* mb) {
    if (launched) N1_THROW(N1GPU_E_INVALID, "a scan is outstanding");
    if (peer_table && mailbox) { mailbox->arena_free(peer_off[1], peer_bytes); mailbox->arena_free(peer_off[0], peer_bytes); }
    if (peer_part && mailbox) { mailbox->arena_free(peer_cur_off, peer_cur_bytes); mailbox->arena_free(peer_recs_off, peer_recs_bytes); }
    peer_part = false;
    mailbox = mb;
    peer_table = false;
    peer_seq = 0;
    peer_steps = 0;
    // a direct-indexed table (slot == packed key on every rank) moves into the arena: peers fold it slot range by slot range
    if (mb && mb->arena_bytes && kp.mode == MODE_DENSE && kp.dense_global && kp.ndistinct == 0 && device_final_ok()) {
        peer_bytes = (size_t)cap * ops.n * 8;
        peer_off[0] = mb->arena_alloc(peer_bytes);
        peer_off[1] = mb->arena_alloc(peer_bytes);
        peer_table = true;
    }
    if (mb && mb->arena_bytes && mb->nranks > 1 && use_part() && table->global_rows > 0) {
        // every rank must lay its records out alike (peers index them): the share is derived from agreed numbers only
        const u64 np = (u64)1 << kp.part_bits;
        part_cap = ((u64)table->global_rows / (u64)mb->nranks / np + 1) * 3 / 2 + 4096;
        peer_recs_bytes = (size_t)(np * part_cap) * 4;
        peer_cur_bytes = (size_t)np * 4;
        peer_recs_off = mb->arena_alloc(peer_recs_bytes);
        peer_cur_off = mb->arena_alloc(peer_cur_bytes);
        peer_part = true;
        part_seq = 0;
    }
}

Mailbox::~Mailbox() {
    for (int r = 0; r < (int)peers.size(); ++r)
        if (r != rank && peers[r]) cudaIpcCloseMemHandle(peers[r]);
    if (base) cudaFree(base);
}

void Query::reset_state() {
    if (uses_status()) CK(cudaMemsetAsync(d_status.p, 0, 64, stream));
    if (kp.mode != MODE_UNGROUPED) launch_init_words(acc(), cap, ops, stream);
    if (kp.mode == MODE_HASH64 || kp.mode == MODE_HASH128) CK(cudaMemsetAsync(d_keys.p, 0xff, (size_t)cap * (kp.mode == MODE_HASH128 ? 16 : 8), stream));
    if (kp.ndistinct) CK(cudaMemsetAsync(d_set.p, kp.set_bitmap ? 0 : 0xff, set_bytes(), stream));
}

void Query::launch_scan() {
    if (!kernel) N1_THROW(N1GPU_E_CUDA, "no CUDA device: libn1gpu has no CPU fallback");
    if (launched) N1_THROW(N1GPU_E_INVALID, "a scan is already outstanding on this query");
    launches_at_start = g_launches.load();
    if (peer_table) { peer_seq = ++mailbox->seq; ++peer_steps; }  // flags are numbered per mailbox, table buffers alternate per query (acc())
    NqParams p{};
    p.nrows = table->nrows;
    for (size_t c = 0; c < table->cols.size(); ++c) { p.col[c] = table->cols[c].d_payload.p; p.tag[c] = table->cols[c].d_tags.as<u8>(); }
    for (size_t k = 0; k < kp.consts.size() && k < 32; ++k) p.cst[k] = kp.consts[k];
    for (size_t k = 0; k < in_descs.size(); ++k) p.inset[k] = in_descs[k];
    p.cancel = d_cancel.as<int>();
    p.acc = kp.mode == MODE_UNGROUPED ? d_accum.as<u64>() : acc();
    p.partials = d_partials.as<u64>();
    p.keys = d_keys.as<u64>();
    p.cap_mask = cap - 1;
    p.set_keys = d_set.as<u64>();
    p.set_mask = set_cap ? set_cap - 1 : 0;
    p.status = d_status.as<int>();
    p.dense_groups = (u64)kp.dense_slots;
    p.final_dev = acc();
    p.final_host = h_records.as<u64>();  // pinned memory is device-addressable under UVA: zero-copy result
    p.ticket = d_ticket.as<unsigned>();
    const bool small = small_state() && kp.ndistinct == 0;
    u64 mb_slot_base = 0, mb_seq = 0;
    if (mailbox && small && mailbox->nranks > 1) {
        const u64 words = cap * (u64)ops.n;
        if (words + 1 > mailbox->stride) N1_THROW(N1GPU_E_INVALID, "mailbox cells hold %llu words, the chain needs %llu", mailbox->stride - 1, words);
        mb_seq = ++mailbox->seq;
        const u64 slot = mb_seq % (u64)mailbox->slots;
        mb_slot_base = slot * (u64)mailbox->nranks * mailbox->stride;
        p.peer_mail = (u64* const*)mailbox->d_peers.p;
        p.nranks = mailbox->nranks;
        p.rank = mailbox->rank;
        p.mail_base = mb_slot_base + (u64)mailbox->rank * mailbox->stride;
        p.mail_words = words;
        p.mail_seq = mb_seq;
    }
    part_done = false;
    if (use_part()) {
        // partitioned DISTINCT aggregation: records partitioned by group range, then one block per partition
        const int np = 1 << kp.part_bits;
        const bool peers = peer_part_merge();
        u32* recs = peers ? (u32*)((char*)mailbox->base + peer_recs_off) : d_part_recs.as<u32>();
        u32* cur = peers ? (u32*)((char*)mailbox->base + peer_cur_off) : d_part_cur.as<u32>();
        const u64 nr = peers ? (u64)mailbox->nranks : 1;
        const u64* flags = peers ? (const u64*)((const char*)mailbox->base + mailbox->flags_off) : nullptr;
        CK(cudaMemsetAsync(d_status.p, 0, 64, stream));
        u64 seq = 0;
        if (peers) {
            seq = ++mailbox->seq;
            // the records of this rank's previous step may still be read by a peer: wait for everybody's "consumed" flag
            if (part_seq) launch_peer_wait(flags + (64 + part_seq % 64) * nr, (int)nr, part_seq, d_status.as<int>(), stream);
        }
        CK(cudaMemsetAsync(cur, 0, (size_t)np * 4, stream));
        if (timing) CK(cudaEventRecord(ev0, stream));
        p.set_keys = (u64*)recs;
        p.keys = (u64*)cur;
        p.set_mask = part_cap;
        const i64 tile = (i64)PART_THREADS * 4;
        const i64 tiles = (table->nrows + tile - 1) / tile;
        const int pgrid = (int)std::max<i64>(1, std::min<i64>((tiles + 7) / 8, (i64)device_sm_count()));
        jit_launch(*part_kernel, pgrid, stream, &p, sizeof p, false);
        PartPeers P;
        memset(&P, 0, sizeof P);
        P.n = (int)nr;
        P.recs[0] = recs;
        P.cur[0] = cur;
        if (peers) {
            launch_peer_signal((u64* const*)mailbox->d_peers.p, (int)nr, mailbox->rank, mailbox->flags_off / 8, seq, stream);
            launch_peer_wait(flags + (seq % 64) * nr, (int)nr, seq, d_status.as<int>(), stream);
            for (int r = 0; r < (int)nr; ++r) {
                P.recs[r] = (const u32*)((const char*)mailbox->peers[(size_t)r] + peer_recs_off);
                P.cur[r] = (const u32*)((const char*)mailbox->peers[(size_t)r] + peer_cur_off);
            }
        }
        int part0, part1;
        part_range(&part0, &part1);
        const DistinctDescs D = distinct_descs();
        const PackComp* dc = nullptr;
        for (auto& ap : kp.aggs) if (ap.distinct) { dc = &ap.dcomp; break; }
        launch_part_aggregate(P, part_cap, part0, part1, kp.part_gbits, kp.part_vbits, kp.phys_of[0], D, dc->classes[0] == C_INT, dc->bias, acc(), cap, stream);
        if (peers) {
            launch_peer_signal((u64* const*)mailbox->d_peers.p, (int)nr, mailbox->rank, mailbox->flags_off / 8 + 64 * nr, seq, stream);
            part_seq = seq;
        }
        if (timing) CK(cudaEventRecord(ev1, stream));
        timed_launch = timing;
        CK(cudaMemcpyAsync(h_status.p, d_status.p, 8, cudaMemcpyDeviceToHost, stream));
        launched = true;
        ungrouped_live = true;
        part_done = true;
        return;
    }
    reset_state();
    if (timing) CK(cudaEventRecord(ev0, stream));
    // ungrouped / dense: the whole step is this one launch.  Programmatic dependent launch only when nothing this
    // step enqueued before the scan (status / DISTINCT set clears) has to be complete when its first block starts.
    p.set_pass = 0;
    p.set_shift = kp.set_passes > 1 ? kp.entry_bits - bits_for((u64)kp.set_passes) : 63;
    jit_launch(*kernel, grid, stream, &p, sizeof p, kp.pdl && !uses_status());
    for (int pass = 1; pass < kp.set_passes; ++pass) {  // the other slices of the DISTINCT bitmap (see NqParams)
        p.set_pass = pass;
        jit_launch(*kernel, grid, stream, &p, sizeof p, false);
    }
    if (timing) CK(cudaEventRecord(ev1, stream));
    timed_launch = timing;
    if (peer_merge())  // this rank's table of step peer_seq is complete: tell every peer (stores over NVLink, release at system scope)
        launch_peer_signal((u64* const*)mailbox->d_peers.p, mailbox->nranks, mailbox->rank, mailbox->flags_off / 8, peer_seq, stream);
    if (mb_seq)  // receive side of the fused all-gather: fold every rank's words once they have landed
        launch_merge_mailbox((const u64*)mailbox->base, mailbox->nranks, mb_slot_base, mailbox->stride, cap * (u64)ops.n, mb_seq, cap, ops,
                             acc(), h_records.as<u64>(), d_status.as<int>(), stream);
    if (uses_status()) CK(cudaMemcpyAsync(h_status.p, d_status.p, 8, cudaMemcpyDeviceToHost, stream));
    launched = true;
    ungrouped_live = true;
}

bool Query::wait_scan() {
    if (!launched) N1_THROW(N1GPU_E_INVALID, "no scan outstanding");
    launched = false;
    CK(cudaStreamSynchronize(stream));
    if (timed_launch) {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ev0, ev1));
        last_scan_ms = ms;
    }
    if (cancelled.load()) N1_THROW(N1GPU_E_CANCELLED, "query cancelled");  // (the running kernel saw the flag and stopped early)
    int st = uses_status() ? h_status.as<int>()[0] : 0;
    if (st == 3) N1_THROW(N1GPU_E_CUDA, "multi-GPU merge timed out: a peer rank never delivered its partial state");
    if (st == 4 && peer_part_merge())
        N1_THROW(N1GPU_E_NOMEM, "a partition of the partitioned DISTINCT aggregation overflowed its share (skewed group keys): run this chain with N1GPU_NO_PART=1 on every rank");
    if (st == 4) {  // a partition overflowed (skewed group keys): the general one-kernel scan takes over for this handle
        part_disabled = true;
        part_done = false;
        return false;
    }
    if (st == 1) {
        if (cap >= ((u64)1 << 31)) N1_THROW(N1GPU_E_NOMEM, "group table would exceed 2^31 slots");
        cap *= 4;
        d_keys.alloc((size_t)cap * (kp.mode == MODE_HASH128 ? 16 : 8));
        d_acc.alloc((size_t)cap * ops.n * 8);
        return false;
    }
    if (st == 2) {
        if (set_cap >= ((u64)1 << 32)) N1_THROW(N1GPU_E_NOMEM, "DISTINCT set would exceed 2^32 slots");
        set_cap *= 4;
        d_set.alloc(set_bytes());
        return false;
    }
    host_acc_valid = small_state();
    return true;
}

void Query::scan_blocking() {
    for (;;) {
        if (cancelled.load()) N1_THROW(N1GPU_E_CANCELLED, "query cancelled");
        launch_scan();
        if (wait_scan()) return;
    }
}

// ---- partial state exchange -------------------------------------------------------------------------------------
static void count_and_export(Query& q, int kw, const u64* keys, const u64* acc, u64 cap, int W, int nranks, int gk_pos, int gk_bits,
                             u64* dev_out, i64 out_cap, i64* counts) {
    if (nranks > 256) N1_THROW(N1GPU_E_INVALID, "at most 256 ranks");
    CK(cudaMemsetAsync(q.d_counts.p, 0, 4096, q.stream));
    launch_count_owners(kw, keys, acc, cap, nranks, gk_pos, gk_bits, q.d_counts.as<unsigned long long>(), q.stream);
    CK(cudaMemcpyAsync(q.h_counts.p, q.d_counts.p, (size_t)nranks * 8, cudaMemcpyDeviceToHost, q.stream));
    CK(cudaStreamSynchronize(q.stream));
    unsigned long long* hc = q.h_counts.as<unsigned long long>();
    unsigned long long offs[256];
    unsigned long long total = 0;
    for (int r = 0; r < nranks; ++r) { counts[r] = (i64)hc[r]; offs[r] = total; total += hc[r]; }
    if (!dev_out) return;
    if ((i64)total > out_cap) N1_THROW(N1GPU_E_INVALID, "export buffer too small: %llu records > capacity %lld", total, (long long)out_cap);
    CK(cudaMemcpyAsync(q.d_counts.p, offs, (size_t)nranks * 8, cudaMemcpyHostToDevice, q.stream));
    launch_export_records(kw, keys, acc, cap, W, nranks, gk_pos, gk_bits, q.d_counts.as<unsigned long long>(), dev_out, (u64)out_cap, q.stream);
    CK(cudaStreamSynchronize(q.stream));
}

void Query::partial_counts(i64* ngroups, i64* ndistinct) {
    i64 c[1] = {0};
    count_and_export(*this, kw(), d_keys.as<u64>(), acc(), cap, ops.n, 1, 0, std::max(kp.key_bits, 0), nullptr, 0, c);
    if (kp.mode == MODE_UNGROUPED && !ungrouped_live) c[0] = 0;
    *ngroups = c[0];
    i64 d[1] = {0};
    if (kp.ndistinct) count_and_export(*this, set_kw(), d_set.as<u64>(), nullptr, set_cap, 0, 1, kp.abits, kp.key_bits, nullptr, 0, d);
    *ndistinct = d[0];
}

void Query::partial_export(int nranks, void* dev_records, i64 cap_records, i64* counts, void* dev_distinct, i64 cap_distinct, i64* dcounts) {
    count_and_export(*this, kw(), d_keys.as<u64>(), acc(), cap, ops.n, nranks, 0, kp.key_bits, (u64*)dev_records, cap_records, counts);
    if (kp.ndistinct)
        count_and_export(*this, set_kw(), d_set.as<u64>(), nullptr, set_cap, 0, nranks, kp.abits, kp.key_bits, (u64*)dev_distinct, cap_distinct, dcounts);
    else for (int r = 0; r < nranks; ++r) dcounts[r] = 0;
}

void Query::partial_reset() {
    if (!kernel) N1_THROW(N1GPU_E_CUDA, "no CUDA device");
    reset_state();
    if (kp.mode == MODE_UNGROUPED) launch_init_words(acc(), cap, ops, stream);
    CK(cudaStreamSynchronize(stream));
    ungrouped_live = false;
    host_acc_valid = false;
}

void Query::partial_import(const void* dev_records, i64 n, const void* dev_distinct, i64 nd) {
    if (!kernel) N1_THROW(N1GPU_E_CUDA, "no CUDA device");
    host_acc_valid = false;
    for (;;) {
        CK(cudaMemsetAsync(d_status.p, 0, 64, stream));
        if (n > 0) launch_merge_records(kw(), d_keys.as<u64>(), acc(), cap, ops, (const u64*)dev_records, (u64)n, d_status.as<int>(), stream);
        if (nd > 0) {
            OpsArr none{};
            none.n = 0;
            launch_merge_records(set_kw(), d_set.as<u64>(), nullptr, set_cap, none, (const u64*)dev_distinct, (u64)nd, d_status.as<int>() + 1, stream);
        }
        CK(cudaMemcpyAsync(h_status.p, d_status.p, 8, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        int s0 = h_status.as<int>()[0], s1 = h_status.as<int>()[1];
        if (!s0 && !s1) break;
        // The owner's table (sized for its own partition's groups) is too small for everybody's records: grow what
        // overflowed, clear the state (a half-applied merge cannot be kept: additions are not idempotent) and merge again -
        // the records are still in the caller's buffers.
        if (s0) {
            if (kp.mode != MODE_HASH64 && kp.mode != MODE_HASH128) N1_THROW(N1GPU_E_INVALID, "a record does not belong to this rank's table (bad key)");
            if (cap >= ((u64)1 << 31)) N1_THROW(N1GPU_E_NOMEM, "group table would exceed 2^31 slots");
            cap *= 4;
            d_keys.alloc((size_t)cap * (kp.mode == MODE_HASH128 ? 16 : 8));
            d_acc.alloc((size_t)cap * ops.n * 8);
        }
        if (s1) {
            if (kp.set_bitmap) N1_THROW(N1GPU_E_INVALID, "a DISTINCT entry lies outside this rank's bitmap");
            if (set_cap >= ((u64)1 << 32)) N1_THROW(N1GPU_E_NOMEM, "DISTINCT set would exceed 2^32 slots");
            set_cap *= 4;
            d_set.alloc(set_bytes());
        }
        reset_state();
    }
    if (n > 0) ungrouped_live = true;
}

// ---- finalisation (FinalGroup / ComputeFinal) -----------------------------------------------------------------------
namespace {
FinalComp final_comp(const PackComp& pc) {  // the plain data final_group.hpp decodes (keys, DISTINCT entry values)
    FinalComp c{};
    c.cbits = pc.cbits; c.pbits = pc.pbits; c.nfree = pc.nfree; c.biased = pc.biased; c.dict_col = pc.dict_col; c.bias = pc.bias;
    c.nclasses = (int)std::min<size_t>(8, pc.classes.size());
    for (int i = 0; i < c.nclasses; ++i) c.classes[i] = pc.classes[i];  // the rest stay C_MISSING
    return c;
}
}  // namespace

// slot of a shared-memory dense table -> the bit-packed group key (slots are the mixed-radix number of the components
// when that is tighter than the packed key: KernelPlan::dense_dom)
u64 Query::dense_key(u64 slot) const {
    if (kp.dense_dom.empty()) return slot;
    u64 key = 0;
    int pos = 0;
    for (size_t k = 0; k < kp.keys.size(); ++k) { key |= (slot % kp.dense_dom[k]) << pos; slot /= kp.dense_dom[k]; pos += kp.keys[k].bits(); }
    return key;
}

DistinctDescs Query::distinct_descs() const {
    DistinctDescs D{};
    for (auto& ap : kp.aggs) {
        if (!ap.distinct) continue;
        DistinctDesc& d = D.d[D.n++];
        d.sid = ap.distinct_id;
        d.numbers_only = ap.kind != AggKind::COUNT;
        d.w_cnt = ap.w_cnt; d.w_ilo = ap.w_ilo; d.w_ihi = ap.w_ihi; d.w_neg = ap.w_neg; d.w_fsum = ap.w_fsum; d.w_nflt = ap.w_nflt;
        d.value = final_comp(ap.dcomp);
    }
    return D;
}

FinalDesc Query::final_desc() const {
    FinalDesc D{};
    D.nkeys = (int)keys.size();
    D.naggs = (int)aggs.size();
    D.LW = (int)kp.word_ops.size();
    D.PW = ops.n;
    for (int l = 0; l < D.LW; ++l) {
        D.phys_of[l] = (unsigned char)kp.phys_of[l]; D.shift_of[l] = (unsigned char)kp.shift_of[l];
        D.bits_of[l] = (unsigned char)kp.bits_of[l]; D.complement[l] = kp.word_complement[l] ? 1 : 0;
    }
    if (device_final_ok())  // D.keys serves the device only: the host takes chains of more than 16 key components
        for (int k = 0; k < D.nkeys; ++k) D.keys[k] = final_comp(kp.keys[k]);
    for (int a = 0; a < D.naggs; ++a) D.aggs[a] = kp.aggs[a];
    return D;
}

i64 Query::finalize_device(Result& res, const PeerTables& tables, u64 slot0, u64 slot1) {
    const size_t nk = keys.size(), na = aggs.size();
    const u64 span = slot1 > slot0 ? slot1 - slot0 : 0;
    // Output capacity: every slot could hold a group.  When that worst case is large (sparse hash tables) the live slots
    // are counted first; the count needs a host round trip either way (the result arrays are sized by it).
    u64 out_cap = span;
    unsigned long long* counter = d_counts.as<unsigned long long>();
    const FinalDesc D = final_desc();
    const size_t per_group = (nk + na) * 9;
    if (span * per_group > ((size_t)256 << 20) && tables.n == 1) {
        i64 c[1] = {0};
        CK(cudaMemsetAsync(d_counts.p, 0, 64, stream));
        launch_count_owners(kw(), d_keys.as<u64>(), acc(), cap, 1, 0, std::max(kp.key_bits, 0), counter, stream);
        CK(cudaMemcpyAsync(h_counts.p, d_counts.p, 8, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        c[0] = (i64)h_counts.as<unsigned long long>()[0];
        out_cap = (u64)c[0];
    }
    auto up8 = [](size_t n) { return (n + 7) & ~(size_t)7; };
    const size_t o_kc = 0, o_ac = o_kc + up8(out_cap * nk), o_kv = o_ac + up8(out_cap * na), o_av = o_kv + out_cap * nk * 8;
    const size_t total = o_av + out_cap * na * 8;
    d_final.ensure(std::max<size_t>(total, 64));
    char* d = d_final.as<char>();
    CK(cudaMemsetAsync(d_counts.p, 0, 64, stream));
    launch_finalize_groups(D, kw(), d_keys.as<u64>(), tables, ops, cap, 1, slot0, slot1, counter, out_cap, (u8*)(d + o_kc), (i64*)(d + o_kv),
                           (u8*)(d + o_ac), (i64*)(d + o_av), stream);
    CK(cudaMemcpyAsync(h_counts.p, d_counts.p, 8, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    const u64 ng = h_counts.as<unsigned long long>()[0];
    if (tables.wait_flags) {
        CK(cudaMemcpy(h_status.p, d_status.p, 8, cudaMemcpyDeviceToHost));
        if (h_status.as<int>()[0] == 3) N1_THROW(N1GPU_E_CUDA, "multi-GPU merge timed out: a peer rank never signalled its partial table");
    }
    if (ng > out_cap) N1_THROW(N1GPU_E_INVALID, "finalisation found %llu groups in a table counted at %llu", (unsigned long long)ng, (unsigned long long)out_cap);
    const size_t h_kc = 0, h_ac = h_kc + up8(ng * nk), h_kv = h_ac + up8(ng * na), h_av = h_kv + ng * nk * 8;
    res.pinned.ensure(std::max<size_t>(h_av + ng * na * 8, 64));
    char* h = res.pinned.as<char>();
    if (ng) {
        if (nk) { CK(cudaMemcpyAsync(h + h_kc, d + o_kc, ng * nk, cudaMemcpyDeviceToHost, stream)); CK(cudaMemcpyAsync(h + h_kv, d + o_kv, ng * nk * 8, cudaMemcpyDeviceToHost, stream)); }
        if (na) { CK(cudaMemcpyAsync(h + h_ac, d + o_ac, ng * na, cudaMemcpyDeviceToHost, stream)); CK(cudaMemcpyAsync(h + h_av, d + o_av, ng * na * 8, cudaMemcpyDeviceToHost, stream)); }
        CK(cudaStreamSynchronize(stream));
    }
    res.key_cls.view((u8*)(h + h_kc), ng * nk);
    res.key_val.view((i64*)(h + h_kv), ng * nk);
    res.agg_cls.view((u8*)(h + h_ac), ng * na);
    res.agg_val.view((i64*)(h + h_av), ng * na);
    return (i64)ng;
}

std::unique_ptr<Result> Query::finalize() {
    const int W = ops.n;
    const int rw = 2 + W;
    std::vector<u64> recs;
    i64 ngroups = 0;
    const bool trace = getenv("N1GPU_TRACE") != nullptr;
    double tp = now_sec();
    auto phase = [&](const char* name) { if (trace) { double t = now_sec(); fprintf(stderr, "[n1gpu finalize] %-22s %8.3f ms\n", name, (t - tp) * 1e3); tp = t; } };
    if (kp.ndistinct && !part_done) {
        // DISTINCT aggregates are finalised on the device: every set entry adds itself to its group's result words
        const DistinctDescs D = distinct_descs();
        for (auto& ap : kp.aggs) {
            if (!ap.distinct) continue;
            for (int w : {ap.w_cnt, ap.w_ilo, ap.w_ihi, ap.w_neg, ap.w_fsum, ap.w_nflt})
                if (w >= 0) launch_fill_u64(acc() + (u64)w * cap, cap, 0, stream);  // idempotent finalize
        }
        launch_distinct_finalize(d_set.as<u64>(), set_cap, kp.set_bitmap ? 2 : (kp.set128 ? 1 : 0), kp.abits, kp.key_bits, kw(), d_keys.as<u64>(), cap,
                                 acc(), D, stream);
        CK(cudaStreamSynchronize(stream));
    }
    std::unique_ptr<Result> res(new Result());
    res->nkeys = (int)keys.size();
    res->naggs = (int)aggs.size();
    res->agg_texts = agg_texts;
    res->key_texts = key_texts;
    res->alias = alias;
    for (auto& k : keys) {
        std::vector<std::string> path;
        if (k->kind == EK::FIELD && k->col >= 0) path = table->cols[k->col].path;
        res->key_paths.push_back(path);
    }
    const bool host_words = small_state() && h_records.p && !import_dirty() && !kp.ndistinct;
    // Everything but the few-slot states is finalised ON THE DEVICE (k_finalize_groups): a scan of 10^9 rows leaves up
    // to 10^6 groups, and ComputeFinal + key decoding of those on host cores took 17x the scan itself.
    const bool on_device = !host_words && kp.mode != MODE_UNGROUPED && device_final_ok() && kp.dense_dom.empty();
    if (on_device) {
        PeerTables T;
        memset(&T, 0, sizeof T);
        T.n = 1;
        T.acc[0] = acc();
        u64 s0 = 0, s1 = cap;
        if (part_done && peer_part_merge()) {  // this rank aggregated (and now finalises) its range of partitions only
            int part0, part1;
            part_range(&part0, &part1);
            s0 = (u64)part0 << kp.part_gbits;
            s1 = std::min<u64>(cap, (u64)part1 << kp.part_gbits);
        }
        if (peer_merge() && peer_seq) {
            // IntermediateGroup + FinalGroup fused and owner-sharded: this rank folds ITS slot range of every rank's table
            T.n = mailbox->nranks;
            for (int r = 0; r < T.n; ++r) T.acc[r] = (const u64*)((const char*)mailbox->peers[(size_t)r] + peer_off[peer_steps & 1]);
            s0 = cap * (u64)mailbox->rank / (u64)T.n;
            s1 = cap * (u64)(mailbox->rank + 1) / (u64)T.n;
            T.wait_flags = (const u64*)((const char*)mailbox->base + mailbox->flags_off) + (peer_seq % 64) * (u64)T.n;
            T.wait_seq = peer_seq;
            T.status = d_status.as<int>();
        }
        ngroups = finalize_device(*res, T, s0, s1);
        res->ngroups = ngroups;
        phase("device finalize + D2H");
    } else {
    if (host_words) {
        // small state: the scan already published the table words to pinned host memory
        const u64* h = h_records.as<u64>();
        for (u64 i = 0; i < cap; ++i) {
            if (kp.mode == MODE_DENSE && h[i] == 0) continue;  // word 0 = rows in group
            if (kp.mode == MODE_UNGROUPED && !ungrouped_live) continue;
            recs.push_back(dense_key(i)); recs.push_back(0);
            for (int w = 0; w < W; ++w) recs.push_back(h[(u64)w * cap + i]);
            ++ngroups;
        }
    } else {
        i64 c[1];
        count_and_export(*this, kw(), d_keys.as<u64>(), acc(), cap, W, 1, 0, kp.key_bits, nullptr, 0, c);
        if (kp.mode == MODE_UNGROUPED && !ungrouped_live) c[0] = 0;
        ngroups = c[0];
        if (ngroups) {
            d_records.ensure((size_t)ngroups * rw * 8);
            i64 c2[1];
            count_and_export(*this, kw(), d_keys.as<u64>(), acc(), cap, W, 1, 0, kp.key_bits, d_records.as<u64>(), ngroups, c2);
            recs.resize((size_t)ngroups * rw);
            CK(cudaMemcpy(recs.data(), d_records.p, recs.size() * 8, cudaMemcpyDeviceToHost));
            if (!kp.dense_dom.empty()) for (i64 g = 0; g < ngroups; ++g) recs[(size_t)g * rw] = dense_key(recs[(size_t)g * rw]);
        }
    }

    phase("distinct + export");
    res->ngroups = ngroups;
    res->key_cls.resize((size_t)ngroups * res->nkeys);
    res->key_val.resize((size_t)ngroups * res->nkeys);
    res->agg_cls.resize((size_t)ngroups * res->naggs);
    res->agg_val.resize((size_t)ngroups * res->naggs);

    phase("result allocation");
    // FinalGroup of every group (final_group.hpp, as on the device); a large group table (config 4: 10^6 groups) is
    // finalised by all host cores
    const FinalDesc D = final_desc();
    std::vector<FinalComp> kcomps;
    for (auto& pc : kp.keys) kcomps.push_back(final_comp(pc));
    const int nk = res->nkeys, na = res->naggs;
    auto final_range = [&](i64 g0, i64 g1) {
        for (i64 g = g0; g < g1; ++g) {
            const u64* r = &recs[(size_t)g * rw];  // [key lo, key hi, physical words]
            final_group(D, kcomps.data(), nk, r[0], r[1], r + 2, res->key_cls.data() + g * nk, res->key_val.data() + g * nk,
                        res->agg_cls.data() + g * na, res->agg_val.data() + g * na);
        }
    };
    {
        const int nthr = ngroups < 32768 ? 1 : (int)std::min<i64>(std::max(1u, std::thread::hardware_concurrency()), 32);
        if (nthr <= 1) final_range(0, ngroups);
        else {
            std::vector<std::thread> pool;
            for (int t = 0; t < nthr; ++t) pool.emplace_back([&, t] { final_range(ngroups * t / nthr, ngroups * (t + 1) / nthr); });
            for (auto& th : pool) th.join();
        }
    }
    }  // host finalisation
    bool any_string = false;  // can a key or an aggregate be a string at all?
    for (auto& pc : kp.keys) any_string = any_string || (pc.mask & bit(C_STRING));
    for (auto& ap : kp.aggs) any_string = any_string || ap.w_ms >= 0;
    if (any_string) {   // strings stay (column, rank) references: the result shares the dictionaries, nothing is copied
        res->string_refs = true;
        res->dicts.resize(table->cols.size());
        for (auto& pc : kp.keys) if (pc.dict_col >= 0) res->dicts[(size_t)pc.dict_col] = table->cols[(size_t)pc.dict_col].dict.share();
        for (auto& ap : kp.aggs) if (ap.w_ms >= 0 && ap.dict_col >= 0) res->dicts[(size_t)ap.dict_col] = table->cols[(size_t)ap.dict_col].dict.share();
    }
    phase("ComputeFinal");
    i64 scan_bytes = (i64)kp.scan_bytes_per_row * table->nrows;
    res->stats[0] = table->nrows;
    res->stats[1] = ngroups;
    res->stats[2] = (i64)(last_scan_ms * 1e6);
    res->stats[3] = (i64)((table->shred_sec + table->upload_sec) * 1e9);
    res->stats[4] = scan_bytes;
    res->stats[5] = (i64)(g_launches.load() - launches_at_start);
    return res;
}

}  // namespace n1
