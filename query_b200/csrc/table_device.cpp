// table_device.cpp — host orchestration of the device-side shredder (shred.cu): raw JSON goes to HBM once, the
// columns are produced there (no column H2D at all), dictionaries are built from a device hash set of distinct
// strings whose (few) members the host sorts bytewise, and only the documents the device could not decide exactly
// are re-shredded on the host (fix-up rows) and patched in.
#include <algorithm>
#include <cstdlib>
#include <functional>
#include <thread>

#include "shred.hpp"
#include "table.hpp"

namespace n1 {

namespace {

void build_trie(const std::vector<Column>& cols, ShredTrie& T) {
    // adjacency first (node -> list of (name, child)), then flatten so that every node's kids are contiguous
    struct N { std::vector<std::pair<std::string, int>> kids; int col = -1; };
    std::vector<N> nodes(1);
    for (size_t c = 0; c < cols.size(); ++c) {
        int n = 0;
        for (auto& name : cols[c].path) {
            int next = -1;
            for (auto& k : nodes[n].kids) if (k.first == name) next = k.second;
            if (next < 0) { nodes.emplace_back(); next = (int)nodes.size() - 1; nodes[n].kids.emplace_back(name, next); }
            n = next;
        }
        nodes[n].col = (int)c;
    }
    if (nodes.size() > 64) N1_THROW(N1GPU_E_INELIGIBLE, "device shredder: more than 64 path nodes");
    memset(&T, 0, sizeof T);
    T.nnodes = (int)nodes.size();
    int kid = 0, name_at = 0;
    for (size_t n = 0; n < nodes.size(); ++n) {
        T.col[n] = nodes[n].col;
        T.kid_begin[n] = kid;
        for (auto& k : nodes[n].kids) {
            if (kid >= 64) N1_THROW(N1GPU_E_INELIGIBLE, "device shredder: more than 64 field names");
            if (name_at + (int)k.first.size() > (int)sizeof T.names) N1_THROW(N1GPU_E_INELIGIBLE, "device shredder: field names too long");
            T.name_off[kid] = name_at;
            T.name_len[kid] = (int)k.first.size();
            memcpy(T.names + name_at, k.first.data(), k.first.size());
            name_at += (int)k.first.size();
            T.kid_node[kid] = k.second;
            ++kid;
        }
        T.kid_end[n] = kid;
    }
    T.nkids = kid;
}

u64 pow2_at_least(u64 n) { u64 p = 1; while (p < n) p <<= 1; return p; }

// A column in device memory: class bytes and, for 8-byte payloads, the payload words (k_col_stats reads those of INT rows)
struct DevColumn { const u8* tags; const i64* pay8; i64 rows; };

// Statistics of device columns (the dictionary's aside), k_col_stats on `s` - one round trip for all of them
std::vector<ColumnStats> device_stats(const std::vector<DevColumn>& cols, cudaStream_t s) {
    const size_t n = cols.size();
    if (!n) return {};
    std::vector<u64> w(n * 8, 0);  // per column: class mask, int min, int max, has float, absent rows, (unused)
    for (size_t c = 0; c < n; ++c) { w[c * 8 + 1] = (u64)INT64_MAX; w[c * 8 + 2] = (u64)INT64_MIN; }
    DevBuf d;
    d.alloc(n * 64);
    CK(cudaMemcpyAsync(d.p, w.data(), n * 64, cudaMemcpyHostToDevice, s));
    for (size_t c = 0; c < n; ++c)
        if (cols[c].rows) launch_col_stats(cols[c].tags, cols[c].pay8, cols[c].rows, d.as<u64>() + c * 8, s);
    CK(cudaMemcpyAsync(w.data(), d.p, n * 64, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    std::vector<ColumnStats> out(n);
    for (size_t c = 0; c < n; ++c) {
        const u64* x = &w[c * 8];
        ColumnStats& st = out[c];
        st.class_mask = (u32)x[0];
        st.has_int = (st.class_mask & bit(C_INT)) != 0;
        if (st.has_int) { st.int_min = (i64)x[1]; st.int_max = (i64)x[2]; }
        st.has_float = x[3] != 0;
        st.absent_rows = (i64)x[4];
    }
    return out;
}

}  // namespace

void Table::append_json_device(const char* buf, const i64* offsets, i64 ndocs) {
    if (ndocs < 0) N1_THROW(N1GPU_E_INVALID, "negative document count");
    append_text_device(buf, offsets, ndocs, 0, nullptr);
}

// One JSON document per line, `size` bytes at text (readable up to text + size + 64): the document offsets are computed on
// the device from the text itself (k_ndjson_lines) - no host pass over the text, no offsets over PCIe.
void Table::append_ndjson_device(const char* text, i64 size, const std::function<void(i64, i64)>& fill) { append_text_device(text, nullptr, -1, size, fill); }

void Table::append_text_device(const char* buf, const i64* offsets, i64 ndocs, i64 text_size, const std::function<void(i64, i64)>& fill) {
    const bool lines = offsets == nullptr;  // NDJSON: offsets come from the device
    admit(Entry::APPEND_DEVICE);
    if (cols.empty() && lines) N1_THROW(N1GPU_E_INVALID, "a table without columns cannot split lines on the device");
    if (cols.empty()) {  // a chain that references no field (COUNT(*) only): rows are all that matters
        nrows = ndocs;
        filled = Fill::DEVICE_DOCS;
        return;
    }
    double t0 = now_sec();
    const bool trace = getenv("N1GPU_TRACE") != nullptr;
    double tp = t0;
    auto phase = [&](const char* name) { if (trace) { double t = now_sec(); fprintf(stderr, "[n1gpu shred] %-22s %8.3f ms\n", name, (t - tp) * 1e3); tp = t; } };
    const i64 base_off = lines ? 0 : (ndocs ? offsets[0] : 0);
    const i64 nbytes = lines ? text_size : (ndocs ? offsets[ndocs] - base_off : 0);
    const int ncols = (int)cols.size();
    cudaStream_t s = nullptr;
    CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    struct StreamGuard { cudaStream_t s; ~StreamGuard() { cudaStreamDestroy(s); } } sg{s};

    ShredTrie trie;
    build_trie(cols, trie);
    DevBuf d_trie, d_buf, d_offs, d_fixcount, d_fixrows, d_ptrs;
    d_trie.alloc(sizeof trie);
    CK(cudaMemcpyAsync(d_trie.p, &trie, sizeof trie, cudaMemcpyHostToDevice, s));
    d_buf.alloc((size_t)nbytes + 64);
    std::vector<i64> rel;
    const i64* offs_src = offsets;
    if (lines) {
        // the whole text, then its line starts: counts per segment, scan, offsets (all on `s`, one host round trip for ndocs)
        CK(cudaMemsetAsync((char*)d_buf.p + nbytes, '\n', 64, s));
        const i64 chunk = (i64)64 << 20;
        for (i64 at = 0; at < nbytes; at += chunk) {
            const i64 hi = std::min(at + chunk, nbytes);
            if (fill) fill(at, hi);  // (the copy of the chunk before this one is in flight meanwhile)
            CK(cudaMemcpyAsync((char*)d_buf.p + at, buf + at, (size_t)(hi - at), cudaMemcpyHostToDevice, s));
        }
        const i64 nseg = ndjson_segments(nbytes);
        DevBuf d_counts, d_first;
        d_counts.alloc((size_t)(nseg + 1) * 4);
        d_first.alloc((size_t)(nseg + 1) * 8);
        launch_ndjson_count((const unsigned char*)d_buf.p, nbytes, d_counts.as<unsigned>(), s);
        DevBuf d_tiles;
        d_tiles.alloc((size_t)(ndjson_scan_tiles(nseg) + 1) * 8);
        launch_ndjson_scan(d_counts.as<unsigned>(), nseg, d_first.as<i64>(), d_tiles.as<i64>(), s);
        i64 total = 0;
        CK(cudaMemcpyAsync(&total, d_first.as<i64>() + nseg, 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        ndocs = total;
        d_offs.alloc((size_t)(ndocs + 1) * 8);
        launch_ndjson_write((const unsigned char*)d_buf.p, nbytes, d_first.as<i64>(), d_offs.as<i64>(), s);
        CK(cudaMemcpyAsync(d_offs.as<i64>() + ndocs, &nbytes, 8, cudaMemcpyHostToDevice, s));
        CK(cudaStreamSynchronize(s));  // (&nbytes and the temporaries above go out of scope)
        phase("h2d + line starts");
    } else {
        d_offs.alloc((size_t)(ndocs + 1) * 8);
        if (base_off != 0) {  // device offsets are relative to d_buf
            rel.resize((size_t)ndocs + 1);
            for (i64 i = 0; i <= ndocs; ++i) rel[(size_t)i] = offsets[i] - base_off;
            offs_src = rel.data();
        }
        if (!ndocs) { i64 z = 0; CK(cudaMemcpyAsync(d_offs.p, &z, 8, cudaMemcpyHostToDevice, s)); }
    }

    nrows = ndocs;
    const i64 pad = std::max(padded_rows(), ROW_PAD);
    std::vector<DevBuf> pay8((size_t)ncols);
    std::vector<u8*> h_tags((size_t)ncols);
    std::vector<i64*> h_pay((size_t)ncols);
    for (int c = 0; c < ncols; ++c) {
        cols[c].d_tags = device_rows(1, C_MISSING, s);
        pay8[c] = device_rows(8, 0, s);
        h_tags[c] = cols[c].d_tags.as<u8>();
        h_pay[c] = pay8[c].as<i64>();
    }
    d_ptrs.alloc((size_t)ncols * 16);
    CK(cudaMemcpyAsync(d_ptrs.p, h_tags.data(), (size_t)ncols * 8, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync((char*)d_ptrs.p + (size_t)ncols * 8, h_pay.data(), (size_t)ncols * 8, cudaMemcpyHostToDevice, s));
    const i64 fix_cap = std::max<i64>(1024, std::min<i64>(ndocs, 1 << 22));
    d_fixcount.alloc(64);
    CK(cudaMemsetAsync(d_fixcount.p, 0, 64, s));
    d_fixrows.alloc((size_t)fix_cap * 8);

    // The raw JSON crosses PCIe in chunks on a copy stream while the parse kernel of the chunks that have landed runs on
    // `s`: the document bytes and their offsets of chunk i+1 travel while chunk i is shredded (the H2D of the text is what
    // bounds this path - 13 ms per 664 MB - so the ~4 ms of parsing hide behind it).
    if (lines)
        launch_shred_json((const unsigned char*)d_buf.p, d_offs.as<i64>(), 0, ndocs, (const ShredTrie*)d_trie.p, (u8* const*)d_ptrs.p,
                          (i64* const*)((char*)d_ptrs.p + (size_t)ncols * 8), ncols, d_fixcount.as<unsigned>(), d_fixrows.as<i64>(), fix_cap, s);
    else if (ndocs) {
        cudaStream_t cs = nullptr;
        CK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
        struct CopyGuard { cudaStream_t s; ~CopyGuard() { cudaStreamDestroy(s); } } cg{cs};
        cudaEvent_t ready_to_copy, landed;
        CK(cudaEventCreateWithFlags(&ready_to_copy, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&landed, cudaEventDisableTiming));
        CK(cudaEventRecord(ready_to_copy, s));       // allocations / clears above are ordered before the first copy
        CK(cudaStreamWaitEvent(cs, ready_to_copy, 0));
        const i64 chunk_bytes = (i64)48 << 20;
        i64 d0 = 0;
        while (d0 < ndocs) {
            i64 d1 = d0;  // documents [d0, d1): about chunk_bytes of text
            {
                const i64 want = offs_src[d0] + chunk_bytes;
                i64 lo = d0 + 1, hi = ndocs;
                while (lo < hi) { const i64 mid = (lo + hi) >> 1; if (offs_src[mid] >= want) hi = mid; else lo = mid + 1; }
                d1 = lo;
            }
            CK(cudaMemcpyAsync(d_offs.as<i64>() + d0, offs_src + d0, (size_t)(d1 - d0 + 1) * 8, cudaMemcpyHostToDevice, cs));
            CK(cudaMemcpyAsync((char*)d_buf.p + offs_src[d0], buf + base_off + offs_src[d0], (size_t)(offs_src[d1] - offs_src[d0]), cudaMemcpyHostToDevice, cs));
            CK(cudaEventRecord(landed, cs));
            CK(cudaStreamWaitEvent(s, landed, 0));
            launch_shred_json((const unsigned char*)d_buf.p, d_offs.as<i64>(), d0, d1 - d0, (const ShredTrie*)d_trie.p, (u8* const*)d_ptrs.p,
                              (i64* const*)((char*)d_ptrs.p + (size_t)ncols * 8), ncols, d_fixcount.as<unsigned>(), d_fixrows.as<i64>(), fix_cap, s);
            d0 = d1;
        }
        CK(cudaStreamSynchronize(cs));
        CK(cudaEventDestroy(ready_to_copy));
        CK(cudaEventDestroy(landed));
    }
    unsigned nfix = 0;
    CK(cudaMemcpyAsync(&nfix, d_fixcount.p, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if ((i64)nfix > fix_cap)
        N1_THROW(N1GPU_E_INVALID, "device shredder: %u documents need host handling (escapes / long numbers); shred this keyspace with host threads", nfix);

    phase("alloc+h2d+parse kernel");
    // ---- fix-up rows: the host shredder decides these documents -----------------------------------------------------
    std::string extra;  // unescaped string values of fix-up rows (device refs carry REF_EXTRA_BIT)
    DevBuf d_extra;
    if (nfix) {
        std::vector<i64> rows(nfix);
        CK(cudaMemcpy(rows.data(), d_fixrows.p, (size_t)nfix * 8, cudaMemcpyDeviceToHost));
        std::sort(rows.begin(), rows.end());
        std::vector<HostShredOut> fx;
        if (lines) {
            // the documents' offsets live on the device: fetch those of the fix-up rows and shred them as a compact list
            DevBuf d_r, d_o;
            d_r.alloc((size_t)nfix * 8);
            d_o.alloc((size_t)nfix * 16);
            CK(cudaMemcpyAsync(d_r.p, rows.data(), (size_t)nfix * 8, cudaMemcpyHostToDevice, s));
            launch_gather_offsets(d_offs.as<i64>(), d_r.as<i64>(), (i64)nfix, d_o.as<i64>(), s);
            std::vector<i64> pairs((size_t)nfix * 2), idx(nfix);
            CK(cudaMemcpyAsync(pairs.data(), d_o.p, pairs.size() * 8, cudaMemcpyDeviceToHost, s));
            CK(cudaStreamSynchronize(s));
            // host_shred_docs reads document i as [offs[i], offs[i + 1]): lay the pairs out as their own offset list
            std::vector<i64> fo;
            std::string ftext;
            fo.push_back(0);
            for (unsigned i = 0; i < nfix; ++i) { ftext.append(buf + pairs[2 * i], (size_t)(pairs[2 * i + 1] - pairs[2 * i])); fo.push_back((i64)ftext.size()); idx[i] = (i64)i; }
            host_shred_docs(cols, ftext.data(), fo.data(), idx.data(), (i64)nfix, fx);
        } else
        host_shred_docs(cols, buf, offsets, rows.data(), (i64)nfix, fx);
        std::vector<std::vector<i64>> pays((size_t)ncols);
        for (int c = 0; c < ncols; ++c) {
            pays[c] = fx[c].payload;
            for (size_t i = 0; i < rows.size(); ++i) {
                if (fx[c].tags[i] != C_STRING) continue;
                const std::string& str = fx[c].strings[(size_t)fx[c].payload[i]];
                if (str.size() >= (1u << 24)) N1_THROW(N1GPU_E_INELIGIBLE, "string value longer than 16 MiB");
                pays[c][i] = (i64)(0x8000000000000000ULL | ((u64)extra.size() << 24) | (u64)str.size());
                extra += str;
            }
        }
        d_extra.alloc(extra.size() + 64);
        if (!extra.empty()) CK(cudaMemcpyAsync(d_extra.p, extra.data(), extra.size(), cudaMemcpyHostToDevice, s));
        DevBuf d_rows, d_pt, d_pp;
        d_rows.alloc((size_t)nfix * 8);
        d_pt.alloc((size_t)nfix);
        d_pp.alloc((size_t)nfix * 8);
        CK(cudaMemcpyAsync(d_rows.p, rows.data(), (size_t)nfix * 8, cudaMemcpyHostToDevice, s));
        for (int c = 0; c < ncols; ++c) {
            CK(cudaMemcpyAsync(d_pt.p, fx[c].tags.data(), (size_t)nfix, cudaMemcpyHostToDevice, s));
            CK(cudaMemcpyAsync(d_pp.p, pays[c].data(), (size_t)nfix * 8, cudaMemcpyHostToDevice, s));
            launch_patch(cols[c].d_tags.as<u8>(), pay8[c].as<i64>(), d_rows.as<i64>(), d_pt.as<u8>(), d_pp.as<i64>(), (i64)nfix, s);
            CK(cudaStreamSynchronize(s));  // d_pt / d_pp are reused by the next column
        }
    } else d_extra.alloc(64);

    phase("fix-up rows");
    // ---- statistics (class mask, int range) -------------------------------------------------------------------------
    std::vector<DevColumn> dc;
    for (int c = 0; c < ncols; ++c) dc.push_back(DevColumn{cols[c].d_tags.as<u8>(), pay8[c].as<i64>(), ndocs});
    std::vector<ColumnStats> stats = device_stats(dc, s);

    phase("statistics");
    // ---- dictionaries + final payload width ------------------------------------------------------------------------------
    DevBuf d_slots, d_keys, d_status, d_count, d_oslots, d_orefs, d_rank;
    d_status.alloc(64);
    d_count.alloc(64);
    for (int c = 0; c < ncols; ++c) {
        Column& col = cols[c];
        ColumnStats& st = stats[c];
        col.dict.clear();
        const bool has_str = st.class_mask & bit(C_STRING);
        col.width = width_of(st.class_mask);
        if (has_str) {
            d_slots.ensure((size_t)pad * 8);
            // (a sparse table is cheap - 8 bytes per slot, cleared by a memset - a dense one costs string compares per probe)
            u64 cap = std::max<u64>((u64)1 << 16, std::min<u64>((u64)1 << 21, pow2_at_least((u64)ndocs / 4)));
            std::vector<u64> oslots, orefs;
            for (;;) {
                d_keys.ensure((size_t)cap * 8);
                CK(cudaMemsetAsync(d_keys.p, 0xff, (size_t)cap * 8, s));
                CK(cudaMemsetAsync(d_status.p, 0, 64, s));
                launch_dict_insert((const unsigned char*)d_buf.p, (const unsigned char*)d_extra.p, col.d_tags.as<u8>(), pay8[c].as<i64>(),
                                   d_slots.as<i64>(), ndocs, d_keys.as<u64>(), cap, d_status.as<int>(), s);
                int status = 0;
                CK(cudaMemcpyAsync(&status, d_status.p, 4, cudaMemcpyDeviceToHost, s));
                CK(cudaStreamSynchronize(s));
                if (status == 0) {
                    // the table must stay sparse enough for cheap probing; a dense one means high cardinality: grow
                    d_oslots.ensure((size_t)cap * 8);
                    d_orefs.ensure((size_t)cap * 8);
                    CK(cudaMemsetAsync(d_count.p, 0, 64, s));
                    launch_dict_collect(d_keys.as<u64>(), cap, d_count.as<unsigned>(), d_oslots.as<u64>(), d_orefs.as<u64>(), cap, s);
                    unsigned m = 0;
                    CK(cudaMemcpyAsync(&m, d_count.p, 4, cudaMemcpyDeviceToHost, s));
                    CK(cudaStreamSynchronize(s));
                    if ((u64)m * 2 <= cap || cap >= pow2_at_least((u64)ndocs * 2)) {
                        oslots.resize(m);
                        orefs.resize(m);
                        if (m) {
                            CK(cudaMemcpy(oslots.data(), d_oslots.p, (size_t)m * 8, cudaMemcpyDeviceToHost));
                            CK(cudaMemcpy(orefs.data(), d_orefs.p, (size_t)m * 8, cudaMemcpyDeviceToHost));
                        }
                        break;
                    }
                }
                if (cap > ((u64)1 << 33)) N1_THROW(N1GPU_E_NOMEM, "dictionary table too large");
                cap *= 8;
            }
            phase("  dictionary insert");
            // sort the distinct strings bytewise on the host: rank = N1QL collation order (value/string.go:116-126)
            // The distinct strings lie scattered over the raw text (hundreds of megabytes): every compare of a sort over
            // them would be two cache misses.  They are gathered once, on all cores, into one compact blob together with
            // their first 8 bytes as a big-endian integer; the sort compares those integers and touches the (compact)
            // bytes only for ties.  10^5 strings of config 5: 6.8 ms -> about 1.5 ms.
            struct Ent { u64 prefix; u32 at; u32 len; u64 slot; };
            const size_t nent = oslots.size();
            std::vector<Ent> ents(nent);
            std::vector<u32> starts(nent + 1, 0);
            for (size_t i = 0; i < nent; ++i) starts[i + 1] = starts[i] + (u32)(orefs[i] & 0xffffff);
            std::string compact((size_t)starts[nent], '\0');
            const int nthr = nent < 20000 ? 1 : (int)std::min<size_t>(std::max(1u, std::thread::hardware_concurrency()), 16);
            parallel_for(nthr, [&](size_t r) {
                for (size_t i = nent * r / nthr; i < nent * (r + 1) / nthr; ++i) {
                    const u64 ref = orefs[i];
                    const u64 off = (ref & ~0x8000000000000000ULL) >> 24;
                    const char* src = (ref >> 63) ? extra.data() + off : buf + base_off + off;
                    const u32 len = (u32)(ref & 0xffffff);
                    memcpy(&compact[starts[i]], src, len);
                    u64 pre = 0;
                    for (u32 k = 0; k < 8; ++k) pre = (pre << 8) | (k < len ? (unsigned char)src[k] : 0u);
                    ents[i] = Ent{pre, starts[i], len, oslots[i]};
                }
            });
            phase("    strings gathered");
            const char* cb = compact.data();
            auto less = [cb](const Ent& a, const Ent& b) {
                if (a.prefix != b.prefix) return a.prefix < b.prefix;  // big-endian image of the first 8 bytes: bytewise order
                if (a.len <= 8 || b.len <= 8) return a.len < b.len;    // equal padded prefixes: the shorter one is a prefix of the other
                const int c = memcmp(cb + a.at + 8, cb + b.at + 8, std::min(a.len, b.len) - 8);
                return c != 0 ? c < 0 : a.len < b.len;
            };
            if (nthr > 1) {
                // sample sort: buckets by splitters drawn from the prefixes (equal prefixes share a bucket), every bucket sorted on
                // its own core - no merge levels.  Strings that all share their first 8 bytes degenerate to one bucket.
                const size_t B = (size_t)nthr, S = 64 * B;
                std::vector<u64> sample(S);
                for (size_t i = 0; i < S; ++i) sample[i] = ents[nent * i / S].prefix;
                std::sort(sample.begin(), sample.end());
                std::vector<u64> split(B - 1);
                for (size_t k = 0; k + 1 < B; ++k) split[k] = sample[(k + 1) * S / B];
                std::vector<u32> bucket(nent);
                std::vector<std::vector<size_t>> cnt(B, std::vector<size_t>(B, 0));  // [thread][bucket]
                parallel_for(nthr, [&](size_t r) {
                    for (size_t i = nent * r / B; i < nent * (r + 1) / B; ++i) {
                        const u32 k = (u32)(std::upper_bound(split.begin(), split.end(), ents[i].prefix) - split.begin());
                        bucket[i] = k;
                        ++cnt[r][k];
                    }
                });
                // bucket k = [count[k], count[k + 1]); inside it thread r's entries follow those of the threads before it
                std::vector<size_t> count(B + 1, 0);
                for (size_t k = 0; k < B; ++k) { size_t tot = 0; for (size_t r = 0; r < B; ++r) tot += cnt[r][k]; count[k + 1] = count[k] + tot; }
                phase("    buckets counted");
                std::vector<Ent> sorted(nent);
                parallel_for(nthr, [&](size_t r) {
                    std::vector<size_t> cursor(B);
                    for (size_t k = 0; k < B; ++k) { size_t at = count[k]; for (size_t q = 0; q < r; ++q) at += cnt[q][k]; cursor[k] = at; }
                    for (size_t i = nent * r / B; i < nent * (r + 1) / B; ++i) sorted[cursor[bucket[i]]++] = ents[i];
                });
                phase("    buckets filled");
                parallel_for(nthr, [&](size_t k) { std::sort(sorted.begin() + (i64)count[k], sorted.begin() + (i64)count[k + 1], less); });
                ents.swap(sorted);
            } else {
                std::sort(ents.begin(), ents.end(), less);
            }
            phase("  dictionary sort");
            // rank of every occupied slot: the (few) slots travel in rank order and a kernel scatters their ranks
            std::vector<u64> slot_of_rank(ents.size());
            col.dict.resize(ents.size());
            parallel_for(nthr, [&](size_t t) {
                for (size_t r = ents.size() * t / nthr; r < ents.size() * (t + 1) / nthr; ++r) {
                    slot_of_rank[r] = ents[r].slot;
                    col.dict[r].assign(cb + ents[r].at, ents[r].len);
                }
            });
            phase("    dictionary strings");
            d_rank.ensure((size_t)cap * 4);
            d_oslots.ensure(std::max<size_t>(slot_of_rank.size() * 8, 64));
            if (!slot_of_rank.empty()) CK(cudaMemcpyAsync(d_oslots.p, slot_of_rank.data(), slot_of_rank.size() * 8, cudaMemcpyHostToDevice, s));
            launch_dict_ranks(d_oslots.as<u64>(), (u64)slot_of_rank.size(), d_rank.as<u32>(), s);
            u32* out32 = nullptr;
            if (col.width == 4) {
                col.d_payload = device_rows(4, 0, s);
                out32 = col.d_payload.as<u32>();
            }
            launch_dict_remap(col.d_tags.as<u8>(), d_slots.as<i64>(), pay8[c].as<i64>(), out32, ndocs, d_rank.as<u32>(), s);
            CK(cudaStreamSynchronize(s));
            phase("  dictionary remap");
        }
        if (col.width == 8) col.d_payload = std::move(pay8[c]);
        else { pay8[c].release(); if (col.width == 0) col.d_payload = device_rows(0, 0, s); }
        st.set_dictionary(col.dict);
        if (!col.stats_forced) col.stats = st;
        col.dict_staged = false;
    }
    phase("dictionaries");
    filled = Fill::DEVICE_DOCS;
    json_bytes += nbytes;
    shred_sec += now_sec() - t0;
}

void Table::splice(const Table& old, const Table* patch, const std::vector<SpliceRun>& runs) {
    if (!have_device()) N1_THROW(N1GPU_E_CUDA, "splicing columns needs a CUDA device");
    admit(Entry::SPLICE);
    if (old.cols.size() != cols.size() || (patch && patch->cols.size() != cols.size())) N1_THROW(N1GPU_E_INVALID, "splice sources have other columns");
    const double t0 = now_sec();
    const size_t R = runs.size();
    std::vector<i64> h_runs(2 * R + 1);  // new_lo[0..R], then src_lo[0..R)
    for (size_t k = 0; k < R; ++k) {
        const SpliceRun& r = runs[k];
        const Table* src = r.patch ? patch : &old;
        if (!src || r.len <= 0 || r.src_lo < 0 || r.src_lo + r.len > src->nrows || r.new_lo != (k ? h_runs[k - 1] + runs[k - 1].len : 0))
            N1_THROW(N1GPU_E_INVALID, "splice run %zu does not follow its sources", k);
        h_runs[k] = r.new_lo;
        h_runs[R + 1 + k] = (i64)((u64)r.src_lo | (r.patch ? 0x8000000000000000ULL : 0));
    }
    nrows = R ? runs.back().new_lo + runs.back().len : 0;
    h_runs[R] = nrows;
    const i64 pad = std::max(padded_rows(), ROW_PAD);
    cudaStream_t s = nullptr;
    CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    struct StreamGuard { cudaStream_t s; ~StreamGuard() { cudaStreamDestroy(s); } } sg{s};
    DevBuf d_runs, d_used, d_oremap, d_premap;
    d_runs.alloc(h_runs.size() * 8);
    CK(cudaMemcpyAsync(d_runs.p, h_runs.data(), h_runs.size() * 8, cudaMemcpyHostToDevice, s));
    const SpliceRuns sr{d_runs.as<i64>(), d_runs.as<i64>() + R + 1, (i64)R, nrows};
    auto pay8 = [](const Column& c) { return c.width == 8 ? c.d_payload.as<i64>() : nullptr; };
    auto pay4 = [](const Column& c) { return c.width == 4 ? c.d_payload.as<u32>() : nullptr; };
    for (size_t c = 0; c < cols.size(); ++c) {
        const Column& oc = old.cols[c];
        const Column* pc = patch ? &patch->cols[c] : nullptr;
        Column& col = cols[c];
        // the old ranks the kept rows still use, and the classes of those rows
        const size_t words = (oc.dict.size() + 31) / 32, mask_at = (words * 4 + 7) / 8 * 8;  // bitmap, then the class mask
        d_used.ensure(mask_at + 8);
        CK(cudaMemsetAsync(d_used.p, 0, mask_at + 8, s));
        u64* d_mask = (u64*)((char*)d_used.p + mask_at);
        launch_splice_used(sr, oc.d_tags.as<u8>(), pay8(oc), pay4(oc), d_used.as<u32>(), d_mask, s);
        std::vector<u32> used(words);
        u64 mask = 0;
        if (words) CK(cudaMemcpyAsync(used.data(), d_used.p, words * 4, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(&mask, d_mask, 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        if (pc) mask |= pc->stats.class_mask;
        // new dictionary: the used old strings and the patch's, sorted and unique; both inputs are sorted, so one merge walk
        // gives the new rank of every old and every patch rank
        const std::vector<std::string>& od = oc.dict.vec();
        static const std::vector<std::string> none;
        const std::vector<std::string>& pd = pc ? pc->dict.vec() : none;
        std::vector<u32> oremap(od.size(), 0), premap(pd.size(), 0);
        std::vector<std::string> dict;
        dict.reserve(pd.size() + od.size());
        size_t i = 0, j = 0;
        auto next_used = [&](size_t from) { while (from < od.size() && !((used[from >> 5] >> (from & 31)) & 1u)) ++from; return from; };
        i = next_used(0);
        while (i < od.size() || j < pd.size()) {
            const bool take_old = j == pd.size() || (i < od.size() && od[i] <= pd[j]);
            const bool take_patch = i == od.size() || (j < pd.size() && pd[j] <= od[i]);
            const u32 rank = (u32)dict.size();
            dict.push_back(take_old ? od[i] : pd[j]);
            if (take_old) { oremap[i] = rank; i = next_used(i + 1); }
            if (take_patch) premap[j++] = rank;
        }
        col.dict = std::move(dict);
        col.width = width_of((u32)mask);
        d_oremap.ensure(std::max<size_t>(oremap.size() * 4, 64));
        d_premap.ensure(std::max<size_t>(premap.size() * 4, 64));
        if (!oremap.empty()) CK(cudaMemcpyAsync(d_oremap.p, oremap.data(), oremap.size() * 4, cudaMemcpyHostToDevice, s));
        if (!premap.empty()) CK(cudaMemcpyAsync(d_premap.p, premap.data(), premap.size() * 4, cudaMemcpyHostToDevice, s));
        col.d_tags = device_rows(1, C_MISSING, s);
        col.d_payload = device_rows(col.width, 0, s);
        launch_splice_gather(sr, pad, oc.d_tags.as<u8>(), pay8(oc), pay4(oc), d_oremap.as<u32>(), pc ? pc->d_tags.as<u8>() : nullptr,
                             pc ? pay8(*pc) : nullptr, pc ? pay4(*pc) : nullptr, d_premap.as<u32>(), col.d_tags.as<u8>(), pay8(col), pay4(col), s);
        col.dict_staged = false;
    }
    // statistics of the spliced columns, as the device shredder computes them
    std::vector<DevColumn> dc;
    for (auto& col : cols) dc.push_back(DevColumn{col.d_tags.as<u8>(), pay8(col), nrows});
    std::vector<ColumnStats> stats = device_stats(dc, s);
    for (size_t c = 0; c < cols.size(); ++c) {
        cols[c].stats = stats[c];
        cols[c].stats.set_dictionary(cols[c].dict);
    }
    filled = Fill::DEVICE_DOCS;
    sealed = true;
    splice_sec += now_sec() - t0;
}

void Table::remap_ranks_device(int ci, const std::vector<u32>& remap) {
    Column& c = cols[(size_t)ci];
    DevBuf d_map;
    d_map.alloc(std::max<size_t>(remap.size() * 4, 64));
    CK(cudaMemcpy(d_map.p, remap.data(), remap.size() * 4, cudaMemcpyHostToDevice));
    launch_rank_remap(c.d_tags.as<u8>(), c.width == 8 ? c.d_payload.as<i64>() : nullptr, c.width == 4 ? c.d_payload.as<u32>() : nullptr, nrows,
                      d_map.as<u32>(), (u32)remap.size(), nullptr);
    CK(cudaDeviceSynchronize());
}

void Table::set_column_device(int c, int width, const void* dev_payload, const u8* dev_tags, i64 n, const char* blob,
                              const i64* offs, i64 ndict) {
    if (!have_device()) N1_THROW(N1GPU_E_CUDA, "no CUDA device: device columns need one");
    admit(Entry::SET_COLUMN_DEVICE, c);
    check_column_args(c, width, n);
    for (auto& other : cols)
        if (&other != &cols[c] && other.on_device && nrows != n)
            N1_THROW(N1GPU_E_INVALID, "column lengths differ (%lld vs %lld)", (long long)nrows, (long long)n);
    std::vector<std::string> dict;
    if (blob && offs) dict = read_dictionary(blob, offs, ndict, "dictionary");
    Column& col = cols[c];
    nrows = n;
    col.d_tags = device_rows(1, C_MISSING, nullptr);
    if (n) {
        if (dev_tags) CK(cudaMemcpy(col.d_tags.p, dev_tags, (size_t)n, cudaMemcpyDeviceToDevice));
        else CK(cudaMemset(col.d_tags.p, width == 8 ? C_INT : C_STRING, (size_t)n));
    }
    col.d_payload = device_rows(width, 0, nullptr);
    if (n) CK(cudaMemcpy(col.d_payload.p, dev_payload, (size_t)n * width, cudaMemcpyDeviceToDevice));
    col.dict = std::move(dict);
    col.dict_staged = false;
    // canonical numbers + statistics, on the device
    if (width == 8) launch_canon_floats(col.d_tags.as<u8>(), col.d_payload.as<i64>(), n, nullptr);
    // a 4-byte column holds string ranks only: the kernel reads payload words of INT rows, of which there are none
    ColumnStats st = device_stats({DevColumn{col.d_tags.as<u8>(), width == 8 ? col.d_payload.as<i64>() : nullptr, n}}, nullptr)[0];
    if (st.class_mask >> (C_OTHER + 1)) N1_THROW(N1GPU_E_INVALID, "bad class byte in column %d", c);
    if (width == 4 && (st.class_mask & M_NUM)) N1_THROW(N1GPU_E_INVALID, "a 4-byte column cannot hold numbers");
    if (width == 8 && !(st.class_mask & M_NUM) && (st.class_mask & bit(C_STRING)))
        N1_THROW(N1GPU_E_INVALID, "a column of strings only must be passed as 4-byte ranks");
    st.set_dictionary(col.dict);
    if (!col.stats_forced) col.stats = st;
    col.width = width_of(col.stats.class_mask);
    if (col.width == 0) col.d_payload = device_rows(0, 0, nullptr);
    col.on_device = true;
    filled = Fill::DEVICE_COLUMNS;  // nothing left to do at seal
}

}  // namespace n1
