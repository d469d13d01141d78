// segment.cpp — persistent columnar segments and the packed document source (SURVEY.md 8f row 3).
//
// The reference's file datastore keeps one JSON file per document (datastore/file/file.go:312-353,711-749): a scan
// opens, reads and validates every file, every time.  A segment is the shredded form of a keyspace for one set of
// field paths - typed columns, class bytes, sorted dictionaries - written once next to (never inside: every plain file
// of a keyspace directory is a document, file.go:715-729) the datastore and loaded instead of parsing while the
// keyspace has not changed.  What "not changed" means is the caller's business: a segment carries an opaque source
// tag (the operator uses directory mtime + file count + newest file mtime + total bytes, see execution.cpp) and only
// loads under the very same tag - the counterpart of the invalidation on performOp / Delete (file.go:375-471).
//
// Layout (little endian): "N1SEG02\n" | u64 header bytes | header JSON | per column: dictionary offsets i64[ndict+1],
// dictionary bytes, payload (nrows x width bytes: int64 / float64 bits, or u32 ranks), class bytes (nrows) | u64 FNV-1a
// checksum of everything after the magic.  A loader checks every size the header claims against the file size before
// it allocates, the checksum, and that dictionaries are strictly increasing (string constants are binary-searched).
#include <sys/stat.h>

#include <cstdio>
#include <cstring>
#include <fstream>

#include "json.hpp"
#include <cstdint>
#include <fcntl.h>
#include <unistd.h>
#include "table.hpp"

namespace n1 {

namespace {
const char MAGIC[8] = {'N', '1', 'S', 'E', 'G', '0', '2', '\n'};

// FNV-1a over 8-byte words (the tail bytewise): a corruption check, not a cryptographic one, at memory speed
struct Sum {
    u64 h = 0xcbf29ce484222325ULL;
    unsigned char pend[8];
    int np = 0;  // bytes waiting for a full word: the sum must not depend on how the stream is cut into calls
    void word(const unsigned char* b) { u64 w; memcpy(&w, b, 8); h = (h ^ w) * 0x100000001b3ULL; }
    void add(const void* p, size_t n) {
        const unsigned char* b = (const unsigned char*)p;
        size_t i = 0;
        while (np && i < n) { pend[np++] = b[i++]; if (np == 8) { word(pend); np = 0; } }
        for (; i + 8 <= n; i += 8) word(b + i);
        for (; i < n; ++i) pend[np++] = b[i];
    }
    u64 done() const { u64 r = h; for (int i = 0; i < np; ++i) r = (r ^ pend[i]) * 0x100000001b3ULL; return r; }
};
struct Writer {
    std::ofstream& f; Sum sum;
    void put(const void* p, size_t n) { f.write((const char*)p, (std::streamsize)n); sum.add(p, n); }
};
struct Reader {
    std::ifstream& f; Sum sum; u64 left;  // bytes of the file not yet consumed
    bool get(void* p, size_t n) {
        if (n > left) return false;
        f.read((char*)p, (std::streamsize)n);
        if ((size_t)f.gcount() != n) return false;
        left -= n; sum.add(p, n);
        return true;
    }
    bool room(u64 n) const { return n <= left; }  // asked BEFORE allocating what a header field claims
};
}  // namespace

// Called by seal() once dictionaries are sorted and payloads hold ranks, before the host staging is dropped, or on a sealed
// table whose columns live in HBM.
void Table::write_segment(const std::string& segment_out, const std::string& segment_source) const {
    const std::string tmp = segment_out + ".tmp";
    std::ofstream f(tmp, std::ios::binary | std::ios::trunc);
    if (!f) N1_THROW(N1GPU_E_IO, "cannot write segment %s", tmp.c_str());
    std::string h = "{\"version\":2,\"nrows\":" + std::to_string(nrows) + ",\"source\":";
    json::quote(segment_source, h);
    h += ",\"columns\":[";
    for (size_t c = 0; c < cols.size(); ++c) {
        const Column& col = cols[c];
        size_t dict_bytes = 0;
        for (auto& s : col.dict) dict_bytes += s.size();
        if (c) h += ",";
        h += "{\"path\":";
        json::quote(join_path(col.path, '\x1f'), h);
        h += ",\"width\":" + std::to_string(col.width) + ",\"ndict\":" + std::to_string(col.dict.size()) + ",\"dict_bytes\":" + std::to_string(dict_bytes) + "}";
    }
    h += "]}";
    const u64 hl = h.size();
    f.write(MAGIC, 8);
    Writer w{f, {}};
    auto put = [&](std::ofstream&, const void* p, size_t n) { w.put(p, n); };
    put(f, &hl, 8);
    put(f, h.data(), h.size());
    // seal() writes from the host staging; a sealed table (a refreshed one) holds its columns in HBM only: they are copied
    // back column by column
    const bool device = sealed;
    if (device && !have_device()) N1_THROW(N1GPU_E_INVALID, "a sealed table without a device has no columns to write");
    std::vector<u8> dtags;
    std::vector<char> dpay;
    for (auto& col : cols) {
        std::vector<i64> offs(col.dict.size() + 1, 0);
        for (size_t i = 0; i < col.dict.size(); ++i) offs[i + 1] = offs[i] + (i64)col.dict[i].size();
        put(f, offs.data(), offs.size() * 8);
        for (auto& s : col.dict) put(f, s.data(), s.size());
        if (device) {
            dtags.resize((size_t)nrows);
            dpay.resize((size_t)nrows * (size_t)col.width);
            if (nrows) {
                CK(cudaMemcpyAsync(dtags.data(), col.d_tags.p, (size_t)nrows, cudaMemcpyDeviceToHost, nullptr));
                if (col.width) CK(cudaMemcpyAsync(dpay.data(), col.d_payload.p, dpay.size(), cudaMemcpyDeviceToHost, nullptr));
                CK(cudaStreamSynchronize(nullptr));
            }
            put(f, dpay.data(), dpay.size());
            put(f, dtags.data(), dtags.size());
            continue;
        }
        if (col.width == 8) put(f, col.payload.data(), (size_t)nrows * 8);
        else if (col.width == 4) {
            std::vector<u32> narrow((size_t)nrows);
            for (i64 i = 0; i < nrows; ++i) narrow[(size_t)i] = (u32)col.payload[(size_t)i];
            put(f, narrow.data(), narrow.size() * 4);
        }
        put(f, col.tags.data(), (size_t)nrows);
    }
    const u64 total = w.sum.done();
    f.write((const char*)&total, 8);
    f.close();
    if (!f || rename(tmp.c_str(), segment_out.c_str()) != 0) { remove(tmp.c_str()); N1_THROW(N1GPU_E_IO, "cannot write segment %s", segment_out.c_str()); }
}

// Fills the (unsealed, empty) table from a segment written for the same columns under the same source tag.
// Returns false - and leaves the table untouched - when the file is absent, foreign, truncated or stale.
// a refused segment is not an error (the caller shreds the documents instead); N1GPU_TRACE says which check refused it
#define REFUSE(check) do { if (getenv("N1GPU_TRACE")) fprintf(stderr, "[n1gpu segment] %s not loaded (check %d)\n", file.c_str(), check); return false; } while (0)
bool Table::load_segment(const std::string& file, const std::string& source) {
    admit(Entry::LOAD_SEGMENT);
    std::ifstream f(file, std::ios::binary);
    if (!f) REFUSE(3);
    f.seekg(0, std::ios::end);
    const std::streamoff fsize = f.tellg();
    f.seekg(0, std::ios::beg);
    if (fsize < 24) REFUSE(7);
    char magic[8];
    u64 hl = 0;
    f.read(magic, 8);
    if ((size_t)f.gcount() != 8 || memcmp(magic, MAGIC, 8) != 0) REFUSE(11);
    Reader rd{f, {}, (u64)fsize - 8 - 8};  // the trailing checksum is not payload
    auto get = [&](std::ifstream&, void* p, size_t n) { return rd.get(p, n); };
    if (!get(f, &hl, 8) || hl > (64u << 20) || !rd.room(hl)) REFUSE(14);
    std::string h((size_t)hl, '\0');
    if (!get(f, &h[0], h.size())) REFUSE(16);
    json::Node root;
    if (!json::parse(h, root) || root.kind != json::Node::OBJ) REFUSE(18);
    const json::Node* ver = root.get("version");
    const json::Node* nr = root.get("nrows");
    const json::Node* cs = root.get("columns");
    if (!ver || ver->kind != json::Node::INT || ver->i != 2 || !nr || nr->kind != json::Node::INT || nr->i < 0) REFUSE(22);
    if (root.str_or("source", "\x01") != source) REFUSE(23);  // the keyspace changed since the segment was written
    if (!cs || cs->kind != json::Node::ARR || cs->arr.size() != cols.size()) REFUSE(24);
    const i64 n = nr->i;
    struct Staged { std::vector<std::string> dict; std::vector<i64> payload; std::vector<u8> tags; };
    std::vector<Staged> staged(cols.size());
    for (size_t c = 0; c < cols.size(); ++c) {
        const json::Node& cn = cs->arr[c];
        if (cn.kind != json::Node::OBJ || cn.str_or("path", "\x01") != join_path(cols[c].path, '\x1f')) REFUSE(30);
        const json::Node *w = cn.get("width"), *nd = cn.get("ndict"), *db = cn.get("dict_bytes");
        if (!w || !nd || !db || w->kind != json::Node::INT || nd->kind != json::Node::INT || db->kind != json::Node::INT) REFUSE(32);
        if ((w->i != 8 && w->i != 4 && w->i != 0) || nd->i < 0 || db->i < 0) REFUSE(33);
        Staged& st = staged[c];
        // sizes the header claims, against what the file still holds - before anything is allocated for them
        if (!rd.room(((u64)nd->i + 1) * 8) || !rd.room((u64)db->i) || !rd.room((u64)n * (u64)(w->i + 1))) REFUSE(36);
        std::vector<i64> offs((size_t)nd->i + 1);
        if (!get(f, offs.data(), offs.size() * 8) || offs[0] != 0 || offs.back() != db->i) REFUSE(38);
        std::string blob((size_t)db->i, '\0');
        if (db->i && !get(f, &blob[0], blob.size())) REFUSE(40);
        st.dict.reserve((size_t)nd->i);
        for (i64 i = 0; i < nd->i; ++i) {
            if (offs[(size_t)i + 1] < offs[(size_t)i] || offs[(size_t)i + 1] > db->i) REFUSE(43);
            st.dict.emplace_back(blob.data() + offs[(size_t)i], (size_t)(offs[(size_t)i + 1] - offs[(size_t)i]));
            if (i && !(st.dict[(size_t)i - 1] < st.dict[(size_t)i])) REFUSE(45);  // sorted bytewise, unique
        }
        st.payload.assign((size_t)n, 0);
        if (w->i == 8) { if (n && !get(f, st.payload.data(), (size_t)n * 8)) REFUSE(48); }
        else if (w->i == 4) {
            std::vector<u32> narrow((size_t)n);
            if (n && !get(f, narrow.data(), narrow.size() * 4)) REFUSE(51);
            for (i64 i = 0; i < n; ++i) st.payload[(size_t)i] = narrow[(size_t)i];
        }
        st.tags.resize((size_t)n);
        if (n && !get(f, st.tags.data(), (size_t)n)) REFUSE(55);
        for (i64 i = 0; i < n; ++i) {
            const u8 t = st.tags[(size_t)i];
            if (t > C_OTHER || (t == C_STRING && (u64)st.payload[(size_t)i] >= (u64)nd->i)) REFUSE(58);
        }
    }
    u64 total = 0;
    f.read((char*)&total, 8);
    if ((size_t)f.gcount() != 8 || rd.left != 0 || total != rd.sum.done()) REFUSE(63);
    for (size_t c = 0; c < cols.size(); ++c) {
        Column& col = cols[c];
        col.dict = std::move(staged[c].dict);
        col.payload = std::move(staged[c].payload);
        col.tags = std::move(staged[c].tags);
        col.local_strings.clear();
        col.dict_staged = false;
    }
    nrows = n;
    filled = Fill::HOST_DOCS;  // like appended documents: no further input may be mixed in
    return true;
}

#undef REFUSE

// A packed document source: one JSON document per line (NDJSON), in primary-key order - the form a keyspace of more
// than a few million documents takes when one file per document (file.go) stops being practical.
void Table::load_ndjson(const std::string& file, int threads) {
    const int fd = open(file.c_str(), O_RDONLY | O_CLOEXEC);
    if (fd < 0) N1_THROW(N1GPU_E_IO, "cannot read %s", file.c_str());
    struct FdGuard { int fd; ~FdGuard() { close(fd); } } fg{fd};
    struct stat st;
    size_t size = 0;
    if (fstat(fd, &st) == 0 && S_ISREG(st.st_mode)) size = (size_t)st.st_size;
    // The text goes straight into pinned memory when the device shredder will take it (the H2D copy then runs at PCIe
    // speed without a staging copy), read and scanned for line starts by all cores: a keyspace of 10^7 documents is
    // hundreds of megabytes, and one core reads and scans ~8 GB/s.
    const bool device = threads < 0;
    const bool trace = getenv("N1GPU_TRACE") != nullptr;
    double tp = now_sec();
    auto phase = [&](const char* name) { if (trace) { double t = now_sec(); fprintf(stderr, "[n1gpu ndjson] %-22s %8.3f ms\n", name, (t - tp) * 1e3); tp = t; } };
    PinnedBuf pin;
    std::string heap;
    char* data = nullptr;
    if (device && have_device()) { pin.ensure(size + 64); data = pin.as<char>(); }
    else { heap.resize(size + 64); data = &heap[0]; }
    int nthr = (int)std::min<size_t>(std::max(1u, std::thread::hardware_concurrency()), 16);
    if ((size_t)nthr > size / ((size_t)4 << 20) + 1) nthr = (int)(size / ((size_t)4 << 20) + 1);
    auto slice = [&](int t) { return size * (size_t)t / (size_t)nthr; };
    // bytes [lo, hi) of the file, read by all threads at once
    auto read_range = [&](size_t lo, size_t hi) {
        const size_t span = hi - lo;
        parallel_for(nthr, [&](int t) {
            size_t at = lo + span * (size_t)t / (size_t)nthr;
            const size_t end = lo + span * (size_t)(t + 1) / (size_t)nthr;
            while (at < end) {
                const ssize_t got = pread(fd, data + at, end - at, (off_t)at);
                if (got <= 0) N1_THROW(N1GPU_E_IO, "short read of %s", file.c_str());
                at += (size_t)got;
            }
        });
    };
    if (device && have_device()) {
        // the device finds the line starts itself (shred.cu k_ndjson_lines); the file is read chunk by chunk while the chunks
        // before it cross PCIe
        append_ndjson_device(data, (i64)size, [&](i64 lo, i64 hi) { read_range((size_t)lo, (size_t)hi); });
        phase("read + shred");
        return;
    }
    read_range(0, size);
    phase("alloc + parallel read");
    // document i = [start of its line, start of the next non-blank line): the line end and blank lines are trailing white
    // space of the document before them (value/parsed.go:76-98 skips leading ' ', '\t', '\n'; JSON allows trailing space)
    auto blank = [](char c) { return c == ' ' || c == '\t' || c == '\r'; };
    // Two passes over the text, both store-free on the way (a growing vector per thread spends more time faulting fresh pages
    // in than the scan itself): pass 1 counts the documents of every slice, pass 2 writes their line starts at their final
    // positions - in pinned memory when the offsets cross PCIe with the text.
    auto scan = [&](int t, auto&& emit) {
        const size_t lo = slice(t), hi = slice(t + 1);
        auto consider = [&](size_t s0) {  // a line that begins at s0: a document unless it is blank
            size_t a = s0;
            while (a < size && blank(data[a])) ++a;
            if (a < size && data[a] != '\n') emit((i64)s0);
        };
        if (t == 0 && size) consider(0);
        size_t i = lo;
        // eight bytes at a time: a zero byte of (word ^ 0x0a..0a) is a line end (the classic has-zero-byte test)
        while (i < hi && (reinterpret_cast<uintptr_t>(data + i) & 7)) { if (data[i] == '\n' && i + 1 < size) consider(i + 1); ++i; }
        for (; i + 8 <= hi; i += 8) {
            u64 w;
            memcpy(&w, data + i, 8);
            const u64 x = w ^ 0x0a0a0a0a0a0a0a0aULL;
            u64 z = (x - 0x0101010101010101ULL) & ~x & 0x8080808080808080ULL;
            while (z) {
                const size_t e = i + (size_t)(__builtin_ctzll(z) >> 3);
                // (the borrow of the subtraction can flag the byte above a real line end: check it)
                if (data[e] == '\n' && e + 1 < size) {
                    if (data[e + 1] == '{') emit((i64)(e + 1)); else consider(e + 1);
                }
                z &= z - 1;
            }
        }
        for (; i < hi; ++i) if (data[i] == '\n' && i + 1 < size) consider(i + 1);
    };
    std::vector<size_t> run_at((size_t)nthr + 1, 0);
    parallel_for(nthr, [&](int t) { size_t n = 0; scan(t, [&](i64) { ++n; }); run_at[(size_t)t + 1] = n; });
    for (int t = 0; t < nthr; ++t) run_at[(size_t)t + 1] += run_at[(size_t)t];
    const size_t ndocs = run_at[(size_t)nthr];
    phase("count documents");
    PinnedBuf pin_offs;
    std::vector<i64> heap_offs;
    i64* offsets = nullptr;
    if (device && have_device()) { pin_offs.ensure((ndocs + 1) * 8 + 64); offsets = pin_offs.as<i64>(); }
    else { heap_offs.resize(ndocs + 1); offsets = heap_offs.data(); }
    parallel_for(nthr, [&](int t) { i64* out = offsets + run_at[(size_t)t]; scan(t, [&](i64 s0) { *out++ = s0; }); });
    offsets[ndocs] = (i64)size;
    if (ndocs == 0) offsets[0] = 0;
    phase("offsets");
    if (device) append_json_device(data, offsets, (i64)ndocs);
    else append_json(data, offsets, (i64)ndocs, threads);
    phase("shred");
}

}  // namespace n1
