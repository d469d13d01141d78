// table.cpp — the columnar shredder (replaces PrimaryScan + Fetch over datastore/file) and the HBM
// column store.
//
// Reference behaviour restated (file:line under /root/reference):
//   datastore/file/file.go:711-730  ScanEntries = sorted ReadDir, every non-directory entry is a document
//   datastore/file/file.go:732-749  fetch = ReadFile + value.NewValue(bytes); key = name minus extension
//   value/parsed.go:38-98           type sniff skips ' ', '\t', '\n'; invalid JSON -> BINARY (all fields MISSING)
//   value/parsed.go:159-207         Field(): first occurrence of the name; non-object -> MISSING
//   value/value.go:367-430          NewValue: integral float64 -> int64
#include "table.hpp"

#include <dirent.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cerrno>
#include <chrono>
#include <fstream>
#include <string_view>
#include <thread>

#include "json.hpp"

namespace n1 {

double now_sec() {
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

std::vector<std::string> split_path(const std::string& path) {
    std::vector<std::string> out;
    size_t s = 0;
    for (;;) {
        size_t e = path.find('\x1f', s);
        if (e == std::string::npos) { out.push_back(path.substr(s)); break; }
        out.push_back(path.substr(s, e - s));
        s = e + 1;
    }
    return out;
}
std::string join_path(const std::vector<std::string>& p, char sep) {
    std::string s;
    for (size_t i = 0; i < p.size(); ++i) { if (i) s.push_back(sep); s += p[i]; }
    return s;
}

// The one place that decides which entry point may follow which: rows come in by one route (Fill), documents and segments
// in full, columns one by one.
void Table::admit(Entry e, int col) const {
    const bool docs = filled == Fill::HOST_DOCS || filled == Fill::DEVICE_DOCS;  // documents, a segment or a splice: the rows are in
    auto refuse = [](const char* why) { N1_THROW(N1GPU_E_INVALID, "%s", why); };
    if (e == Entry::ADD_COLUMN) { if (sealed || docs) refuse("columns must be declared before documents are appended"); return; }
    if (e == Entry::LOAD_SEGMENT) { if (sealed || docs || nrows) refuse("a segment loads into an empty, unsealed table"); return; }
    if (e == Entry::SPLICE) { if (sealed || docs || nrows) refuse("a splice fills an empty, unsealed table"); return; }
    if (sealed) refuse("table is sealed");
    if (e == Entry::APPEND_HOST) {
        if (rows_in_hbm()) refuse("table already holds device-shredded rows");
        for (auto& c : cols)
            if (!c.dict_staged) refuse("append after dictionary import / pre-shredded columns is not supported");
    } else if (e == Entry::APPEND_DEVICE) {
        if (!have_device()) N1_THROW(N1GPU_E_CUDA, "the device shredder needs a CUDA device (there is no CPU fallback for it; use host threads explicitly)");
        if (docs || nrows) refuse("the device shredder takes the whole keyspace in one append");
    } else {  // SET_COLUMN, SET_COLUMN_DEVICE (of column `col`)
        if (docs) refuse("cannot mix appended documents and pre-shredded columns");
        for (size_t c = 0; c < cols.size(); ++c)
            if (e == Entry::SET_COLUMN ? filled == Fill::DEVICE_COLUMNS : c != (size_t)col && !cols[c].tags.empty())
                refuse("cannot mix host and device columns in one table");
    }
}

int Table::add_column(const std::string& path) {
    admit(Entry::ADD_COLUMN);
    int f = find_column(path);
    if (f >= 0) return f;
    if (cols.size() >= 16) N1_THROW(N1GPU_E_INELIGIBLE, "more than 16 referenced columns");
    cols.emplace_back();
    cols.back().path = split_path(path);
    return (int)cols.size() - 1;
}
int Table::find_column(const std::string& path) const {
    auto p = split_path(path);
    for (size_t i = 0; i < cols.size(); ++i) if (cols[i].path == p) return (int)i;
    return -1;
}

// ---- path trie -----------------------------------------------------------------------------------
namespace {
struct Trie {
    struct Node { std::vector<std::pair<std::string, int>> kids; int col = -1; };
    std::vector<Node> nodes;
    Trie() { nodes.emplace_back(); }
    void add(const std::vector<std::string>& path, int col) {
        int n = 0;
        for (auto& name : path) {
            int next = -1;
            for (auto& k : nodes[n].kids) if (k.first == name) next = k.second;
            if (next < 0) { nodes.emplace_back(); next = (int)nodes.size() - 1; nodes[n].kids.emplace_back(name, next); }
            n = next;
        }
        nodes[n].col = col;
    }
    int child(int n, const char* b, const char* e) const {
        size_t len = (size_t)(e - b);
        for (auto& k : nodes[n].kids) if (k.first.size() == len && memcmp(k.first.data(), b, len) == 0) return k.second;
        return -1;
    }
};

struct ChunkCol {
    std::vector<i64> payload;
    std::vector<u8> tags;
    std::unordered_map<std::string, u32> index;
    std::vector<std::string> strings;
    u32 code(const std::string& s) {
        auto it = index.find(s);
        if (it != index.end()) return it->second;
        u32 c = (u32)strings.size();
        index.emplace(s, c);
        strings.push_back(s);
        return c;
    }
};

struct Shredder {
    const Trie& trie;
    std::vector<ChunkCol>& cols;
    i64 row = 0;
    std::string tmp;
    Shredder(const Trie& t, std::vector<ChunkCol>& c) : trie(t), cols(c) {}

    void put(int col, u8 tag, i64 payload) {
        if (cols[col].tags[row] != C_MISSING) return;  // first occurrence wins (FirstFind)
        cols[col].tags[row] = tag;
        cols[col].payload[row] = payload;
    }

    // value at trie node `n` (n has a column and/or children)
    bool value(json::Scanner& sc, int n) {
        sc.ws();
        if (sc.p >= sc.end) return sc.fail();
        const Trie::Node& node = trie.nodes[n];
        char c = *sc.p;
        if (c == '{') {
            if (node.col >= 0) put(node.col, C_OTHER, 0);
            if (node.kids.empty()) return sc.skip();
            return object(sc, n);
        }
        if (c == '[') {
            if (node.col >= 0) put(node.col, C_OTHER, 0);
            return sc.skip();
        }
        if (node.col < 0) return sc.skip();
        if (c == '"') {
            const char *rb, *re; bool esc;
            if (!sc.string_raw(rb, re, esc)) return false;
            if (cols[node.col].tags[row] == C_MISSING) {
                if (esc) json::Scanner::unescape(rb, re, tmp); else tmp.assign(rb, re);
                put(node.col, C_STRING, (i64)cols[node.col].code(tmp));
            }
            return true;
        }
        if (c == 't') { if (!sc.literal("true")) return false; put(node.col, C_TRUE, 0); return true; }
        if (c == 'f') { if (!sc.literal("false")) return false; put(node.col, C_FALSE, 0); return true; }
        if (c == 'n') { if (!sc.literal("null")) return false; put(node.col, C_NULL, 0); return true; }
        bool ii; i64 iv; double dv;
        if (!sc.number(ii, iv, dv)) return false;
        if (ii) put(node.col, C_INT, iv);
        else if (f_is_int(dv)) put(node.col, C_INT, go_i64(dv));  // NewValue canonicalisation
        else { i64 b; memcpy(&b, &dv, 8); put(node.col, C_FLOAT, b); }
        return true;
    }

    bool object(json::Scanner& sc, int n) {
        ++sc.p;  // '{'
        sc.ws();
        if (sc.p < sc.end && *sc.p == '}') { ++sc.p; return true; }
        for (;;) {
            sc.ws();
            const char *rb, *re; bool esc;
            if (!sc.string_raw(rb, re, esc)) return false;
            int kid;
            if (esc) { json::Scanner::unescape(rb, re, tmp); kid = trie.child(n, tmp.data(), tmp.data() + tmp.size()); }
            else kid = trie.child(n, rb, re);
            sc.ws();
            if (sc.p >= sc.end || *sc.p != ':') return sc.fail();
            ++sc.p;
            if (kid >= 0) { if (!value(sc, kid)) return false; }
            else if (!sc.skip()) return false;
            sc.ws();
            if (sc.p < sc.end && *sc.p == ',') { ++sc.p; continue; }
            if (sc.p < sc.end && *sc.p == '}') { ++sc.p; return true; }
            return sc.fail();
        }
    }

    void document(const char* b, const char* e) {
        const char* s = b;
        while (s < e && (*s == ' ' || *s == '\t' || *s == '\n')) ++s;  // identifyType, parsed.go:76-98
        bool valid = false;
        if (s < e && *s == '{') {
            json::Scanner sc(s, e);
            if (object(sc, 0)) { sc.ws(); valid = sc.p == sc.end; }
        }
        if (!valid)  // non-object or BINARY document: every field access is MISSING
            for (auto& c : cols) { c.tags[row] = C_MISSING; c.payload[row] = 0; }
        ++row;
    }
};
}  // namespace

void host_shred_docs(const std::vector<Column>& cols, const char* buf, const i64* offs, const i64* rows, i64 n,
                     std::vector<HostShredOut>& out) {
    Trie trie;
    for (size_t c = 0; c < cols.size(); ++c) trie.add(cols[c].path, (int)c);
    std::vector<ChunkCol> cc(cols.size());
    for (auto& c : cc) { c.payload.assign((size_t)n, 0); c.tags.assign((size_t)n, C_MISSING); }
    Shredder sh(trie, cc);
    for (i64 i = 0; i < n; ++i) sh.document(buf + offs[rows[i]], buf + offs[rows[i] + 1]);
    out.resize(cols.size());
    for (size_t c = 0; c < cols.size(); ++c) {
        out[c].tags.swap(cc[c].tags);
        out[c].payload.swap(cc[c].payload);
        out[c].strings.swap(cc[c].strings);
    }
}

void Table::append_json(const char* buf, const i64* offsets, i64 ndocs, int threads) {
    if (sealed) N1_THROW(N1GPU_E_INVALID, "table is sealed");
    if (threads == -1) { append_json_device(buf, offsets, ndocs); return; }
    admit(Entry::APPEND_HOST);
    if (ndocs < 0) N1_THROW(N1GPU_E_INVALID, "negative document count");
    double t0 = now_sec();
    filled = Fill::HOST_DOCS;
    Trie trie;
    for (size_t c = 0; c < cols.size(); ++c) trie.add(cols[c].path, (int)c);
    int nthreads = threads > 0 ? threads : (int)std::thread::hardware_concurrency();
    if (nthreads < 1) nthreads = 1;
    if ((i64)nthreads > (ndocs + 4095) / 4096) nthreads = (int)std::max<i64>(1, (ndocs + 4095) / 4096);
    std::vector<std::vector<ChunkCol>> chunks(nthreads);
    parallel_for(nthreads, [&](int t) {
        i64 lo = ndocs * t / nthreads, hi = ndocs * (t + 1) / nthreads;
        auto& cc = chunks[t];
        cc.resize(cols.size());
        for (auto& c : cc) { c.payload.assign((size_t)(hi - lo), 0); c.tags.assign((size_t)(hi - lo), C_MISSING); }
        Shredder sh(trie, cc);
        for (i64 d = lo; d < hi; ++d) sh.document(buf + offsets[d], buf + offsets[d + 1]);
    });
    // merge chunk-local string codes into the column's staging dictionary (parallel over columns)
    std::vector<std::unordered_map<std::string, u32>> colindex(cols.size());
    auto merge = [&](int c) {
        Column& col = cols[c];
        auto& index = colindex[c];
        for (u32 i = 0; i < col.local_strings.size(); ++i) index.emplace(col.local_strings[i], i);
        size_t base = col.payload.size();
        col.payload.resize(base + (size_t)ndocs);
        col.tags.resize(base + (size_t)ndocs);
        size_t at = base;
        for (int t = 0; t < nthreads; ++t) {
            ChunkCol& cc = chunks[t][c];
            std::vector<u32> remap(cc.strings.size());
            for (size_t i = 0; i < cc.strings.size(); ++i) {
                auto it = index.find(cc.strings[i]);
                if (it == index.end()) {
                    u32 id = (u32)col.local_strings.size();
                    col.local_strings.push_back(cc.strings[i]);
                    index.emplace(cc.strings[i], id);
                    remap[i] = id;
                } else remap[i] = it->second;
            }
            size_t n = cc.tags.size();
            memcpy(col.tags.data() + at, cc.tags.data(), n);
            for (size_t r = 0; r < n; ++r)
                col.payload[at + r] = cc.tags[r] == C_STRING ? (i64)remap[(size_t)cc.payload[r]] : cc.payload[r];
            at += n;
        }
    };
    if (cols.size() > 1 && nthreads > 1) parallel_for((int)cols.size(), merge);
    else for (int c = 0; c < (int)cols.size(); ++c) merge(c);
    nrows += ndocs;
    json_bytes += offsets[ndocs] - offsets[0];
    shred_sec += now_sec() - t0;
}

DocFp DocFp::of(const struct stat& st) {
    DocFp f;
    f.state = DOC;
    f.ino = (u64)st.st_ino;
    f.size = (i64)st.st_size;
    f.mtime_ns = (i64)st.st_mtim.tv_sec * 1000000000 + st.st_mtim.tv_nsec;
    f.ctime_ns = (i64)st.st_ctim.tv_sec * 1000000000 + st.st_ctim.tv_nsec;
    return f;
}

void Table::load_dir(const std::string& dir, int threads, std::vector<std::string>* entries, std::vector<DocFp>* fps) {
    DIR* d = opendir(dir.c_str());
    if (!d) N1_THROW(N1GPU_E_IO, "cannot open keyspace directory %s", dir.c_str());
    std::vector<std::string> names;
    while (dirent* e = readdir(d)) {
        std::string n = e->d_name;
        if (n == "." || n == "..") continue;
        if (e->d_type == DT_DIR) continue;
        if (e->d_type != DT_REG) {  // links / file systems without d_type: ask
            struct stat st;
            if (stat((dir + "/" + n).c_str(), &st) != 0 || S_ISDIR(st.st_mode)) continue;
        }
        names.push_back(n);
    }
    closedir(d);
    std::sort(names.begin(), names.end());  // ioutil.ReadDir order
    if (entries) *entries = names;
    load_entries(dir, names, threads, fps);
}

std::string document_file(const std::string& entry) {
    // The primary index scans IDS, not files: every non-directory entry yields the id "name minus its last extension"
    // (documentPathToId, file.go:757-761), and Fetch reads <id>.json (file.go:346) - a missing file is silently no document
    // (file.go:319-322), an unreadable one is an error the request reports while it carries on.  So foo.txt is a document only
    // if foo.json exists (and a.json + a.txt are TWO rows of a.json), .DS_Store and editor backups are none.
    const size_t dot = entry.rfind('.');
    return (dot == std::string::npos ? entry : entry.substr(0, dot)) + ".json";
}

void Table::load_entries(const std::string& dir, const std::vector<std::string>& entries, int threads, std::vector<DocFp>* fps) {
    std::vector<std::string> names(entries.size());
    for (size_t i = 0; i < entries.size(); ++i) names[i] = document_file(entries[i]);
    if (fps) fps->assign(names.size(), DocFp());
    // The reference opens and reads one file per document, serially (file.go:732-743).  Here the reads of contiguous
    // ranges of the sorted names run on all cores - they are system calls on (mostly cached) small files - and the
    // documents are then laid end to end in primary-key order for the shredder.
    const size_t nfiles = names.size();
    int nthreads = (int)std::thread::hardware_concurrency();
    if (nthreads < 1) nthreads = 1;
    if ((size_t)nthreads > (nfiles + 255) / 256) nthreads = (int)std::max<size_t>(1, (nfiles + 255) / 256);
    struct Part { std::string bytes; std::vector<i64> sizes; };
    std::vector<Part> parts((size_t)nthreads);
    parallel_for(nthreads, [&](int t) {
        Part& part = parts[(size_t)t];
        const size_t lo = nfiles * (size_t)t / (size_t)nthreads, hi = nfiles * (size_t)(t + 1) / (size_t)nthreads;
        part.sizes.reserve(hi - lo);
        std::string path;
        for (size_t i = lo; i < hi; ++i) {
            path.assign(dir).append("/").append(names[i]);
            const int fd = open(path.c_str(), O_RDONLY | O_CLOEXEC);
            if (fd < 0) {  // ENOENT: the id denotes no document; anything else: the reference reports and continues
                if (fps) (*fps)[i].state = errno == ENOENT ? DocFp::ABSENT : DocFp::UNREADABLE;
                continue;
            }
            const size_t before = part.bytes.size();
            size_t cap = 4096;
            struct stat st;
            DocFp fp;
            fp.racy = true;  // no fingerprint: read again at the next check
            if (fstat(fd, &st) == 0) { fp = DocFp::of(st); if (st.st_size > 0) cap = (size_t)st.st_size + 1; }
            bool failed = false;
            for (;;) {
                part.bytes.resize(part.bytes.size() + cap);
                const ssize_t got = read(fd, &part.bytes[part.bytes.size() - cap], cap);
                if (got < 0) { part.bytes.resize(before); failed = true; break; }  // (a directory named x.json, an I/O error): no document
                part.bytes.resize(part.bytes.size() - cap + (size_t)got);
                if (got == 0) break;
            }
            close(fd);
            fp.state = failed ? DocFp::UNREADABLE : DocFp::DOC;
            if (fps) (*fps)[i] = fp;
            if (!failed) part.sizes.push_back((i64)(part.bytes.size() - before));
        }
    });
    size_t total = 0;
    for (auto& part : parts) total += part.bytes.size();
    // laid end to end - in pinned memory when the device shredder takes the text (its H2D copy then needs no staging)
    PinnedBuf pin;
    std::string heap;
    char* buf = nullptr;
    if (threads < 0 && have_device()) { pin.ensure(total + 64); buf = pin.as<char>(); }
    else { heap.resize(total + 64); buf = &heap[0]; }
    std::vector<i64> offsets;
    offsets.reserve(nfiles + 1);
    offsets.push_back(0);
    std::vector<size_t> part_at(parts.size() + 1, 0);
    for (size_t i = 0; i < parts.size(); ++i) {
        part_at[i + 1] = part_at[i] + parts[i].bytes.size();
        for (i64 sz : parts[i].sizes) offsets.push_back(offsets.back() + sz);
    }
    parallel_for((int)parts.size(), [&](int i) {
        if (!parts[i].bytes.empty()) memcpy(buf + part_at[i], parts[i].bytes.data(), parts[i].bytes.size());
        std::string().swap(parts[i].bytes);
    });
    append_json(buf, offsets.data(), (i64)offsets.size() - 1, threads);  // ids without a document were skipped
}

std::vector<std::string> read_dictionary(const char* blob, const i64* offs, i64 n, const char* what) {
    std::vector<std::string> d;
    d.reserve((size_t)std::max<i64>(n, 0));
    for (i64 i = 0; i < n; ++i) {
        d.emplace_back(blob + offs[i], blob + offs[i + 1]);
        if (i && !(d[(size_t)i - 1] < d[(size_t)i])) N1_THROW(N1GPU_E_INVALID, "%s must be sorted bytewise and unique", what);
    }
    return d;
}

void Table::check_column_args(int c, int width, i64 n) const {
    if (c < 0 || c >= (int)cols.size()) N1_THROW(N1GPU_E_INVALID, "no such column %d", c);
    if (width != 8 && width != 4) N1_THROW(N1GPU_E_INVALID, "payload width must be 8 or 4");
    if (n < 0) N1_THROW(N1GPU_E_INVALID, "negative row count");
}

void Table::set_column(int c, int width, const void* payload, const u8* tags, i64 n, const char* blob,
                       const i64* offs, i64 ndict) {
    admit(Entry::SET_COLUMN);
    check_column_args(c, width, n);
    for (auto& other : cols)
        if (&other != &cols[c] && !other.tags.empty() && (i64)other.tags.size() != n)
            N1_THROW(N1GPU_E_INVALID, "column lengths differ (%lld vs %lld)", (long long)other.tags.size(), (long long)n);
    std::vector<std::string> dict;
    if (blob && offs) dict = read_dictionary(blob, offs, ndict, "dictionary");
    Column& col = cols[c];
    col.payload.resize((size_t)n);
    col.tags.resize((size_t)n);
    if (width == 8) memcpy(col.payload.data(), payload, (size_t)n * 8);
    else for (i64 i = 0; i < n; ++i) col.payload[(size_t)i] = ((const u32*)payload)[i];
    if (tags) memcpy(col.tags.data(), tags, (size_t)n);
    else memset(col.tags.data(), width == 8 ? C_INT : C_STRING, (size_t)n);
    col.dict = std::move(dict);
    col.dict_staged = false;
    nrows = n;
    filled = Fill::HOST_COLUMNS;
}

void Table::adopt_dictionary(int ci, std::vector<std::string>& global) {
    Column& c = cols[(size_t)ci];
    std::vector<u32> remap(c.dict.size());
    size_t g = 0;  // both sorted: one walk
    for (size_t i = 0; i < c.dict.size(); ++i) {
        while (g < global.size() && global[g] < c.dict[i]) ++g;
        if (g == global.size() || global[g] != c.dict[i]) N1_THROW(N1GPU_E_INVALID, "global dictionary lacks a local string");
        remap[i] = (u32)g;
    }
    bool identity = remap.size() == global.size();
    if (!identity || !remap.empty()) for (size_t i = 0; i < remap.size() && identity; ++i) identity = remap[i] == (u32)i;
    if (!identity && !remap.empty()) {
        if (c.d_payload.p && rows_in_hbm()) remap_ranks_device(ci, remap);
        else for (size_t r = 0; r < c.tags.size(); ++r) if (c.tags[r] == C_STRING) c.payload[r] = remap[(size_t)c.payload[r]];
    }
    c.dict.swap(global);
    if (rows_in_hbm()) c.stats.set_dictionary(c.dict);  // (staged columns take theirs at seal)
}

Column& Table::exchange_column(int c) {
    if (c < 0 || c >= (int)cols.size()) N1_THROW(N1GPU_E_INVALID, "no such column");
    if (sealed) N1_THROW(N1GPU_E_INVALID, "dictionary exchange happens before seal");
    build_dictionary(c);
    return cols[(size_t)c];
}

void Table::import_dictionary(int c, const char* blob, const i64* offs, i64 n) {
    exchange_column(c);
    std::vector<std::string> global = read_dictionary(blob, offs, n, "global dictionary");
    adopt_dictionary(c, global);
}

// k-way merge of the sorted, unique dictionaries (the column's own included) into the global sorted dictionary.  The value
// range is cut at splitters taken from the longest list and every thread merges one cut (8 ranks x 100 k strings: 32 ms
// single-threaded, most of an end-to-end step at 8 GPUs).
void Table::merge_dictionaries(int c, int nparts, const char* const* blobs, const i64* const* offsets, const i64* ndicts) {
    const std::vector<std::string>& own = exchange_column(c).dict.vec();
    struct List {
        const char* blob; const i64* off; const std::vector<std::string>* own; i64 n;
        std::string_view at(i64 i) const {
            return own ? std::string_view((*own)[(size_t)i]) : std::string_view(blob + off[i], (size_t)(off[i + 1] - off[i]));
        }
        i64 lower_bound(std::string_view v) const {
            i64 lo = 0, hi = n;
            while (lo < hi) { const i64 m = (lo + hi) / 2; if (at(m) < v) lo = m + 1; else hi = m; }
            return lo;
        }
    };
    std::vector<List> lists;
    for (int p = 0; p < nparts; ++p) if (ndicts[p] > 0) lists.push_back(List{blobs[p], offsets[p], nullptr, ndicts[p]});
    if (!own.empty()) lists.push_back(List{nullptr, nullptr, &own, (i64)own.size()});
    std::vector<std::string> global;
    if (!lists.empty()) {
        size_t longest = 0;
        i64 total = 0;
        for (size_t l = 0; l < lists.size(); ++l) { total += lists[l].n; if (lists[l].n > lists[longest].n) longest = l; }
        const int nthr = total < 32768 ? 1 : (int)std::min<i64>(std::max(1u, std::thread::hardware_concurrency()), 16);
        // strictly increasing lists are the premise of the cuts: checked first (every thread takes a stripe of every list)
        parallel_for(nthr, [&](int th) {
            for (const List& L : lists)
                for (i64 i = std::max<i64>(L.n * th / nthr, 1); i < L.n * (th + 1) / nthr; ++i)
                    if (!(L.at(i - 1) < L.at(i))) N1_THROW(N1GPU_E_INVALID, "dictionaries to merge must be sorted bytewise and unique");
        });
        std::vector<std::vector<std::string_view>> out((size_t)nthr);
        parallel_for(nthr, [&](int th) {
            const List& L = lists[longest];
            const bool first = th == 0, last = th == nthr - 1;
            const std::string_view lo = first ? std::string_view() : L.at(L.n * th / nthr);
            const std::string_view hi = last ? std::string_view() : L.at(L.n * (th + 1) / nthr);
            std::vector<i64> at(lists.size()), end(lists.size());
            i64 room = 0;
            for (size_t l = 0; l < lists.size(); ++l) {
                at[l] = first ? 0 : lists[l].lower_bound(lo);
                end[l] = last ? lists[l].n : lists[l].lower_bound(hi);
                room = std::max(room, end[l] - at[l]);
            }
            auto& o = out[(size_t)th];
            o.reserve((size_t)room + 64);
            for (;;) {
                bool any = false;
                std::string_view best;
                for (size_t l = 0; l < lists.size(); ++l)
                    if (at[l] < end[l]) { const std::string_view v = lists[l].at(at[l]); if (!any || v < best) { best = v; any = true; } }
                if (!any) break;
                o.push_back(best);
                for (size_t l = 0; l < lists.size(); ++l)
                    if (at[l] < end[l]) {
                        const std::string_view v = lists[l].at(at[l]);
                        if (v.size() == best.size() && (v.data() == best.data() || memcmp(v.data(), best.data(), v.size()) == 0)) ++at[l];
                    }
            }
        });
        size_t n = 0;
        for (auto& o : out) n += o.size();
        global.reserve(n);
        for (auto& o : out) for (const std::string_view v : o) global.emplace_back(v);
    }
    adopt_dictionary(c, global);
}

void Table::build_dictionary(int c) {
    Column& col = cols[c];
    if (!col.dict_staged) return;
    std::vector<u32> order(col.local_strings.size());
    for (u32 i = 0; i < order.size(); ++i) order[i] = i;
    std::sort(order.begin(), order.end(), [&](u32 a, u32 b) { return col.local_strings[a] < col.local_strings[b]; });
    std::vector<u32> rank(order.size());
    col.dict.resize(order.size());
    for (u32 r = 0; r < order.size(); ++r) { rank[order[r]] = r; col.dict[r] = col.local_strings[order[r]]; }
    for (size_t i = 0; i < col.tags.size(); ++i)
        if (col.tags[i] == C_STRING) col.payload[i] = rank[(size_t)col.payload[i]];
    col.local_strings.clear();
    col.local_strings.shrink_to_fit();
    col.dict_staged = false;
}

ColumnStats host_stats(const std::vector<u8>& tags, const std::vector<i64>& payload) {
    ColumnStats st;
    for (size_t i = 0; i < tags.size(); ++i) {
        u8 t = tags[i];
        i64 v = payload[i];
        double d;
        memcpy(&d, &v, 8);
        if (t == C_FLOAT && f_is_int(d)) { t = C_INT; v = go_i64(d); }
        st.has_float |= t == C_FLOAT;
        if (t == C_INT) {
            st.int_min = st.has_int ? std::min(st.int_min, v) : v;
            st.int_max = st.has_int ? std::max(st.int_max, v) : v;
            st.has_int = true;
        }
        st.class_mask |= bit(t);
        st.absent_rows += t <= C_NULL;
    }
    return st;
}

DevBuf Table::device_rows(int width, int byte, cudaStream_t s) const {
    const size_t bytes = (size_t)std::max(padded_rows(), ROW_PAD) * (size_t)width;
    DevBuf b;
    b.alloc(bytes ? bytes : 256);
    if (bytes) CK(cudaMemsetAsync(b.p, byte, bytes, s));
    return b;
}

int Table::scan_bytes(int c) const {
    const Column& col = cols[c];
    return col.width + (col.stats.uniform_tag() ? 0 : 1);
}

void Table::seal() {
    if (sealed) return;
    if (rows_in_hbm()) {  // columns, dictionaries and statistics already final in HBM
        bool any_set = false;
        for (auto& col : cols) any_set = any_set || col.on_device;
        if (any_set)
            for (auto& col : cols)
                if (!col.on_device) N1_THROW(N1GPU_E_INVALID, "column %s was never set", join_path(col.path, '.').c_str());
        sealed = true;
        return;
    }
    double t0 = now_sec();
    for (auto& col : cols)
        if ((i64)col.tags.size() != nrows) N1_THROW(N1GPU_E_INVALID, "column %s has %lld rows, table has %lld",
                                                    join_path(col.path, '.').c_str(), (long long)col.tags.size(), (long long)nrows);
    auto finish = [&](int c) {
        Column& col = cols[c];
        build_dictionary(c);
        for (size_t i = 0; i < col.tags.size(); ++i) {
            const u8 t = col.tags[i];
            if (t > C_OTHER) N1_THROW(N1GPU_E_INVALID, "bad class byte %d", (int)t);
            if (t == C_FLOAT) {  // pre-shredded input may hold integral floats: canonicalise (NewValue)
                double d; memcpy(&d, &col.payload[i], 8);
                if (f_is_int(d)) { col.tags[i] = C_INT; col.payload[i] = go_i64(d); }
            }
        }
        if (!col.stats_forced) { col.stats = host_stats(col.tags, col.payload); col.stats.set_dictionary(col.dict); }
        col.width = width_of(col.stats.class_mask);
    };
    try {
        parallel_for((int)cols.size(), finish);
    } catch (const std::exception& e) {
        N1_THROW(N1GPU_E_INVALID, "%s", e.what());
    }
    shred_sec += now_sec() - t0;
    if (!segment_out.empty()) write_segment();
    t0 = now_sec();
    if (!have_device()) {
        // build / CPU-test container: dictionaries and statistics only; queries can still be compiled
        // (NVRTC -> sm_100a cubin) but never executed - there is no CPU fallback.
        for (auto& col : cols) { std::vector<i64>().swap(col.payload); std::vector<u8>().swap(col.tags); }
        sealed = true;
        return;
    }
    for (auto& col : cols) {
        col.d_tags = device_rows(1, C_MISSING, nullptr);
        col.d_payload = device_rows(col.width, 0, nullptr);
        if (nrows) CK(cudaMemcpy(col.d_tags.p, col.tags.data(), (size_t)nrows, cudaMemcpyHostToDevice));
        if (col.width == 8 && nrows) CK(cudaMemcpy(col.d_payload.p, col.payload.data(), (size_t)nrows * 8, cudaMemcpyHostToDevice));
        if (col.width == 4 && nrows) {
            std::vector<u32> narrow((size_t)nrows);
            for (i64 i = 0; i < nrows; ++i) narrow[(size_t)i] = (u32)col.payload[(size_t)i];
            CK(cudaMemcpy(col.d_payload.p, narrow.data(), (size_t)nrows * 4, cudaMemcpyHostToDevice));
        }
        std::vector<i64>().swap(col.payload);
        std::vector<u8>().swap(col.tags);
    }
    CK(cudaDeviceSynchronize());
    upload_sec += now_sec() - t0;
    sealed = true;
}

}  // namespace n1
