// execution.cpp — see execution.hpp
#include "execution.hpp"

#include <dirent.h>
#include <fcntl.h>
#include <sys/stat.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <thread>

namespace n1 {
namespace plan {

std::string node_to_json(const json::Node& n) {
    std::string s;
    switch (n.kind) {
        case json::Node::NUL: return "null";
        case json::Node::BOOL: return n.b ? "true" : "false";
        case json::Node::INT: return std::to_string(n.i);
        case json::Node::FLOAT: return json::format_float(n.d);
        case json::Node::STR: json::quote(n.s, s); return s;
        case json::Node::ARR:
            s = "[";
            for (size_t i = 0; i < n.arr.size(); ++i) { if (i) s += ","; s += node_to_json(n.arr[i]); }
            return s + "]";
        case json::Node::OBJ:
            s = "{";
            for (size_t i = 0; i < n.obj.size(); ++i) {
                if (i) s += ",";
                json::quote(n.obj[i].first, s);
                s += ":";
                s += node_to_json(n.obj[i].second);
            }
            return s + "}";
    }
    return s;
}

static std::string q(const std::string& s) { std::string o; json::quote(s, o); return o; }
static std::string list(const std::vector<std::string>& v) {
    std::string s = "[";
    for (size_t i = 0; i < v.size(); ++i) { if (i) s += ","; s += q(v[i]); }
    return s + "]";
}
static std::string term_fields(const KeyspaceTerm& t) {
    std::string s = "\"keyspace\":" + q(t.keyspace) + ",\"namespace\":" + q(t.nspace);
    if (!t.as.empty()) s += ",\"as\":" + q(t.as);
    return s;
}

void PrimaryScan::Accept(Visitor& v) { v.VisitPrimaryScan(*this); }
void Fetch::Accept(Visitor& v) { v.VisitFetch(*this); }
void Filter::Accept(Visitor& v) { v.VisitFilter(*this); }
void Group::Accept(Visitor& v) { if (phase == 0) v.VisitInitialGroup(*this); else if (phase == 1) v.VisitIntermediateGroup(*this); else v.VisitFinalGroup(*this); }
void Parallel::Accept(Visitor& v) { v.VisitParallel(*this); }
void Sequence::Accept(Visitor& v) { v.VisitSequence(*this); }
void Authorize::Accept(Visitor& v) { v.VisitAuthorize(*this); }
void Opaque::Accept(Visitor& v) { v.VisitOpaque(*this); }

std::string PrimaryScan::MarshalJSON() const {
    std::string s = "{\"#operator\":\"PrimaryScan\",\"index\":" + q(index) + "," + term_fields(term) + ",\"using\":" + q(using_);
    if (!limit.empty()) s += ",\"limit\":" + q(limit);
    return s + "}";
}
std::string Fetch::MarshalJSON() const { return "{\"#operator\":\"Fetch\"," + term_fields(term) + "}"; }
std::string Filter::MarshalJSON() const { return "{\"#operator\":\"Filter\",\"condition\":" + q(condition) + "}"; }
std::string Group::MarshalJSON() const {
    return std::string("{\"#operator\":\"") + Name() + "\",\"aggregates\":" + list(aggregates) + ",\"group_keys\":" + list(keys) + "}";
}
std::string Parallel::MarshalJSON() const {
    std::string s = "{\"#operator\":\"Parallel\"";
    if (maxParallelism > 0) s += ",\"maxParallelism\":" + std::to_string(maxParallelism);
    return s + ",\"~child\":" + child->MarshalJSON() + "}";
}
std::string Sequence::MarshalJSON() const {
    std::string s = "{\"#operator\":\"Sequence\",\"~children\":[";
    for (size_t i = 0; i < children.size(); ++i) { if (i) s += ","; s += children[i]->MarshalJSON(); }
    return s + "]}";
}
std::string Authorize::MarshalJSON() const {
    return "{\"#operator\":\"Authorize\",\"privileges\":" + (privileges_json.empty() ? std::string("null") : privileges_json) +
           ",\"~child\":" + child->MarshalJSON() + "}";
}

static std::vector<std::string> str_list(const json::Node* n) {
    std::vector<std::string> out;
    if (n && n->kind == json::Node::ARR)
        for (auto& e : n->arr) {
            if (e.kind != json::Node::STR) N1_THROW(N1GPU_E_PARSE, "plan JSON: expected a list of expression strings");
            out.push_back(e.s);
        }
    return out;
}

OperatorP MakeOperator(const json::Node& n) {
    if (n.kind != json::Node::OBJ) N1_THROW(N1GPU_E_PARSE, "plan JSON: operator must be an object");
    std::string name = n.str_or("#operator", "");
    if (name.empty()) N1_THROW(N1GPU_E_PARSE, "plan JSON: missing #operator");
    auto term = [&]() { KeyspaceTerm t; t.nspace = n.str_or("namespace", ""); t.keyspace = n.str_or("keyspace", ""); t.as = n.str_or("as", ""); return t; };
    if (name == "PrimaryScan") {
        auto* p = new PrimaryScan();
        p->term = term(); p->index = n.str_or("index", ""); p->using_ = n.str_or("using", ""); p->limit = n.str_or("limit", "");
        return OperatorP(p);
    }
    if (name == "Fetch") { auto* p = new Fetch(); p->term = term(); return OperatorP(p); }
    if (name == "Filter") { auto* p = new Filter(); p->condition = n.str_or("condition", ""); return OperatorP(p); }
    if (name == "InitialGroup" || name == "IntermediateGroup" || name == "FinalGroup") {
        auto* p = new Group();
        p->phase = name == "InitialGroup" ? 0 : (name == "IntermediateGroup" ? 1 : 2);
        p->keys = str_list(n.get("group_keys"));
        p->aggregates = str_list(n.get("aggregates"));
        return OperatorP(p);
    }
    if (name == "Parallel") {
        auto* p = new Parallel();
        OperatorP hold(p);
        const json::Node* c = n.get("~child");
        if (!c) N1_THROW(N1GPU_E_PARSE, "plan JSON: Parallel without ~child");
        p->child = MakeOperator(*c);
        const json::Node* mp = n.get("maxParallelism");
        if (mp && mp->kind == json::Node::INT) p->maxParallelism = (int)mp->i;
        return hold;
    }
    if (name == "Sequence") {
        auto* p = new Sequence();
        OperatorP hold(p);
        const json::Node* c = n.get("~children");
        if (c && c->kind == json::Node::ARR) for (auto& e : c->arr) p->children.push_back(MakeOperator(e));
        return hold;
    }
    if (name == "Authorize") {
        auto* p = new Authorize();
        OperatorP hold(p);
        const json::Node* c = n.get("~child");
        if (!c) N1_THROW(N1GPU_E_PARSE, "plan JSON: Authorize without ~child");
        p->child = MakeOperator(*c);
        if (const json::Node* pr = n.get("privileges")) p->privileges_json = node_to_json(*pr);
        return hold;
    }
    auto* p = new Opaque();
    p->name = name;
    p->body = node_to_json(n);
    return OperatorP(p);
}

}  // namespace plan

namespace execution {

namespace {

// A resident table and what it was built from: the source tag, and for a directory keyspace every entry (sorted) with the
// fingerprint of the file its row was read from - the rows are those of the entries whose state is DOC, in order.
struct Records {
    std::vector<std::string> entries;
    std::vector<DocFp> fps;
    // the directory as readdir listed it, and that listing's sorted order: the next stat pass sorts nothing while the
    // listing stays the same (sorting 10^6 names costs a quarter of a second)
    std::vector<std::string> listed;
    std::vector<u32> order;
};
struct CacheEntry {
    std::shared_ptr<Table> table;
    std::string source;
    std::shared_ptr<const Records> recs;  // null: the rows cannot be told apart by entry (a packed keyspace)
};
std::mutex g_cache_mu;
std::map<std::string, CacheEntry> g_tables;  // keyspace dir + columns -> resident shredded table (A.9)

std::string g_segment_dir;
bool g_segment_dir_set = false;

std::string segment_dir() {
    std::lock_guard<std::mutex> lk(g_cache_mu);
    if (!g_segment_dir_set) { const char* e = getenv("N1GPU_SEGMENT_DIR"); g_segment_dir = e ? e : ""; g_segment_dir_set = true; }
    return g_segment_dir;
}

// A keyspace directory as one stat pass sees it.
struct KeyspaceScan {
    // What a segment is valid for: the keyspace directory as the file datastore sees it (file.go:711-749) - modification
    // time of the directory (documents added / removed), number of documents, newest document (rewritten in place by
    // UPDATE, file.go:375-471) and their total size.
    std::string tag;
    std::vector<std::string> entries;  // non-directory entries, sorted (the primary-key order of load_dir)
    std::vector<DocFp> fps;            // the stat of each entry's document file (document_file)
    std::vector<std::string> listed;   // see Records
    std::vector<u32> order;
};

// One stat per entry (two for an entry that is not its own document file, a.txt -> a.json); no document is opened.
KeyspaceScan scan_keyspace(const std::string& dir, const Records* prev) {
    DIR* d = opendir(dir.c_str());
    if (!d) N1_THROW(N1GPU_E_IO, "cannot open keyspace directory %s", dir.c_str());
    struct stat ds;
    long long dir_s = 0, dir_ns = 0;
    if (stat(dir.c_str(), &ds) == 0) { dir_s = ds.st_mtim.tv_sec; dir_ns = ds.st_mtim.tv_nsec; }
    std::vector<std::string> names;
    while (dirent* e = readdir(d)) {
        const char* n = e->d_name;
        if (n[0] == '.' && (n[1] == 0 || (n[1] == '.' && n[2] == 0))) continue;
        names.emplace_back(n);
    }
    std::vector<u32> order;
    if (prev && prev->listed == names) order = prev->order;
    else {
        order.resize(names.size());
        for (u32 i = 0; i < order.size(); ++i) order[i] = i;
        std::sort(order.begin(), order.end(), [&](u32 a, u32 b) { return names[a] < names[b]; });
    }
    // fstatat relative to the open directory, on all cores for a large keyspace (10^4 documents: 7 ms -> under 1 ms; this is
    // the whole cost of a query over a resident keyspace)
    const int dfd = dirfd(d);
    const size_t nthr = names.size() < 2048 ? 1 : std::min<size_t>(std::max(1u, std::thread::hardware_concurrency()), 16);
    struct Part { long long files = 0, bytes = 0, newest_s = 0, newest_ns = 0; };
    std::vector<Part> parts(nthr);
    std::vector<DocFp> fps(names.size());
    std::vector<char> is_entry(names.size(), 0);
    auto work = [&](size_t t) {
        Part& p = parts[t];
        for (size_t i = names.size() * t / nthr; i < names.size() * (t + 1) / nthr; ++i) {
            struct stat st;
            if (fstatat(dfd, names[i].c_str(), &st, 0) != 0 || S_ISDIR(st.st_mode)) continue;
            ++p.files;
            p.bytes += (long long)st.st_size;
            if (st.st_mtim.tv_sec > p.newest_s || (st.st_mtim.tv_sec == p.newest_s && st.st_mtim.tv_nsec > p.newest_ns)) { p.newest_s = st.st_mtim.tv_sec; p.newest_ns = st.st_mtim.tv_nsec; }
            is_entry[i] = 1;
            const std::string doc = document_file(names[i]);
            if (doc == names[i]) { fps[i] = DocFp::of(st); continue; }
            struct stat ss;
            if (fstatat(dfd, doc.c_str(), &ss, 0) == 0) {
                if (S_ISDIR(ss.st_mode)) fps[i].state = DocFp::UNREADABLE;
                else fps[i] = DocFp::of(ss);
            } else fps[i].state = errno == ENOENT ? DocFp::ABSENT : DocFp::UNREADABLE;
        }
    };
    if (nthr == 1) work(0);
    else {
        std::vector<std::thread> pool;
        for (size_t t = 0; t < nthr; ++t) pool.emplace_back(work, t);
        for (auto& th : pool) th.join();
    }
    closedir(d);
    Part all;
    for (const Part& p : parts) {
        all.files += p.files; all.bytes += p.bytes;
        if (p.newest_s > all.newest_s || (p.newest_s == all.newest_s && p.newest_ns > all.newest_ns)) { all.newest_s = p.newest_s; all.newest_ns = p.newest_ns; }
    }
    KeyspaceScan ks;
    ks.tag = strf("dir=%lld.%09lld files=%lld newest=%lld.%09lld bytes=%lld", dir_s, dir_ns, all.files, all.newest_s, all.newest_ns, all.bytes);
    ks.entries.reserve((size_t)all.files);
    ks.fps.reserve((size_t)all.files);
    for (const u32 i : order)
        if (is_entry[i]) { ks.entries.push_back(names[i]); ks.fps.push_back(fps[i]); }
    ks.listed = std::move(names);
    ks.order = std::move(order);
    return ks;
}

i64 realtime_ns() {
    struct timespec ts;
    clock_gettime(CLOCK_REALTIME, &ts);
    return (i64)ts.tv_sec * 1000000000 + ts.tv_nsec;
}

// Racily clean files (git's rule): a file changed less than a timestamp tick before it was read can change again within
// the same tick without its stat showing it.  Every file whose ctime is not older than the start of the load, less this
// margin (coarse kernel timestamps lag the clock by up to a tick), is read again at the next check.
const i64 RACY_MARGIN_NS = 20 * 1000000;
void mark_racy(std::vector<DocFp>& fps, i64 start_ns) {
    for (DocFp& f : fps) if (f.state == DocFp::DOC && f.ctime_ns >= start_ns - RACY_MARGIN_NS) f.racy = true;
}

void trace_phase(const char* what, const char* name, double& tp) {
    static const bool trace = getenv("N1GPU_TRACE") != nullptr;
    const double t = now_sec();
    if (trace) fprintf(stderr, "[n1gpu %s] %-10s %8.3f ms\n", what, name, (t - tp) * 1e3);
    tp = t;
}

// The cached table refreshed for a directory keyspace that changed: the rows of entries whose fingerprint holds are
// kept, the documents of changed, new and unreadable entries are read again and shredded into a patch table, the rows of
// deleted entries drop out, and the device splices the new columns from the old ones and the patch.  Returns the old table
// itself when no row changed (a touched directory).  The result equals a load of the directory from scratch.
std::shared_ptr<Table> refresh_table(const std::string& dir, const std::vector<std::string>& paths, const std::shared_ptr<Table>& old_table,
                                     const Records& old, const KeyspaceScan& now, i64 start_ns, bool host_shred, std::vector<DocFp>& fps, i64* docs_read) {
    double tp = now_sec();
    // merge of the two sorted entry lists; old_row[i]: the old row of old entry i (-1: none)
    std::vector<i64> old_row(old.entries.size(), -1);
    i64 r = 0;
    for (size_t i = 0; i < old.entries.size(); ++i) if (old.fps[i].state == DocFp::DOC) old_row[i] = r++;
    if (r != old_table->nrows) N1_THROW(N1GPU_E_INVALID, "resident table of %s does not match its entries", dir.c_str());
    std::vector<size_t> reread;           // indices into now.entries
    std::vector<i64> keep(now.entries.size(), -2);  // the old row kept; -1: no row, as before; -2: read again
    for (size_t i = 0, o = 0; i < now.entries.size(); ++i) {
        while (o < old.entries.size() && old.entries[o] < now.entries[i]) ++o;  // deleted entries
        if (o < old.entries.size() && old.entries[o] == now.entries[i]) {
            if (old.fps[o].holds(now.fps[i])) { keep[i] = old_row[o]; fps[i] = old.fps[o]; }
            ++o;
        }
        if (keep[i] == -2) reread.push_back(i);
    }
    trace_phase("refresh", "diff", tp);
    std::shared_ptr<Table> patch;
    std::vector<DocFp> pfps;
    if (!reread.empty()) {
        std::vector<std::string> names(reread.size());
        for (size_t k = 0; k < reread.size(); ++k) names[k] = now.entries[reread[k]];
        patch = std::make_shared<Table>();
        for (auto& p : paths) patch->add_column(p);
        patch->load_entries(dir, names, host_shred ? 0 : -1, &pfps);
        mark_racy(pfps, start_ns);
        for (size_t k = 0; k < reread.size(); ++k) fps[reread[k]] = pfps[k];
        trace_phase("refresh", "read", tp);
        patch->seal();
        trace_phase("refresh", "seal", tp);
        if (patch->nrows == 0) patch.reset();
    }
    *docs_read = patch ? patch->nrows : 0;
    // runs: consecutive new rows from consecutive rows of one source
    std::vector<SpliceRun> runs;
    i64 at = 0, prow = 0;
    auto add = [&](bool from_patch, i64 src) {
        if (!runs.empty() && runs.back().patch == from_patch && runs.back().src_lo + runs.back().len == src) ++runs.back().len;
        else runs.push_back(SpliceRun{at, from_patch, src, 1});
        ++at;
    };
    for (size_t k = 0, i = 0; i < now.entries.size(); ++i) {
        if (keep[i] >= 0) add(false, keep[i]);
        else if (keep[i] == -2 && pfps[k++].state == DocFp::DOC) add(true, prow++);
    }
    if (!patch && at == old_table->nrows && runs.size() <= 1) return old_table;  // the same rows: nothing to splice
    auto t = std::make_shared<Table>();
    for (auto& p : paths) t->add_column(p);
    t->splice(*old_table, patch.get(), runs);
    trace_phase("refresh", "splice", tp);
    return t;
}

std::shared_ptr<Table> resident_table(const std::string& dir, std::vector<std::string> paths, i64* docs_read) {
    std::sort(paths.begin(), paths.end());
    std::string key = dir;
    for (auto& p : paths) { key.push_back('\n'); key += p; }
    struct stat st;
    // A keyspace too large for one file per document (file.go:312-353) is kept packed: <namespace>/<keyspace>.ndjson, one
    // document per line in primary-key order, takes the place of the directory <namespace>/<keyspace>/.
    const std::string packed = dir + ".ndjson";
    const bool is_dir = stat(dir.c_str(), &st) == 0 && S_ISDIR(st.st_mode);
    struct stat pst;
    const bool is_packed = !is_dir && stat(packed.c_str(), &pst) == 0 && S_ISREG(pst.st_mode);
    if (!is_dir && !is_packed) N1_THROW(N1GPU_E_IO, "keyspace directory %s not found", dir.c_str());
    // the resident table and the segment live as long as this tag holds; a directory keyspace's table as long as the
    // fingerprints of its documents hold, and is refreshed from the changed documents when they do not
    *docs_read = 0;
    const i64 start_ns = realtime_ns();
    double tp = now_sec();
    std::shared_ptr<const Records> prev;
    {
        std::lock_guard<std::mutex> lk(g_cache_mu);
        auto it = g_tables.find(key);
        if (it != g_tables.end()) prev = it->second.recs;
    }
    KeyspaceScan scan;
    if (is_dir) scan = scan_keyspace(dir, prev.get());
    const std::string tag = is_dir ? scan.tag
                                   : strf("ndjson mtime=%lld.%09lld bytes=%lld", (long long)pst.st_mtim.tv_sec, (long long)pst.st_mtim.tv_nsec, (long long)pst.st_size);
    trace_phase("load", "stat", tp);
    const std::string segs = segment_dir();
    const std::string file = segs.empty() ? std::string() : segs + "/" + strf("%016llx", (unsigned long long)mix64(std::hash<std::string>()(key))) + ".n1seg";
    CacheEntry old;
    {
        std::lock_guard<std::mutex> lk(g_cache_mu);
        auto it = g_tables.find(key);
        if (it != g_tables.end()) {
            if (it->second.source == tag && !it->second.recs) return it->second.table;  // (packed: the tag is all there is)
            const Records* r = it->second.recs.get();
            bool holds = is_dir && r && r->entries == scan.entries;
            for (size_t i = 0; holds && i < scan.fps.size(); ++i) holds = r->fps[i].holds(scan.fps[i]);
            if (holds) {
                if (it->second.source == tag) return it->second.table;
                // a touched directory: the same rows under a new tag (and the segment rewritten under it)
                it->second.source = tag;
                if (!file.empty() && have_device()) it->second.table->write_segment(file, tag);
                return it->second.table;
            }
            old = it->second;
        }
    }
    // The documents are shredded on the device (raw text -> HBM once, no column crosses PCIe) unless a segment is to be
    // written from the host shredder's staging, or N1GPU_OPERATOR_SHRED=host asks for the host threads.
    const char* how = getenv("N1GPU_OPERATOR_SHRED");
    const bool host_env = (how && std::string(how) == "host") || paths.empty();
    std::vector<DocFp> fps(scan.fps.size());
    bool is_rec = true;
    std::shared_ptr<Table> t;
    if (is_dir && old.recs && have_device()) {
        t = refresh_table(dir, paths, old.table, *old.recs, scan, start_ns, host_env, fps, docs_read);
        t->global_rows = t->nrows;
        if (!file.empty()) { t->write_segment(file, tag); trace_phase("refresh", "segment", tp); }
    } else {
        t = std::make_shared<Table>();
        for (auto& p : paths) t->add_column(p);
        bool from_segment = false;
        if (!file.empty()) {  // persistent columnar segment: skip reading and parsing the documents while nothing changed
            from_segment = t->load_segment(file, tag);
            if (!from_segment) { t->segment_out = file; t->segment_source = tag; }
        }
        if (from_segment) {  // the stat pass that validated the tag gives the fingerprints
            fps = scan.fps;
            i64 docs = 0;
            for (const DocFp& f : fps) docs += f.state == DocFp::DOC;
            if (docs != t->nrows) is_rec = false;  // (rows that were not readable then): no refresh from these
        } else {
            const bool host = !have_device() || !t->segment_out.empty() || host_env;
            const int threads = host ? 0 : -1;
            if (is_dir) t->load_dir(dir, threads, &scan.entries, &fps); else t->load_ndjson(packed, threads);
            *docs_read = t->nrows;
        }
        trace_phase("load", "read", tp);
        t->global_rows = t->nrows;  // the operator runs the whole keyspace in this process: one partition
        t->seal();
        trace_phase("load", "seal", tp);
    }
    mark_racy(fps, start_ns);
    std::shared_ptr<const Records> recs;
    if (is_dir && is_rec) recs = std::make_shared<const Records>(Records{std::move(scan.entries), std::move(fps), std::move(scan.listed), std::move(scan.order)});
    std::lock_guard<std::mutex> lk(g_cache_mu);
    g_tables[key] = CacheEntry{t, tag, recs};
    return t;
}

// plan.Visitor implementation: the builder of execution/build.go restricted to the substitution.
struct Builder : plan::Visitor {
    std::string root;
    std::unique_ptr<GpuGroupAggregate> found;
    int rest = 0;
    bool want_tail = false;                // the caller can run a tail (n1gpu_plan_build_tail): SELECT DISTINCT needs one
    plan::Sequence* chain_seq = nullptr;   // the Sequence that holds the chain
    plan::Sequence* outer_seq = nullptr;   // the Sequence that holds chain_seq as a direct child (ORDER BY / LIMIT plans)
    size_t outer_index = 0;                // ... at this position
    plan::Sequence* cur_parent = nullptr;  // direct-parent bookkeeping while descending
    size_t cur_index = 0;
    std::string why = "plan holds no PrimaryScan/Fetch/Filter/InitialGroup/IntermediateGroup/FinalGroup chain";

    void VisitPrimaryScan(plan::PrimaryScan&) override {}
    void VisitFetch(plan::Fetch&) override {}
    void VisitFilter(plan::Filter&) override {}
    void VisitInitialGroup(plan::Group&) override {}
    void VisitIntermediateGroup(plan::Group&) override {}
    void VisitFinalGroup(plan::Group&) override {}
    void VisitOpaque(plan::Opaque&) override {}
    void VisitParallel(plan::Parallel& p) override { if (!found) { cur_parent = nullptr; p.child->Accept(*this); } }
    void VisitAuthorize(plan::Authorize& a) override { if (!found) { cur_parent = nullptr; a.child->Accept(*this); } }

    // Flattens [Filter?, InitialGroup] out of Parallel(Sequence[..]) / Sequence[..] / bare operators
    // (execution/build.go:455-491 elides Parallel at parallelism 1 and single-child Sequences).
    static void flatten(plan::Operator* op, std::vector<plan::Operator*>& out) {
        if (auto* p = dynamic_cast<plan::Parallel*>(op)) { flatten(p->child.get(), out); return; }
        if (auto* s = dynamic_cast<plan::Sequence*>(op)) { for (auto& c : s->children) flatten(c.get(), out); return; }
        out.push_back(op);
    }

    void VisitSequence(plan::Sequence& s) override {
        if (found) return;
        plan::Sequence* const my_parent = cur_parent;
        const size_t my_index = cur_index;
        auto& ch = s.children;
        auto* scan = ch.size() > 0 ? dynamic_cast<plan::PrimaryScan*>(ch[0].get()) : nullptr;
        auto* fetch = ch.size() > 1 ? dynamic_cast<plan::Fetch*>(ch[1].get()) : nullptr;
        if (scan && fetch) {
            // children[2..]: the Filter/InitialGroup part, then IntermediateGroup, FinalGroup
            size_t i = 2;
            std::vector<plan::Operator*> mid;
            while (i < ch.size()) {
                auto* g = dynamic_cast<plan::Group*>(ch[i].get());
                if (g && g->phase >= 1) break;
                if (dynamic_cast<plan::Opaque*>(ch[i].get())) break;
                flatten(ch[i].get(), mid);
                ++i;
            }
            plan::Filter* filter = nullptr;
            plan::Group* initial = nullptr;
            bool ok = true;
            for (auto* m : mid) {
                if (auto* f = dynamic_cast<plan::Filter*>(m)) { if (filter || initial) ok = false; filter = f; }
                else if (auto* g = dynamic_cast<plan::Group*>(m)) { if (initial || g->phase != 0) ok = false; initial = g; }
                else ok = false;  // Let, Join, Nest, Unnest, ... between Fetch and InitialGroup
            }
            auto* inter = i < ch.size() ? dynamic_cast<plan::Group*>(ch[i].get()) : nullptr;
            auto* fin = i + 1 < ch.size() ? dynamic_cast<plan::Group*>(ch[i + 1].get()) : nullptr;
            // SELECT DISTINCT <terms> FROM ks [WHERE]: [.., Parallel(Sequence[Filter?, InitialProject(distinct), Distinct,
            // FinalProject?]), Distinct, ..] (planner/build_select_sub.go:217-243).  Grouping by the projected terms
            // with no aggregates yields exactly the distinct rows; the projection itself is the operator's tail.
            if (want_tail && !initial && ok == false) {
                plan::Filter* f2 = nullptr;
                plan::Opaque* proj = nullptr;
                bool shape = true;
                for (auto* m : mid) {
                    if (auto* f = dynamic_cast<plan::Filter*>(m)) { if (f2 || proj) shape = false; f2 = f; }
                    else if (auto* o = dynamic_cast<plan::Opaque*>(m)) {
                        if (o->name == "InitialProject" && !proj) proj = o;
                        else if (!(proj && (o->name == "Distinct" || o->name == "FinalProject"))) shape = false;
                    } else shape = false;
                }
                json::Node pn;
                std::vector<std::string> terms;
                if (shape && proj && json::parse(proj->body, pn)) {
                    const json::Node* d = pn.get("distinct");
                    const json::Node* ts = pn.get("result_terms");
                    if (d && d->kind == json::Node::BOOL && d->b && ts && ts->kind == json::Node::ARR)
                        for (auto& t : ts->arr) { const std::string e = t.str_or("expr", ""); if (e.empty() || t.get("star")) { terms.clear(); break; } terms.push_back(e); }
                }
                if (!terms.empty() && scan->limit.empty() && scan->term.keyspace == fetch->term.keyspace && scan->term.nspace == fetch->term.nspace) {
                    std::unique_ptr<GpuGroupAggregate> op(new GpuGroupAggregate());
                    op->term = fetch->term;
                    if (op->term.as.empty()) op->term.as = scan->term.as;
                    op->keyspace_dir = root + "/" + fetch->term.nspace + "/" + fetch->term.keyspace;
                    if (f2) op->condition = f2->condition;
                    op->keys = terms;  // duplicates collapse below: a key per distinct term text
                    std::sort(op->keys.begin(), op->keys.end());
                    op->keys.erase(std::unique(op->keys.begin(), op->keys.end()), op->keys.end());
                    op->tail.distinct_by_keys = true;
                    found = std::move(op);
                    rest = 2;  // the tail starts at the Parallel that holds the projection
                    chain_seq = &s;
                    outer_seq = my_parent;
                    outer_index = my_index;
                    return;
                }
            }
            if (!ok || !initial) why = "operators between Fetch and InitialGroup are not just Filter";
            else if (!inter || inter->phase != 1 || !fin || fin->phase != 2) why = "InitialGroup is not followed by IntermediateGroup, FinalGroup";
            else if (inter->keys != initial->keys || fin->keys != initial->keys || inter->aggregates != initial->aggregates || fin->aggregates != initial->aggregates)
                why = "group phases disagree on keys/aggregates";
            else if (!scan->limit.empty()) why = "PrimaryScan carries a LIMIT";
            else if (scan->term.keyspace != fetch->term.keyspace || scan->term.nspace != fetch->term.nspace) why = "scan and fetch keyspaces differ";
            else {
                std::unique_ptr<GpuGroupAggregate> op(new GpuGroupAggregate());
                op->term = fetch->term;
                if (op->term.as.empty()) op->term.as = scan->term.as;
                op->keyspace_dir = root + "/" + fetch->term.nspace + "/" + fetch->term.keyspace;
                if (filter) op->condition = filter->condition;
                op->keys = initial->keys;
                op->aggregates = initial->aggregates;
                found = std::move(op);
                rest = (int)i + 2;
                chain_seq = &s;
                outer_seq = my_parent;
                outer_index = my_index;
                return;
            }
        }
        for (size_t c = 0; c < ch.size(); ++c) {
            if (found) return;
            cur_parent = &s;
            cur_index = c;
            ch[c]->Accept(*this);
        }
    }
};

std::string dur(double sec) {  // time.Duration.String() style
    if (sec <= 0) return "0s";
    if (sec < 1e-6) return strf("%.0fns", sec * 1e9);
    if (sec < 1e-3) return strf("%.3fµs", sec * 1e6);
    if (sec < 1) return strf("%.6fms", sec * 1e3);
    return strf("%.9fs", sec);
}

std::string value_json(const HValue& v) {
    switch (v.cls) {
        case C_NULL: return "null";
        case C_FALSE: return "false";
        case C_TRUE: return "true";
        case C_INT: return std::to_string(v.bits);
        case C_FLOAT: return json::format_float(v.f());
        case C_STRING: { std::string s; json::quote(v.s, s); return s; }
        default: return "null";
    }
}

struct Tree {
    std::map<std::string, Tree> kids;
    std::string leaf;
    bool has_leaf = false;
    std::string render() const {
        if (has_leaf) return leaf;
        std::string s = "{";
        bool first = true;
        for (auto& kv : kids) {
            if (!first) s += ",";
            first = false;
            json::quote(kv.first, s);
            s += ":";
            s += kv.second.render();
        }
        return s + "}";
    }
};

}  // namespace

std::unique_ptr<GpuGroupAggregate> Build(const std::string& plan_json, const std::string& datastore_root, int* rest_index) {
    return BuildWithTail(plan_json, datastore_root, false, rest_index, nullptr);
}

std::unique_ptr<GpuGroupAggregate> BuildWithTail(const std::string& plan_json, const std::string& datastore_root, bool want_tail,
                                                 int* rest_index, int* outer_rest) {
    json::Node root;
    if (!json::parse(plan_json, root)) N1_THROW(N1GPU_E_PARSE, "plan JSON does not parse");
    const json::Node* pn = &root;
    if (root.kind == json::Node::OBJ && !root.get("#operator") && root.get("plan")) pn = root.get("plan");  // EXPLAIN row {plan, text}
    plan::OperatorP p = plan::MakeOperator(*pn);
    Builder b;
    b.root = datastore_root;
    b.want_tail = want_tail;
    p->Accept(b);
    if (!b.found) N1_THROW(N1GPU_E_INELIGIBLE, "not substituted: %s", b.why.c_str());
    std::unique_ptr<GpuGroupAggregate> op = std::move(b.found);
    // referenced field paths -> resident shredded table
    std::string alias = op->term.Alias();
    std::vector<std::string> paths;
    if (!op->condition.empty()) collect_paths(*parse_expr(op->condition), alias, paths);
    for (auto& k : op->keys) collect_paths(*parse_expr(k), alias, paths);
    for (auto& a : op->aggregates) collect_paths(*parse_expr(a), alias, paths);
    double t0 = now_sec();
    op->table = resident_table(op->keyspace_dir, paths, &op->docs_read);
    op->query = Query::compile(op->table.get(), alias, op->condition.empty() ? nullptr : op->condition.c_str(), op->keys, op->aggregates);
    op->serv_sec = now_sec() - t0;
    if (outer_rest) *outer_rest = 0;
    if (want_tail) {
        // The operators behind FinalGroup: whole children of the chain's Sequence (a Parallel(Sequence[...]) counts as
        // one), then plain operators of the enclosing Sequence.  All or nothing up to FinalProject.
        GroupTail t;
        t.keyspace_alias = alias;
        t.distinct_by_keys = op->tail.distinct_by_keys;
        auto as_node = [](plan::Operator* o, json::Node& n) { return json::parse(o->MarshalJSON(), n); };
        bool ok = true;
        size_t c = (size_t)b.rest;
        for (; c < b.chain_seq->children.size(); ++c) {
            std::vector<plan::Operator*> flat;
            Builder::flatten(b.chain_seq->children[c].get(), flat);
            size_t k = 0;
            // SELECT DISTINCT: the Filter in front of the projection is the WHERE the scan already applied, not a HAVING
            if (t.distinct_by_keys && c == (size_t)b.rest && !flat.empty() && dynamic_cast<plan::Filter*>(flat[0])) flat.erase(flat.begin());
            for (; k < flat.size(); ++k) {
                json::Node n;
                if (!as_node(flat[k], n) || !t.add(n, op->keys, op->aggregates)) break;
            }
            if (k == flat.size()) continue;
            ok = k == 0 && t.final_project;  // a foreign operator behind a finished tail ends it; anything else voids it
            break;
        }
        t.inner_consumed = ok ? (int)(c - (size_t)b.rest) : 0;
        if (ok && b.outer_seq && c == b.chain_seq->children.size()) {
            for (size_t k = b.outer_index + 1; k < b.outer_seq->children.size(); ++k) {
                plan::Operator* o = b.outer_seq->children[k].get();
                json::Node n;
                if (dynamic_cast<plan::Parallel*>(o) || dynamic_cast<plan::Sequence*>(o) || !as_node(o, n) || !t.add(n, op->keys, op->aggregates)) break;
                ++t.outer_consumed;
            }
        }
        if (ok && t.final_project) {
            if (outer_rest) *outer_rest = t.outer_consumed ? (int)b.outer_index + 1 + t.outer_consumed : 0;
            b.rest += t.inner_consumed;
            op->tail = std::move(t);
        } else if (op->tail.distinct_by_keys)
            N1_THROW(N1GPU_E_INELIGIBLE, "not substituted: the projection of this SELECT DISTINCT is outside the subset");
    }
    if (rest_index) *rest_index = b.rest;
    return op;
}

std::unique_ptr<Result> GpuGroupAggregate::RunOnce() {
    if (ran) N1_THROW(N1GPU_E_INVALID, "RunOnce executes exactly once per operator (util.Once); Build a new operator");
    ran = true;
    double t0 = now_sec();
    query->scan_blocking();
    std::unique_ptr<Result> r = query->finalize();
    exec_sec = now_sec() - t0;
    in_docs = table->nrows;
    out_docs = r->ngroups;
    return r;
}

void GpuGroupAggregate::SendStop() { if (query) query->cancel(); }

std::string GpuGroupAggregate::MarshalJSON() const {
    std::string s = "{\"#operator\":\"GpuGroupAggregate\"";
    std::string stats;
    if (in_docs) stats += "\"#itemsIn\":" + std::to_string(in_docs);
    if (out_docs) stats += std::string(stats.empty() ? "" : ",") + "\"#itemsOut\":" + std::to_string(out_docs);
    if (exec_sec > 0) { stats += std::string(stats.empty() ? "" : ",") + "\"execTime\":"; json::quote(dur(exec_sec), stats); }
    if (serv_sec > 0) { stats += std::string(stats.empty() ? "" : ",") + "\"servTime\":"; json::quote(dur(serv_sec), stats); }
    if (docs_read) stats += std::string(stats.empty() ? "" : ",") + "\"#docsRead\":" + std::to_string(docs_read);
    if (!stats.empty()) s += ",\"#stats\":{" + stats + "}";
    s += ",\"aggregates\":[";
    for (size_t i = 0; i < aggregates.size(); ++i) { if (i) s += ","; json::quote(aggregates[i], s); }
    s += "]";
    if (!term.as.empty()) { s += ",\"as\":"; json::quote(term.as, s); }
    if (!condition.empty()) { s += ",\"condition\":"; json::quote(condition, s); }
    s += ",\"group_keys\":[";
    for (size_t i = 0; i < keys.size(); ++i) { if (i) s += ","; json::quote(keys[i], s); }
    s += "],\"keyspace\":";
    json::quote(term.keyspace, s);
    s += ",\"namespace\":";
    json::quote(term.nspace, s);
    // EXPLAIN in the shape the reference uses when somebody else computes the groups (plan/scan_index_groupagg.go:188-222,
    // IndexGroupAggregates: name / group [{id, keypos, expr}] / aggregates [{aggregate, id, keypos, expr, distinct}]; ids number
    // the group keys first, then the aggregates; keypos -1 = an expression, not an index key position; complete groups,
    // so no "partial")
    if (query) {
        s += ",\"group_aggs\":{\"name\":\"GpuGroupAggregate\"";
        if (!keys.empty()) {
            s += ",\"group\":[";
            for (size_t i = 0; i < keys.size(); ++i) { s += strf("%s{\"id\":%d,\"keypos\":-1,\"expr\":", i ? "," : "", (int)i); json::quote(keys[i], s); s += "}"; }
            s += "]";
        }
        if (!query->aggs.empty()) {
            static const char* ops[] = {"COUNT", "COUNTN", "SUM", "AVG", "MIN", "MAX"};
            s += ",\"aggregates\":[";
            for (size_t i = 0; i < query->aggs.size(); ++i) {
                const Expr& a = *query->aggs[i];
                s += strf("%s{\"aggregate\":\"%s\",\"id\":%d,\"keypos\":-1", i ? "," : "", ops[(int)a.agg], (int)(keys.size() + i));
                if (a.distinct) s += ",\"distinct\":true";
                s += ",\"expr\":";
                json::quote(a.star ? std::string("*") : a.ops[0]->str(), s);
                s += "}";
            }
            s += "]";
        }
        s += "}";
    }
    if (!tail.empty()) {  // the operators behind FinalGroup this operator also stands for
        s += ",\"tail\":[";
        for (size_t i = 0; i < tail.operators.size(); ++i) { if (i) s += ","; json::quote(tail.operators[i], s); }
        s += "]";
    }
    if (query) {
        static const char* modes[] = {"ungrouped", "dense-shared-memory", "hbm-hash-64", "hbm-hash-128"};
        s += std::string(",\"kernel\":{\"mode\":\"") + (query->kp.dense_global ? "hbm-direct" : modes[query->kp.mode]) + "\",\"accumulator_words\":" + std::to_string(query->ops.n) +
             ",\"scan_bytes_per_row\":" + std::to_string(query->kp.scan_bytes_per_row) + "}";
    }
    return s + "}";
}

void set_segment_dir(const std::string& dir) {
    std::lock_guard<std::mutex> lk(g_cache_mu);
    g_segment_dir = dir;
    g_segment_dir_set = true;
}

std::string ResultToJSON(const Result& r) {
    std::string s = "[";
    for (i64 g = 0; g < r.ngroups; ++g) {
        if (g) s += ",";
        Tree doc;
        std::string keys = "[";
        for (int k = 0; k < r.nkeys; ++k) {
            const HValue v = r.key(g, k);
            if (k) keys += ",";
            keys += v.cls == C_MISSING ? "{\"#missing\":true}" : value_json(v);
            if (v.cls == C_MISSING) continue;  // MISSING key: field absent (group_util.go:28-30)
            const auto& path = r.key_paths[(size_t)k];
            if (path.empty()) continue;
            Tree* t = &doc;
            for (auto& name : path) t = &t->kids[name];
            t->has_leaf = true;
            t->leaf = value_json(v);
        }
        keys += "]";
        s += "{";
        json::quote(r.alias, s);
        s += ":" + doc.render() + ",\"aggregates\":{";
        for (int a = 0; a < r.naggs; ++a) {
            if (a) s += ",";
            json::quote(r.agg_texts[(size_t)a], s);
            s += ":" + value_json(r.agg(g, a));
        }
        s += "},\"group_keys\":" + keys + "}";
    }
    return s + "]";
}

}  // namespace execution
}  // namespace n1
