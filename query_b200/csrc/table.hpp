// table.hpp — a shredded keyspace: typed columns + per-column sorted dictionaries, resident in HBM.
#pragma once
#include <map>
#include <functional>
#include <memory>
#include <string>
#include <unordered_map>
#include <vector>

#include <sys/stat.h>

#include "common.hpp"

namespace n1 {

const i64 ROW_PAD = 4096;  // device arrays are padded to a multiple of this many rows (vector loads never fault)

// A column's dictionary: a vector of strings that results can keep alive after the table is gone (a result refers to its
// strings as (column, rank) and resolves them on demand - a million-group result copies no string at finalisation).
// The table is immutable once sealed, so sharing needs no copy-on-write.
class SharedDict {
    std::shared_ptr<std::vector<std::string>> p = std::make_shared<std::vector<std::string>>();
public:
    typedef std::vector<std::string>::const_iterator const_iterator;
    size_t size() const { return p->size(); }
    bool empty() const { return p->empty(); }
    const std::string& operator[](size_t i) const { return (*p)[i]; }
    std::string& operator[](size_t i) { return (*p)[i]; }
    const_iterator begin() const { return p->begin(); }
    const_iterator end() const { return p->end(); }
    void clear() { p = std::make_shared<std::vector<std::string>>(); }
    void reserve(size_t n) { p->reserve(n); }
    void resize(size_t n) { p->resize(n); }
    template <class... A> void emplace_back(A&&... a) { p->emplace_back(std::forward<A>(a)...); }
    void push_back(const std::string& s) { p->push_back(s); }
    void swap(std::vector<std::string>& o) { auto n = std::make_shared<std::vector<std::string>>(); n->swap(o); o.swap(*p); p = n; }
    SharedDict& operator=(std::vector<std::string>&& o) { p = std::make_shared<std::vector<std::string>>(std::move(o)); return *this; }
    bool operator!=(const SharedDict& o) const { return *p != *o.p; }
    bool operator==(const SharedDict& o) const { return *p == *o.p; }
    const std::vector<std::string>& vec() const { return *p; }
    std::shared_ptr<const std::vector<std::string>> share() const { return p; }
};

struct ColumnStats {
    u32 class_mask = 0;  // classes that occur (bit per C_*)
    bool has_int = false;
    i64 int_min = 0, int_max = 0;
    bool has_float = false;  // a FLOAT that is not integral occurs
    i64 ndict = 0;
    i64 empty_rank = -1;  // rank of "" in the dictionary, -1 if absent
    i64 absent_rows = 0;  // rows whose class is MISSING or NULL (decides which way a COUNT(x) counter counts)
    bool uniform_tag() const { return class_mask != 0 && (class_mask & (class_mask - 1)) == 0; }
    void set_dictionary(const SharedDict& d) { ndict = (i64)d.size(); empty_rank = (!d.empty() && d[0].empty()) ? 0 : -1; }
};

// Statistics of staged host rows (the dictionary's aside).  An integral FLOAT counts as the INT it canonicalises to
// (NewValue); the rows are left as they are.
ColumnStats host_stats(const std::vector<u8>& tags, const std::vector<i64>& payload);

// Device payload width of a column whose classes are `class_mask`: 8 with numbers, 4 (string ranks) with strings, else 0.
// seal() applies it to the column's statistics - those of all partitions when stats_set replaced them - while the device
// shredder and set_column_device apply it to the classes of their own rows: two partitions whose rows differ in classes
// can then give a device-shredded column different widths.
inline int width_of(u32 class_mask) { return (class_mask & M_NUM) ? 8 : (class_mask & bit(C_STRING)) ? 4 : 0; }

// The strings of a caller's dictionary (blob + offsets), which must be sorted bytewise and unique (`what` names it)
std::vector<std::string> read_dictionary(const char* blob, const i64* offs, i64 n, const char* what);

struct Column {
    std::vector<std::string> path;       // field names below the document root
    // host staging (dropped after seal unless keep_host)
    std::vector<i64> payload;            // 8 bytes per row while staging
    std::vector<u8> tags;
    SharedDict dict;                     // sorted, unique (after seal / import); results keep it alive (share())
    std::vector<std::string> local_strings;  // staging: distinct strings, codes index this until seal
    bool dict_staged = true;             // STRING rows hold codes into local_strings, not ranks into dict (build_dictionary)
    ColumnStats stats;
    bool stats_forced = false;
    int width = 8;                       // device payload width: 8, 4 or 0
    DevBuf d_payload, d_tags;
    bool on_device = false;              // filled by set_column_device
};

// What the file a directory entry's row is read from (<id>.json, file.go:711-749) looked like when it was read or
// stat-ed: the refresh of a resident keyspace keeps the rows of entries whose fingerprint still holds.
struct DocFp {
    enum State : u8 { ABSENT, DOC, UNREADABLE };  // no such file / read (the entry has a row) / there but not readable
    State state = ABSENT;
    bool racy = false;  // changed too close to the read for its timestamps to tell: treated as changed at the next check
    u64 ino = 0;
    i64 size = 0, mtime_ns = 0, ctime_ns = 0;
    static DocFp of(const struct stat& st);
    // the entry's row (or its absence) is still what a read would give
    bool holds(const DocFp& now) const {
        if (state == ABSENT) return now.state == ABSENT;
        return state == DOC && !racy && now.state == DOC && ino == now.ino && size == now.size && mtime_ns == now.mtime_ns && ctime_ns == now.ctime_ns;
    }
};

// One row run of a spliced table: rows [new_lo, new_lo + len) come from rows [src_lo, src_lo + len) of the old table or
// of the patch (the re-read documents).
struct SpliceRun { i64 new_lo; bool patch; i64 src_lo, len; };

struct Table {
    std::vector<Column> cols;
    i64 nrows = 0;
    i64 global_rows = 0;  // rows of the whole keyspace over all partitions (0 = not declared)
    bool sealed = false;
    // How the rows got in so far; which entry point may follow is decided by admit() alone
    enum class Fill : u8 {
        EMPTY,
        HOST_DOCS,       // append_json / load_dir / load_ndjson on host threads, or load_segment: rows staged, seal() uploads
        HOST_COLUMNS,    // set_column: rows staged, seal() uploads
        DEVICE_DOCS,     // the device shredder or a splice: columns final in HBM
        DEVICE_COLUMNS,  // set_column_device: columns in HBM, seal() checks that every one was set
    };
    Fill filled = Fill::EMPTY;
    bool rows_in_hbm() const { return filled == Fill::DEVICE_DOCS || filled == Fill::DEVICE_COLUMNS; }
    enum class Entry { ADD_COLUMN, APPEND_HOST, APPEND_DEVICE, SET_COLUMN, SET_COLUMN_DEVICE, LOAD_SEGMENT, SPLICE };
    void admit(Entry e, int col = -1) const;  // refuses `e` (on column `col`) when it may not follow what filled the table
    double shred_sec = 0, upload_sec = 0;
    i64 json_bytes = 0;

    // persistent segment (segment.cpp): when set, seal() writes the shredded columns to this file under this source tag
    std::string segment_out, segment_source;
    void write_segment() const { write_segment(segment_out, segment_source); }
    void write_segment(const std::string& file, const std::string& source) const;
    bool load_segment(const std::string& file, const std::string& source);
    void load_ndjson(const std::string& file, int threads);  // one document per line; threads as for load_dir

    // threads >= 0: host threads (0 = all cores); threads == -1: the device shredder (shred.cu)
    void append_json_device(const char* buf, const i64* offsets, i64 ndocs);
    // one document per line; offsets computed on the device.  `fill(lo, hi)` (optional) makes bytes [lo, hi) of text valid just
    // before they are copied: a file is read chunk by chunk while the chunks before it cross PCIe
    void append_ndjson_device(const char* text, i64 size, const std::function<void(i64, i64)>& fill = nullptr);
    void append_text_device(const char* buf, const i64* offsets, i64 ndocs, i64 text_size, const std::function<void(i64, i64)>& fill);
    int add_column(const std::string& path);
    int find_column(const std::string& path) const;
    void append_json(const char* buf, const i64* offsets, i64 ndocs, int threads);
    // entries / fps (optional): the directory entries in primary-key order and the fingerprint of what each one was read
    // from; the rows are those of the entries whose state is DOC, in that order
    void load_dir(const std::string& dir, int threads, std::vector<std::string>* entries = nullptr, std::vector<DocFp>* fps = nullptr);
    // the documents of the given directory entries (sorted names; <id>.json of each is read)
    void load_entries(const std::string& dir, const std::vector<std::string>& entries, int threads, std::vector<DocFp>* fps);
    // Fills this table (columns declared, nothing appended) with `runs` of rows of `old` and `patch` (null when no run
    // reads it), both sealed with their columns in HBM.  Dictionaries, statistics and widths are those a load of the
    // spliced rows gives.
    void splice(const Table& old, const Table* patch, const std::vector<SpliceRun>& runs);
    double splice_sec = 0;
    void set_column(int col, int width, const void* payload, const u8* tags, i64 nrows, const char* blob,
                    const i64* offs, i64 ndict);
    // The same for a column that already lives in device memory (caller-owned device pointers, copied device to
    // device): no host staging at all; statistics are computed by a kernel.  Every column of the table must then
    // be set this way.
    void set_column_device(int col, int width, const void* dev_payload, const u8* dev_tags, i64 nrows, const char* blob,
                           const i64* offs, i64 ndict);
    void build_dictionary(int col);  // local strings -> sorted dict, codes -> ranks
    // Dictionary exchange (multi-GPU), before seal: the column whose dictionary is exchanged, its dictionary built
    Column& exchange_column(int col);
    // The column's dictionary becomes `n` sorted strings that every partition agrees on (a superset of its own) /
    // the k-way merge of the given sorted dictionaries with its own
    void import_dictionary(int col, const char* blob, const i64* offs, i64 n);
    void merge_dictionaries(int col, int nparts, const char* const* blobs, const i64* const* offs, const i64* ns);
    // Replaces the column's (sorted) dictionary by a sorted superset and remaps the rows' ranks - staged on the host, or
    // already in HBM (device shredder, set_column_device).
    void adopt_dictionary(int col, std::vector<std::string>& global);
    void remap_ranks_device(int col, const std::vector<u32>& remap);  // rows of a column resident in HBM: rank -> remap[rank]
    void seal();
    int scan_bytes(int col) const;
    i64 padded_rows() const { return (nrows + ROW_PAD - 1) / ROW_PAD * ROW_PAD; }
    // A device column: padded_rows() (at least ROW_PAD) entries of `width` bytes, every byte `byte`, on stream `s` (MISSING
    // tags, zero payload); a payload of width 0 is a 256-byte stub
    DevBuf device_rows(int width, int byte, cudaStream_t s) const;
private:
    void check_column_args(int col, int width, i64 n) const;  // set_column / set_column_device
};

// The host shredder applied to selected documents (the device shredder's fix-up rows).  Per column: tags[n],
// payload[n] (STRING: index into strings).
struct HostShredOut {
    std::vector<u8> tags;
    std::vector<i64> payload;
    std::vector<std::string> strings;
};
void host_shred_docs(const std::vector<Column>& cols, const char* buf, const i64* offs, const i64* rows, i64 n,
                     std::vector<HostShredOut>& out);

// The file a keyspace directory entry's row is read from: <name minus its last extension>.json (file.go:757-761, 346).
std::string document_file(const std::string& entry);

std::vector<std::string> split_path(const std::string& path);
std::string join_path(const std::vector<std::string>& p, char sep);

}  // namespace n1
