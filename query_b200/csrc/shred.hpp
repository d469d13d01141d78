// shred.hpp — host launchers of the device-side JSON shredder (shred.cu)
#pragma once
#include "common.hpp"

namespace n1 {

// Flattened path trie (lives in global memory): node 0 is the document root.
struct ShredTrie {
    int nnodes, nkids;
    int kid_begin[64], kid_end[64], col[64];        // per node: its kids [begin,end) and the column bound to it (-1)
    int name_off[64], name_len[64], kid_node[64];   // per kid: field name in `names`, the node it leads to
    char names[2048];
};

void launch_shred_json(const unsigned char* buf, const i64* offs, i64 first, i64 ndocs, const ShredTrie* T, u8* const* tags, i64* const* payload,
                       int ncols, unsigned* fix_count, i64* fix_rows, i64 fix_cap, cudaStream_t s);
void launch_dict_insert(const unsigned char* buf, const unsigned char* extra, const u8* tags, const i64* payload, i64* slots, i64 nrows,
                        u64* keys, u64 cap, int* status, cudaStream_t s);
void launch_dict_collect(const u64* keys, u64 cap, unsigned* count, u64* out_slots, u64* out_refs, u64 out_cap, cudaStream_t s);
// NDJSON text resident in HBM -> offsets of its documents (see shred.cu): counts per 256-byte segment, their exclusive scan
// (first[nseg] = number of documents), the offsets themselves; the caller appends offs[ndocs] = size
i64 ndjson_segments(i64 size);
void launch_ndjson_count(const unsigned char* text, i64 size, unsigned* counts, cudaStream_t s);
i64 ndjson_scan_tiles(i64 nseg);  // launch_ndjson_scan needs (tiles + 1) x 8 bytes of device scratch
void launch_ndjson_scan(const unsigned* counts, i64 nseg, i64* first, i64* tile_scratch, cudaStream_t s);
void launch_ndjson_write(const unsigned char* text, i64 size, const i64* first, i64* offs, cudaStream_t s);
void launch_gather_offsets(const i64* offs, const i64* rows, i64 n, i64* out, cudaStream_t s);
void launch_rank_remap(const u8* tags, i64* pay8, u32* pay4, i64 nrows, const u32* remap, u32 n, cudaStream_t s);
// 4-byte string ranks -> 8-byte payloads, zero-extended (an 8-byte column stores a rank as it is)
void launch_widen_ranks(const u32* pay4, i64* pay8, i64 nrows, cudaStream_t s);
void launch_dict_ranks(const u64* slot_of_rank, u64 n, u32* rank, cudaStream_t s);
void launch_dict_remap(const u8* tags, const i64* slots, i64* payload, u32* out32, i64 nrows, const u32* rank, cudaStream_t s);
void launch_col_stats(const u8* tags, const i64* payload, i64 nrows, u64* stats, cudaStream_t s);
void launch_canon_floats(u8* tags, i64* payload, i64 nrows, cudaStream_t s);
void launch_patch(u8* tags, i64* payload, const i64* rows, const u8* ptags, const i64* ppay, i64 n, cudaStream_t s);

// The row map of a spliced column, in device memory: run k covers new rows [new_lo[k], new_lo[k + 1]) (new_lo[nruns] = nrows)
// and reads them from row src_lo[k] on of the old column, or of the patch column when bit 63 of src_lo[k] is set.
struct SpliceRuns { const i64* new_lo; const i64* src_lo; i64 nruns, nrows; };
// ranks of the old dictionary used by the kept rows (a bitmap of ceil(ndict / 32) words, zeroed by the caller) and the
// classes of those rows (OR-ed into *class_mask)
void launch_splice_used(const SpliceRuns& r, const u8* tags, const i64* pay8, const u32* pay4, u32* used, u64* class_mask, cudaStream_t s);
// writes all `padded` rows of the new column; a source or target payload pointer is null at that width (0: no payload)
void launch_splice_gather(const SpliceRuns& r, i64 padded, const u8* o_tags, const i64* o_pay8, const u32* o_pay4, const u32* o_remap,
                          const u8* p_tags, const i64* p_pay8, const u32* p_pay4, const u32* p_remap, u8* tags, i64* pay8, u32* pay4, cudaStream_t s);

}  // namespace n1
