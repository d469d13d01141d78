// codegen.hpp — compiles a bound Filter + Group chain into (a) the CUDA source of one specialised
// sm_100a scan kernel built from n1ql_device.cuh and (b) the layout needed to merge and finalise the
// accumulator words it produces.
#pragma once
#include <string>
#include <vector>

#include "expr.hpp"
#include "table.hpp"

namespace n1 {

enum : int { MODE_UNGROUPED = 0, MODE_DENSE = 1, MODE_HASH64 = 2, MODE_HASH128 = 3 };
enum : int { CK_CNT = 0, CK_WIDE = 1, CK_MM32 = 2, CK_OR32 = 3, CK_64 = 4, CK_WIDE1 = 5 };
// threads per block of the partitioning kernel (KernelPlan::part), one block per SM.  Two 512-thread blocks with half
// the bins each lost (config 4, 200 M rows: 1.59 -> 1.78 ms; four 256-thread blocks 2.55 ms; DESIGN.md section 9)
constexpr int PART_THREADS = 1024;

// One bit-packed component: a group-key value or the value of a DISTINCT entry.
struct PackComp {
    u32 mask = 0;
    std::vector<int> classes;  // class index -> class
    int cbits = 0, pbits = 0;
    // "offset" packing (one field, no class bits): when a single class carries a bounded payload (a dictionary rank or a
    // ranged int) the classes without payload take the values 0 .. nfree-1 and the payload class nfree + payload;
    // `classes` then lists the payload-free classes first and the payload class last.  A string key with NULL and
    // MISSING groups packs into bits_for(2 + ndict) bits instead of 2 + bits_for(ndict): a 4x smaller direct table.
    int nfree = -1;            // >= 0: offset packing with this many payload-free classes
    bool biased = false;       // INT payload stored as (v - bias)
    i64 bias = 0;
    int dict_col = -1;         // STRING payload = rank in this column's dictionary
    u64 range = 0;             // offset packing: payload values are 0 .. range-1
    int bits() const { return cbits + pbits; }
};

// IN evaluated through a device-resident set (NqInSet, n1ql_value.cuh) instead of one in_arg per element: see
// in_takes_set (expr.hpp).  The kernel text names only the set's slot, so every binding of a statement shares one cubin.
// A chain has at most NQ_MAX_INSETS of them.
struct InSet {
    std::vector<u32> bits;         // STRING: bitmap over the operand column's dictionary ranks
    std::vector<u64> ikeys, fkeys; // INT / FLOAT hash tables (all ones = empty slot)
    u32 flags = 0;                 // INSET_*
};

// One aggregate: what finalises it (FinalAgg, final_group.hpp) and what only the code generator needs
struct AggPlan : FinalAgg {
    bool star = false;
    std::string text;          // the aggregate's Stringer text (the key of the "aggregates" attachment)
    u32 opmask = 0;            // classes the operand may take
    int distinct_id = -1;      // index among DISTINCT aggregates
    PackComp dcomp;
};

struct KernelPlan {
    int mode = MODE_UNGROUPED;
    std::vector<int> word_ops;   // accumulator words per group
    std::vector<bool> word_count;  // word only ever receives +1 (a row counter): bounded by the rows one block scans
    std::vector<i64> word_lo, word_hi;  // min/max words: proven value range (lo > hi: unknown)
    // Physical layout of the group table.  The words above are LOGICAL (what the aggregates read); in the HBM modes
    // behind the front cache two row counters share one 64-bit physical word as 32-bit fields when the row bound proves
    // that neither can overflow: a cache miss then costs one L2 reduction for both.  Everything that moves or merges
    // table state (init, export, merge, all-reduce) works on the physical words; only finalize() decodes the fields.
    std::vector<int> phys_ops;           // op of every physical word (what Query::ops holds)
    std::vector<int> phys_of, shift_of;  // logical word -> physical word, bit offset of its field
    std::vector<int> bits_of;            // field width (64 = the whole word)
    // A COUNT(x) counter over a column whose values are mostly present counts the rows where x is MISSING / NULL instead
    // (the rarer event: fewer shared-memory atomics per row); finalize() reads it as rows-in-group minus the word.
    std::vector<bool> word_complement;
    std::vector<int> complement_agg;     // complemented word -> the aggregate whose (plain column) operand it counts
    int w_rows = -1;                     // the rows-per-group word (-1: none)
    std::vector<PackComp> keys;
    int key_bits = 0;
    i64 dense_slots = 0;
    // shared-memory dense tables index slots by the mixed-radix number of the key components (TPC-H Q1: 3 x 2 = 6 slots
    // instead of the 2^3 = 8 of the bit-packed key); dense_dom[i] = values component i takes (empty: slot == packed key)
    std::vector<u64> dense_dom;
    bool dense_global = false;   // MODE_DENSE whose table is too large for shared memory: direct-indexed in HBM (slot = packed
                                 // key, no key array, no probing) behind the shared-memory front cache of the hash mode
    bool dense_priv = false;     // tiny dense table: one private copy per THREAD in shared memory (no atomics at all)
    bool pdl = false;            // launched with programmatic stream serialization (ungrouped scans)
    int min_blocks = 0;          // resident blocks per SM in __launch_bounds__ (0: none)
    int dyn_smem = 0;            // dynamic shared memory the kernel is launched with
    int block = 256;             // threads per block (a block scans block * 4 rows per iteration)
    bool cache_key32 = false;    // front-cache keys are u32, direct-mapped (packed key <= 31 bits)
    int cache_slots = 0;         // HASH64: slots of the per-block shared-memory front cache (0 = none)
    // front-cache cell of every word: kind (CK_*) and index of its first cell among the 32-bit / 64-bit cell arrays
    std::vector<int> cell_kind, cell_idx;
    // two neighbouring ranged min / max cells (MIN(x) and MAX(x)) interleaved per slot - [first, second] at 2 * slot - so
    // that ONE 64-bit shared-memory load fetches both for the read-before-atomic check: 0 none, 1 first of a pair, 2 second
    std::vector<int> cell_pair;
    int cache_n32 = 0, cache_n64 = 0;
    std::vector<AggPlan> aggs;
    int ndistinct = 0, abits = 0, entry_bits = 0;
    std::vector<bool> set_any;   // DISTINCT entry set -> holds every value > NULL (else numbers only)
    bool set128 = false;
    int set_passes = 1;          // bitmap beyond what the L2 keeps: scan passes, each filling one L2-resident slice of it
    bool set_bitmap = false;     // DISTINCT entries are few bits: the set is a bitmap indexed by the entry (no hashing)
    // Partitioned DISTINCT aggregation (config 4's shape: a direct-indexed table of many groups, ONE distinct operand of few
    // bits, and no other per-row accumulator than the row count).  Instead of one scattered L2 atomic per row for the
    // DISTINCT bitmap and one for the group table, a first kernel (part_source) only filters, packs (group, value) into a
    // 4-byte record and radix-partitions the records by the high bits of the group key through shared-memory bins; a second
    // (static) kernel gives every partition to one block, whose share of the bitmap and of the counters fits shared memory,
    // and leaves the finished accumulator words in the group table.  part_* describe the record.
    bool part = false;
    std::string part_source;     // the partitioning kernel (entry nq_scan, PART_THREADS threads)
    int part_bits = 0;           // partitions = 2^part_bits, taken from the top of the packed group key
    int part_gbits = 0;          // record bits [0, gbits): group key inside its partition; bit gbits: has a value
    int part_vbits = 0;          // record bits above: the packed DISTINCT value
    int part_bincap = 48;        // records a block stages per partition and round in shared memory
    int part_smem = 0;           // dynamic shared memory of the partitioning kernel
    // payloads of constants / bound parameters, passed to the kernel as NqParams::cst (the source only names the slot)
    std::vector<i64> consts;
    std::vector<InSet> in_sets;  // NqParams::inset[k]
    std::vector<int> used_cols;
    int scan_bytes_per_row = 0;
    std::string source;
    i64 est_groups = 0;          // estimate used to size the hash table
};

// where may be null; keys/aggs are bound + analysed expressions.  total_rows_bound: an upper bound on
// the number of rows any single accumulator may see (all ranks), for the no-overflow proof of int sums.
KernelPlan generate_kernel(const Table& t, const Expr* where, const std::vector<ExprP>& keys,
                           const std::vector<ExprP>& aggs, const std::vector<std::string>& agg_texts,
                           double total_rows_bound);

}  // namespace n1
