// kernels.hpp — host launchers of the static kernels in kernels.cu
#pragma once
#include "common.hpp"
#include "final_group.hpp"

namespace n1 {

struct OpsArr {
    int n;
    int op[64];
};

// one DISTINCT aggregate: where its result words live and how its value component is packed in a set entry
struct DistinctDesc {
    int sid;           // entry set this aggregate reads (aggregates over the same operand share one)
    int numbers_only;  // COUNTN / SUM / AVG DISTINCT: only numeric entries count (COUNT: every entry)
    int w_cnt, w_ilo, w_ihi, w_neg, w_fsum, w_nflt;  // word indices (-1 = not needed)
    FinalComp value;   // the value component of a set entry
};
struct DistinctDescs {
    int n;
    DistinctDesc d[16];
};
// ---- device-side FinalGroup (final_group.hpp), see k_finalize_groups ------------------------------------------------------
// How the table is addressed: word w of slot i lives at acc[w * ws + i * ss] (word-major: ws = capacity, ss = 1).
// The partial tables the groups are read from: one (this rank's) or one per rank, combined word by word with the merge
// operations on the fly (IntermediateGroup fused into FinalGroup; peers are mapped over NVLink).
struct PeerTables {
    int n;
    const u64* acc[16];
    // peer merge only: a one-block kernel ahead of the finalisation waits until wait_flags[r] == wait_seq for all r < n (the
    // ranks' scans of this step are complete and visible); a peer that never arrives sets status[0] = 3 after ~10 s
    const u64* wait_flags;
    u64 wait_seq;
    int* status;
};
// Raises this rank's flag of step `seq` in every rank's flag row: peers[r][flags_word_off + (seq % 64) * nranks + rank] = seq.
void launch_peer_signal(u64* const* peers, int nranks, int rank, u64 flags_word_off, u64 seq, cudaStream_t s);
// One block that returns once flags[r] == seq for every r < nranks (bounded spin: status[0] = 3 after ~10 s).
void launch_peer_wait(const u64* flags, int nranks, u64 seq, int* status, cudaStream_t s);
// Finalises the live groups of slots [slot0, slot1) into compact flat arrays (n1gpu_result_fetch layout); *counter
// (zeroed by the caller) ends as the number of groups written; groups beyond out_cap are counted but not written.
void launch_finalize_groups(const FinalDesc& D, int kw, const u64* keys, const PeerTables& T, const OpsArr& ops, u64 ws, u64 ss, u64 slot0,
                            u64 slot1, unsigned long long* counter, u64 out_cap, u8* key_cls, i64* key_val, u8* agg_cls, i64* agg_val,
                            cudaStream_t s);
// ---- partitioned DISTINCT aggregation, second kernel (KernelPlan::part) --------------------------------------------------
// Records of partition `part` written by rank t: recs[t][part * part_cap .. + min(cur[t][part], part_cap)).
struct PartPeers {
    int n;
    const u32* recs[16];
    const u32* cur[16];
};
// One block per partition in [part0, part1): folds the records of all ranks into a shared-memory bitmap (group x value)
// and per-group row counters, then leaves the finished words of every group of the partition in the table acc[w * cap + slot]
// (slot = part << gbits | group): rows in word w_rows and, per DISTINCT aggregate of D, its count / exact split int sum /
// negative count.  value_is_int: the value component is a biased INT (else a string rank: counts only).
void launch_part_aggregate(const PartPeers& P, u64 part_cap, int part0, int part1, int gbits, int vbits, int w_rows, const DistinctDescs& D,
                           int value_is_int, i64 value_bias, u64* acc, u64 cap, cudaStream_t s);
void launch_distinct_finalize(const u64* set_keys, u64 set_cap, int set128, int abits, int key_bits, int kw, const u64* keys, u64 cap,
                              u64* acc, const DistinctDescs& D, cudaStream_t s);
void launch_merge_mailbox(const u64* mail, int nranks, u64 slot_base, u64 stride, u64 words, u64 seq, u64 cap, const OpsArr& ops,
                          u64* out_dev, u64* out_host, int* status, cudaStream_t s);
void launch_merge_words(const u64* all, int nranks, u64 cap, const OpsArr& ops, u64* out_dev, u64* out_host, cudaStream_t s);
void launch_init_words(u64* acc, u64 cap, const OpsArr& ops, cudaStream_t s);
void launch_fill_u64(u64* p, u64 n, u64 v, cudaStream_t s);
void launch_count_owners(int kw, const u64* keys, const u64* acc, u64 cap, int nranks, int gk_pos, int gk_bits,
                         unsigned long long* counts, cudaStream_t s);
void launch_export_records(int kw, const u64* keys, const u64* acc, u64 cap, int W, int nranks, int gk_pos, int gk_bits,
                           unsigned long long* cursor, u64* out, u64 out_cap, cudaStream_t s);
void launch_merge_records(int kw, u64* keys, u64* acc, u64 cap, const OpsArr& ops, const u64* recs, u64 n, int* status, cudaStream_t s);

}  // namespace n1
