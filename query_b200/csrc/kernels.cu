// kernels.cu — the static (query-independent) sm_100a kernels of libn1gpu.so: accumulator-table
// initialisation, table / DISTINCT set -> record compaction with owner bucketing (the export side of the
// multi-GPU IntermediateGroup exchange, also the compaction step of finalisation), record -> table merging
// (CumulateIntermediate: algebra/agg_*.go, execution/group_intermediate.go:56-104), the element-wise merges of
// small-state chains, the device-side ComputeFinal of DISTINCT aggregates and FinalGroup over HBM tables
// (k_finalize_groups, through final_group.hpp: the one restatement of ComputeFinal, shared with the host finalisation).
#include <algorithm>

#include "kernels.hpp"
#include "n1ql_device.cuh"

namespace n1 {

__global__ void k_init_words(u64* acc, u64 cap, OpsArr ops) {
    u64 total = cap * (u64)ops.n;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (u64)gridDim.x * blockDim.x)
        acc[i] = word_identity(ops.op[i / cap]);
}

__global__ void k_fill_u64(u64* p, u64 n, u64 v) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) p[i] = v;
}

__device__ __forceinline__ void extract_bits(u64 lo, u64 hi, int pos, int n, u64& olo, u64& ohi) {
    // bits [pos, pos+n) of the 128-bit (hi:lo), n <= 127
    unsigned __int128 v = ((unsigned __int128)hi << 64) | lo;
    v >>= pos;
    if (n < 128) v &= (((unsigned __int128)1) << n) - 1;
    olo = (u64)v;
    ohi = (u64)(v >> 64);
}

__device__ __forceinline__ int owner_of(u64 lo, u64 hi, int nranks) {
    return nranks <= 1 ? 0 : (int)(mix64(lo ^ mix64(hi ^ 0x9e3779b97f4a7c15ULL)) % (u64)nranks);
}

// key of slot i and whether the slot holds a group.  kw: 0 dense (key = index, live iff word 0 > 0),
// 1: u64 keys, 2: 128-bit keys, 3: single ungrouped slot (always live)
__device__ __forceinline__ bool slot_key(int kw, const u64* keys, const u64* acc, u64 i, u64& lo, u64& hi) {
    if (kw == 0) { lo = i; hi = 0; return acc[i] != 0; }
    if (kw == 1) { lo = keys[i]; hi = 0; return lo != NQ_U64_MAX; }
    if (kw == 2) { lo = keys[2 * i]; hi = keys[2 * i + 1]; return !(lo == NQ_U64_MAX && hi == NQ_U64_MAX); }
    lo = 0; hi = 0; return true;
}

// pass 1: count live slots per owner.  gk_pos/gk_bits: where the group key sits inside the stored key
// (DISTINCT entries embed it after the aggregate id; group tables store it at bit 0).
// kw == 4: `keys` is a DISTINCT bitmap of `cap` bits (a multiple of 64); bit e set = entry e present.
// Warp-aggregated cursor: the lanes of a warp that bump the same counter elect a leader, which adds their number once;
// every lane gets its own position.  With 10^6 live slots and <= 8 owners a plain atomicAdd per slot serialises on 8
// addresses.  Called by all 32 lanes (lanes with nothing to claim pass live = false).
__device__ __forceinline__ u64 warp_claim(unsigned long long* counters, int owner, bool live) {
    const int lane = threadIdx.x & 31;
    const unsigned m = __match_any_sync(0xffffffffu, live ? owner : -1);
    const int leader = __ffs(m) - 1;
    unsigned long long base = 0;
    if (live && lane == leader) base = atomicAdd(&counters[owner], (unsigned long long)__popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    return base + (u64)__popc(m & ((1u << lane) - 1u));
}

__global__ void k_count_owners(int kw, const u64* keys, const u64* acc, u64 cap, int nranks, int gk_pos, int gk_bits,
                               unsigned long long* counts) {
    const u64 stride = (u64)gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31;
    if (kw == 4) {
        const u64 nw = cap >> 6;
        for (u64 w0 = (u64)blockIdx.x * blockDim.x + (threadIdx.x & ~31); w0 < nw; w0 += stride) {  // warp-uniform trip count
            const u64 w = w0 + lane;
            u64 bits = w < nw ? keys[w] : 0;
            if (nranks <= 1) {
                const unsigned long long n = (unsigned long long)__popcll(bits);
                const unsigned long long tot = warp_reduce_word<OP_ADD_U64>(n);
                if (lane == 0 && tot) atomicAdd(&counts[0], tot);
                continue;
            }
            while (__any_sync(0xffffffffu, bits != 0)) {
                const bool live = bits != 0;
                int owner = 0;
                if (live) {
                    const u64 lo = (w << 6) | (u64)(__ffsll((long long)bits) - 1);
                    bits &= bits - 1;
                    u64 glo, ghi;
                    extract_bits(lo, 0, gk_pos, gk_bits, glo, ghi);
                    owner = owner_of(glo, ghi, nranks);
                }
                warp_claim(counts, owner, live);
            }
        }
        return;
    }
    for (u64 i0 = (u64)blockIdx.x * blockDim.x + (threadIdx.x & ~31); i0 < cap; i0 += stride) {
        const u64 i = i0 + lane;
        u64 lo = 0, hi = 0;
        const bool live = i < cap && slot_key(kw, keys, acc, i, lo, hi);
        int owner = 0;
        if (live) {
            u64 glo, ghi;
            extract_bits(lo, hi, gk_pos, gk_bits, glo, ghi);
            owner = owner_of(glo, ghi, nranks);
        }
        warp_claim(counts, owner, live);
    }
}

// pass 2: write records [lo, hi, words...] at cursor[owner]++ (cursor pre-loaded with bucket offsets).
__global__ void k_export_records(int kw, const u64* keys, const u64* acc, u64 cap, int W, int nranks, int gk_pos, int gk_bits,
                                 unsigned long long* cursor, u64* out, u64 out_cap) {
    const int rw = 2 + W;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31;
    if (kw == 4) {
        const u64 nw = cap >> 6;
        for (u64 w0 = (u64)blockIdx.x * blockDim.x + (threadIdx.x & ~31); w0 < nw; w0 += stride) {
            const u64 w = w0 + lane;
            u64 bits = w < nw ? keys[w] : 0;
            while (__any_sync(0xffffffffu, bits != 0)) {
                const bool live = bits != 0;
                int owner = 0;
                u64 lo = 0;
                if (live) {
                    lo = (w << 6) | (u64)(__ffsll((long long)bits) - 1);
                    bits &= bits - 1;
                    u64 glo, ghi;
                    extract_bits(lo, 0, gk_pos, gk_bits, glo, ghi);
                    owner = owner_of(glo, ghi, nranks);
                }
                const u64 at = warp_claim(cursor, owner, live);
                if (live && at < out_cap) { out[at * rw] = lo; out[at * rw + 1] = 0; }
            }
        }
        return;
    }
    for (u64 i0 = (u64)blockIdx.x * blockDim.x + (threadIdx.x & ~31); i0 < cap; i0 += stride) {
        const u64 i = i0 + lane;
        u64 lo = 0, hi = 0;
        const bool live = i < cap && slot_key(kw, keys, acc, i, lo, hi);
        int owner = 0;
        if (live) {
            u64 glo, ghi;
            extract_bits(lo, hi, gk_pos, gk_bits, glo, ghi);
            owner = owner_of(glo, ghi, nranks);
        }
        const u64 at = warp_claim(cursor, owner, live);
        if (!live || at >= out_cap) continue;
        u64* r = out + at * rw;
        r[0] = lo; r[1] = hi;
        for (int w = 0; w < W; ++w) r[2 + w] = acc[(u64)w * cap + i];
    }
}

// merge: records -> table (IntermediateGroup).  kw as above.
__global__ void k_merge_records(int kw, u64* keys, u64* acc, u64 cap, OpsArr ops, const u64* __restrict__ recs, u64 n, int* status) {
    const int rw = 2 + ops.n;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const u64* r = recs + i * rw;
        if (kw == 4) {  // DISTINCT bitmap: the entry is its own index
            if (r[0] >= cap || r[1] != 0) { status[0] = 1; continue; }
            atomicOr(&keys[r[0] >> 6], 1ULL << (r[0] & 63));
            continue;
        }
        i64 slot;
        if (kw == 0) slot = (i64)r[0];
        else if (kw == 1) slot = table_insert64(keys, cap - 1, r[0], nullptr);
        else if (kw == 2) slot = table_insert128((ulonglong2*)keys, cap - 1, r[0], r[1], nullptr);
        else slot = 0;
        if (slot < 0 || (u64)slot >= cap) { status[0] = 1; continue; }
        for (int w = 0; w < ops.n; ++w) {
            u64 v = r[2 + w];
            if (v != word_identity(ops.op[w])) atomic_word_dyn(ops.op[w], &acc[(u64)w * cap + (u64)slot], v);
        }
    }
}

// DISTINCT finalisation (ComputeFinal of count/countn/sum/avg DISTINCT: algebra/agg_*_distinct.go): every entry of the
// (aggregate, group, value) set adds 1 to its group's distinct count and, for SUM/AVG, its value to the group's exact
// split integer sum / float sum.  kw: how the group slot is found (3 ungrouped, 0 dense, 1 / 2 hash 64 / 128).
__device__ __forceinline__ void distinct_entry(u64 lo, u64 hi, int abits, int key_bits, int kw, const u64* __restrict__ keys, u64 cap,
                                               u64* acc, const DistinctDescs& D) {
    {
        unsigned __int128 v = ((unsigned __int128)hi << 64) | lo;
        const int sid = (int)take_bits(v, abits);
        const u64 klo = take_bits(v, key_bits < 64 ? key_bits : 64);
        const u64 khi = key_bits > 64 ? take_bits(v, key_bits - 64) : 0;
        i64 slot;
        if (kw == 3) slot = 0;
        else if (kw == 0) slot = (i64)klo;
        else if (kw == 1) slot = table_find64(keys, cap - 1, klo);
        else slot = table_find128((const ulonglong2*)keys, cap - 1, klo, khi);
        if (slot < 0 || (u64)slot >= cap) return;  // group owned by another rank
        bool decoded = false;
        Val val{C_MISSING, 0};
        for (int a = 0; a < D.n; ++a) {
            const DistinctDesc& d = D.d[a];
            if (d.sid != sid) continue;
            if (!decoded) {  // the value component is packed identically for every aggregate of the set
                val = decode_comp(d.value, v);
                decoded = true;
            }
            if (d.numbers_only && !(val.c == C_INT || val.c == C_FLOAT)) continue;
            atomicAdd(&acc[(u64)d.w_cnt * cap + (u64)slot], 1ULL);
            if (val.c == C_INT && d.w_ilo >= 0) {
                const i64 x = val.b;
                atomicAdd(&acc[(u64)d.w_ilo * cap + (u64)slot], (u64)x & 0xffffffffULL);
                atomicAdd(&acc[(u64)d.w_ihi * cap + (u64)slot], (u64)(x >> 32));
                if (x < 0) atomicAdd(&acc[(u64)d.w_neg * cap + (u64)slot], 1ULL);
            } else if (val.c == C_FLOAT && d.w_fsum >= 0) {
                atomicAdd((double*)&acc[(u64)d.w_fsum * cap + (u64)slot], __longlong_as_double(val.b));
                atomicAdd(&acc[(u64)d.w_nflt * cap + (u64)slot], 1ULL);
            }
        }
    }
}
// set_kind: 0 hash set of 64-bit entries, 1 of 128-bit entries, 2 bitmap of set_cap bits
__global__ void k_distinct_finalize(const u64* __restrict__ set_keys, u64 set_cap, int set_kind, int abits, int key_bits, int kw,
                                    const u64* __restrict__ keys, u64 cap, u64* acc, DistinctDescs D) {
    if (set_kind == 2) {
        for (u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x; w < (set_cap >> 6); w += (u64)gridDim.x * blockDim.x) {
            u64 bits = set_keys[w];
            while (bits) {
                const u64 lo = (w << 6) | (u64)(__ffsll((long long)bits) - 1);
                bits &= bits - 1;
                distinct_entry(lo, 0, abits, key_bits, kw, keys, cap, acc, D);
            }
        }
        return;
    }
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < set_cap; i += (u64)gridDim.x * blockDim.x) {
        u64 lo, hi;
        if (set_kind == 1) { lo = set_keys[2 * i]; hi = set_keys[2 * i + 1]; if (lo == NQ_U64_MAX && hi == NQ_U64_MAX) continue; }
        else { lo = set_keys[i]; hi = 0; if (lo == NQ_U64_MAX) continue; }
        distinct_entry(lo, hi, abits, key_bits, kw, keys, cap, acc, D);
    }
}

// Small-state IntermediateGroup merge: all[r][w][slot] (the accumulator words of every rank, gathered by one
// all_gather) folded over ranks in rank order (deterministic) into out_dev / out_host (zero-copy result).
__global__ void k_merge_words(const u64* __restrict__ all, int nranks, u64 cap, OpsArr ops, u64* out_dev, u64* out_host) {
    const u64 n = cap * (u64)ops.n;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const int op = ops.op[i / cap];
        u64 v = all[i];
        for (int r = 1; r < nranks; ++r) v = word_combine(op, v, all[(u64)r * n + i]);
        out_dev[i] = v;
        if (out_host) out_host[i] = v;
    }
}

// Mailbox merge (the receive side of the scan kernel's fused all-gather): waits until every rank's words of
// this step have landed (sequence flag, acquire at system scope; bounded spin -> status 3 on timeout), then
// folds them in rank order.  One block; runs on this GPU while the senders are kernels on OTHER GPUs.
__global__ void k_merge_mailbox(const u64* mail, int nranks, u64 slot_base, u64 stride, u64 words, u64 seq, u64 cap, OpsArr ops,
                                u64* out_dev, u64* out_host, int* status) {
    __shared__ int s_ok;
    if (threadIdx.x == 0) s_ok = 1;
    __syncthreads();
    if ((int)threadIdx.x < nranks) {
        const u64* flag = mail + slot_base + (u64)threadIdx.x * stride + words;
        u64 v = 0;
        const long long t0 = clock64();
        for (;;) {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
            if (v == seq) break;
            if (clock64() - t0 > 20000000000LL) { s_ok = 0; break; }  // ~10 s at 2 GHz: a peer never arrived
            __nanosleep(200);
        }
    }
    __syncthreads();
    if (!s_ok) { if (threadIdx.x == 0) status[0] = 3; return; }
    for (u64 i = threadIdx.x; i < words; i += blockDim.x) {
        const int op = ops.op[i / cap];
        u64 v = __ldcg(&mail[slot_base + i]);
        for (int r = 1; r < nranks; ++r) v = word_combine(op, v, __ldcg(&mail[slot_base + (u64)r * stride + i]));
        out_dev[i] = v;
        if (out_host) out_host[i] = v;
    }
}

// ---- FinalGroup on the device -------------------------------------------------------------------------------------------
// One thread per table slot: the slot's words folded over the partial tables, live groups compacted into flat arrays
// through a warp-aggregated cursor and finalised by final_group (final_group.hpp, the restatement of ComputeFinal and of
// the key decoding that the host finalisation shares; execution/group_final.go:55-118 sends one item per group).  Strings
// leave as (dictionary column << 40 | rank); the host resolves them.
__global__ void __launch_bounds__(256) k_finalize_groups(const FinalDesc D, int kw, const u64* __restrict__ keys, const PeerTables T, const OpsArr ops,
                                                         u64 ws, u64 ss, u64 slot0, u64 slot1, unsigned long long* counter, u64 out_cap,
                                                         u8* key_cls, i64* key_val, u8* agg_cls, i64* agg_val) {
    const int lane = threadIdx.x & 31;
    const u64 span = slot1 - slot0;
    const u64 rounds = (span + (u64)gridDim.x * blockDim.x - 1) / ((u64)gridDim.x * blockDim.x);
    for (u64 r = 0; r < rounds; ++r) {  // warp-uniform trip count (the cursor below is claimed per warp)
        const u64 i = slot0 + r * (u64)gridDim.x * blockDim.x + (u64)blockIdx.x * blockDim.x + threadIdx.x;
        bool live = i < slot1;
        u64 klo = 0, khi = 0;
        u64 pw[64];
        if (live) {
            if (kw == 1) { klo = keys[i]; live = klo != NQ_U64_MAX; }
            else if (kw == 2) { klo = keys[2 * i]; khi = keys[2 * i + 1]; live = !(klo == NQ_U64_MAX && khi == NQ_U64_MAX); }
            else if (kw == 0) klo = i;
        }
        if (live) {
            for (int P = 0; P < D.PW; ++P) {
                u64 v = __ldcg(&T.acc[0][(u64)P * ws + i * ss]);
                for (int t = 1; t < T.n; ++t) v = word_combine(ops.op[P], v, __ldcg(&T.acc[t][(u64)P * ws + i * ss]));
                pw[P] = v;
            }
            if (kw == 0) {  // direct-indexed: a slot holds a group iff its row counter (logical word 0) is not zero
                const u64 v = pw[D.phys_of[0]];
                live = (D.bits_of[0] == 64 ? v : (v >> D.shift_of[0]) & 0xffffffffULL) != 0;
            }
        }
        const unsigned m = __ballot_sync(0xffffffffu, live);
        if (m == 0) continue;
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(counter, (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (!live) continue;
        const u64 g = base + (u64)__popc(m & ((1u << lane) - 1u));
        if (g >= out_cap) continue;
        final_group(D, D.keys, D.nkeys, klo, khi, pw, key_cls + g * D.nkeys, key_val + g * D.nkeys, agg_cls + g * D.naggs,
                    agg_val + g * D.naggs);
    }
}

// ---- partitioned DISTINCT aggregation: one partition per block, state in shared memory -----------------------------------
// (replaces, for this shape, one scattered L2 atomic per row on the DISTINCT bitmap + one on the group table + the per-entry
// atomics of k_distinct_finalize: InitialGroup's per-row work of execution/group_initial.go:56-108 with the value.Set of
// algebra/agg_util.go:30-101 as bits, and ComputeFinal of algebra/agg_count_distinct.go / agg_sum_distinct.go per group)
__global__ void __launch_bounds__(1024, 1) k_part_aggregate(const PartPeers P, u64 part_cap, int part0, int part1, int gbits, int vbits, int w_rows,
                                                            const DistinctDescs D, int value_is_int, i64 value_bias, u64* acc, u64 cap) {
    extern __shared__ u32 s_pa[];
    const u32 G = 1u << gbits;
    const int wshift = vbits > 5 ? vbits - 5 : 0;   // 32-bit bitmap words per group = 1 << wshift
    const u32 WPG = 1u << wshift;
    u32* const s_cnt = s_pa;       // [G] rows per group
    u32* const s_bm = s_pa + G;    // [G][WPG] values seen per group
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const u32 gmask = G - 1;
    for (int part = part0 + blockIdx.x; part < part1; part += gridDim.x) {
        for (u32 i = threadIdx.x; i < G * (1 + WPG); i += blockDim.x) s_pa[i] = 0;
        __syncthreads();
        for (int t = 0; t < P.n; ++t) {
            const u64 n = min((u64)__ldcg(&P.cur[t][part]), part_cap);
            const u32* __restrict__ r = P.recs[t] + (u64)part * part_cap;
            for (u64 i0 = threadIdx.x; i0 < n; i0 += (u64)blockDim.x * 8) {
                u32 rec[8];  // eight loads in flight per thread before the first is used
#pragma unroll
                for (int k = 0; k < 8; ++k) { const u64 i = i0 + (u64)k * blockDim.x; rec[k] = i < n ? __ldcg(&r[i]) : 0u; }
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    if (i0 + (u64)k * blockDim.x >= n) break;
                    const u32 g = rec[k] & gmask;
                    atomicAdd(&s_cnt[g], 1u);
                    if ((rec[k] >> gbits) & 1u) {
                        const u32 v = rec[k] >> (gbits + 1);
                        atomicOr(&s_bm[(g << wshift) + (v >> 5)], 1u << (v & 31));
                    }
                }
            }
        }
        __syncthreads();
        // a warp per group: lane k folds bitmap words k, k + 32, ... (bank == lane), then a shuffle reduction
        // codes below this are negative values (unsigned: -INT64_MIN does not fit an i64)
        const u64 neg_below = value_is_int && value_bias < 0 ? 0ULL - (u64)value_bias : 0;
        for (u32 g = warp; g < G; g += nwarps) {
            u64 cnt = 0, code_sum = 0, nneg = 0;
            for (u32 k = lane; k < WPG; k += 32) {
                const u32 w = s_bm[(g << wshift) + k];
                if (!w) continue;
                cnt += __popc(w);
                if (value_is_int) {
                    // sum of the set bit positions: 32 * k * popc + sum over j of 2^j * popc(w & bits whose position has bit j)
                    code_sum += (u64)(32u * k) * __popc(w) + __popc(w & 0xaaaaaaaau) + 2u * __popc(w & 0xccccccccu) + 4u * __popc(w & 0xf0f0f0f0u) +
                                8u * __popc(w & 0xff00ff00u) + 16u * __popc(w & 0xffff0000u);
                    const u64 lo = 32u * k;
                    if (neg_below > lo) nneg += neg_below >= lo + 32 ? (u64)__popc(w) : (u64)__popc(w & ((1u << (u32)(neg_below - lo)) - 1u));
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
                code_sum += __shfl_xor_sync(0xffffffffu, code_sum, o);
                nneg += __shfl_xor_sync(0xffffffffu, nneg, o);
            }
            if (lane == 0) {
                const u64 slot = ((u64)part << gbits) | g;
                acc[(u64)w_rows * cap + slot] = s_cnt[g];
                const __int128 total = (__int128)value_bias * (__int128)cnt + (__int128)code_sum;
                for (int a = 0; a < D.n; ++a) {
                    const DistinctDesc& d = D.d[a];
                    acc[(u64)d.w_cnt * cap + slot] = cnt;
                    if (d.w_ilo >= 0) {
                        acc[(u64)d.w_ilo * cap + slot] = (u64)total & 0xffffffffULL;
                        acc[(u64)d.w_ihi * cap + slot] = (u64)(i64)(total >> 32);
                        acc[(u64)d.w_neg * cap + slot] = nneg;
                    }
                }
            }
        }
        __syncthreads();
    }
}
void launch_part_aggregate(const PartPeers& P, u64 part_cap, int part0, int part1, int gbits, int vbits, int w_rows, const DistinctDescs& D,
                           int value_is_int, i64 value_bias, u64* acc, u64 cap, cudaStream_t s) {
    if (part1 <= part0) return;
    const size_t smem = ((size_t)4 << gbits) * (1 + ((size_t)1 << (vbits > 5 ? vbits - 5 : 0)));
    static size_t configured = 0;
    if (smem > configured) { CK(cudaFuncSetAttribute(k_part_aggregate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); configured = smem; }
    const int grid = std::min(part1 - part0, 148 * (smem <= 100 * 1024 ? 2 : 1));
    k_part_aggregate<<<grid, 1024, smem, s>>>(P, part_cap, part0, part1, gbits, vbits, w_rows, D, value_is_int, value_bias, acc, cap);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}

static int grid_for(u64 n) {
    u64 g = (n + 255) / 256;
    if (g < 1) g = 1;
    if (g > 148 * 16) g = 148 * 16;
    return (int)g;
}

void launch_distinct_finalize(const u64* set_keys, u64 set_cap, int set128, int abits, int key_bits, int kw, const u64* keys, u64 cap,
                              u64* acc, const DistinctDescs& D, cudaStream_t s) {
    k_distinct_finalize<<<grid_for(set128 == 2 ? set_cap >> 6 : set_cap), 256, 0, s>>>(set_keys, set_cap, set128, abits, key_bits, kw, keys, cap, acc, D);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
// One block: returns once every rank's flag of this step has arrived (acquire at system scope; bounded spin -> status 3).
// A kernel of its own, so that the only thing that ever spins on a GPU is one block - the finalisation that follows it in
// stream order starts with the tables complete and visible.
__global__ void k_peer_wait(const u64* flags, int nranks, u64 seq, int* status) {
    if ((int)threadIdx.x < nranks) {
        u64 v = 0;
        const long long t0 = clock64();
        for (;;) {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flags + threadIdx.x) : "memory");
            if (v == seq) break;
            if (clock64() - t0 > 20000000000LL) { status[0] = 3; break; }  // ~10 s: a peer never arrived
            __nanosleep(200);
        }
    }
}
__global__ void k_peer_signal(u64* const* peers, int nranks, int rank, u64 flags_word_off, u64 seq) {
    if ((int)threadIdx.x < nranks) {
        __threadfence_system();
        u64* flag = peers[threadIdx.x] + flags_word_off + (seq % 64) * (u64)nranks + (u64)rank;
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flag), "l"(seq) : "memory");
    }
}
void launch_peer_wait(const u64* flags, int nranks, u64 seq, int* status, cudaStream_t s) {
    k_peer_wait<<<1, 32, 0, s>>>(flags, nranks, seq, status);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_peer_signal(u64* const* peers, int nranks, int rank, u64 flags_word_off, u64 seq, cudaStream_t s) {
    k_peer_signal<<<1, 64, 0, s>>>(peers, nranks, rank, flags_word_off, seq);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_finalize_groups(const FinalDesc& D, int kw, const u64* keys, const PeerTables& T, const OpsArr& ops, u64 ws, u64 ss, u64 slot0,
                            u64 slot1, unsigned long long* counter, u64 out_cap, u8* key_cls, i64* key_val, u8* agg_cls, i64* agg_val,
                            cudaStream_t s) {
    if (T.wait_flags) {
        k_peer_wait<<<1, 32, 0, s>>>(T.wait_flags, T.n, T.wait_seq, T.status);
        g_launches.fetch_add(1);
    }
    if (slot1 <= slot0) return;
    k_finalize_groups<<<grid_for(slot1 - slot0), 256, 0, s>>>(D, kw, keys, T, ops, ws, ss, slot0, slot1, counter, out_cap, key_cls, key_val,
                                                              agg_cls, agg_val);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_merge_mailbox(const u64* mail, int nranks, u64 slot_base, u64 stride, u64 words, u64 seq, u64 cap, const OpsArr& ops,
                          u64* out_dev, u64* out_host, int* status, cudaStream_t s) {
    k_merge_mailbox<<<1, 256, 0, s>>>(mail, nranks, slot_base, stride, words, seq, cap, ops, out_dev, out_host, status);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_merge_words(const u64* all, int nranks, u64 cap, const OpsArr& ops, u64* out_dev, u64* out_host, cudaStream_t s) {
    k_merge_words<<<grid_for(cap * ops.n), 256, 0, s>>>(all, nranks, cap, ops, out_dev, out_host);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_init_words(u64* acc, u64 cap, const OpsArr& ops, cudaStream_t s) {
    k_init_words<<<grid_for(cap * ops.n), 256, 0, s>>>(acc, cap, ops);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_fill_u64(u64* p, u64 n, u64 v, cudaStream_t s) {
    k_fill_u64<<<grid_for(n), 256, 0, s>>>(p, n, v);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_count_owners(int kw, const u64* keys, const u64* acc, u64 cap, int nranks, int gk_pos, int gk_bits,
                         unsigned long long* counts, cudaStream_t s) {
    k_count_owners<<<grid_for(kw == 4 ? cap >> 6 : cap), 256, 0, s>>>(kw, keys, acc, cap, nranks, gk_pos, gk_bits, counts);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_export_records(int kw, const u64* keys, const u64* acc, u64 cap, int W, int nranks, int gk_pos, int gk_bits,
                           unsigned long long* cursor, u64* out, u64 out_cap, cudaStream_t s) {
    k_export_records<<<grid_for(kw == 4 ? cap >> 6 : cap), 256, 0, s>>>(kw, keys, acc, cap, W, nranks, gk_pos, gk_bits, cursor, out, out_cap);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_merge_records(int kw, u64* keys, u64* acc, u64 cap, const OpsArr& ops, const u64* recs, u64 n, int* status, cudaStream_t s) {
    if (n == 0) return;
    k_merge_records<<<grid_for(n), 256, 0, s>>>(kw, keys, acc, cap, ops, recs, n, status);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}

}  // namespace n1
