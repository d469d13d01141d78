// n1ql_device.cuh — hand-written sm_100a device library for the N1QL filter + GROUP BY path.
//
// Every specialised scan kernel (one per compiled query, emitted by codegen.cpp and built with
// NVRTC for sm_100a) is assembled from the typed-value semantics of n1ql_value.cuh (MISSING/NULL/
// BOOLEAN/NUMBER/STRING collation, 4-valued logic, int64->float64 promotion, the NqParams block) and
// the device-only functions in this file: 128/256-bit coalesced column loads, block reductions,
// atomics, the shared-memory front cache, the HBM open-addressing table (64- and 128-bit keys) and
// IN over a device-resident set.
//
// The same header is compiled by nvcc into libn1gpu.so's static kernels (kernels.cu), so it is
// build-checked for sm_100a at build() time.  It must stay free of host/std includes (NVRTC).
#pragma once

#include "n1ql_value.cuh"

#define NQ_DEV __device__ __forceinline__

// ---- coalesced vector loads (4 rows per thread: 256-bit / 128-bit / 32-bit) -----------------------
// ld.global.nc + L1::no_allocate: every column byte is read exactly once per scan.
NQ_DEV void ld_rows4_b64(const i64* __restrict__ p, i64 (&v)[4]) {
#if __CUDA_ARCH__ >= 1000 && !defined(NQ_NO_LD256)
    asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v4.b64 {%0,%1,%2,%3}, [%4];"
                 : "=l"(v[0]), "=l"(v[1]), "=l"(v[2]), "=l"(v[3]) : "l"(p));
#else
    asm volatile("ld.global.nc.L1::no_allocate.v2.b64 {%0,%1}, [%2];" : "=l"(v[0]), "=l"(v[1]) : "l"(p));
    asm volatile("ld.global.nc.L1::no_allocate.v2.b64 {%0,%1}, [%2];" : "=l"(v[2]), "=l"(v[3]) : "l"(p + 2));
#endif
}
NQ_DEV void ld_rows4_b32(const u32* __restrict__ p, u32 (&v)[4]) {
    asm volatile("ld.global.nc.L1::no_allocate.v4.b32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "l"(p));
}
NQ_DEV void ld_rows4_b8(const u8* __restrict__ p, int (&v)[4]) {
    u32 w;
    asm volatile("ld.global.nc.L1::no_allocate.b32 %0, [%1];" : "=r"(w) : "l"(p));
    v[0] = w & 0xff; v[1] = (w >> 8) & 0xff; v[2] = (w >> 16) & 0xff; v[3] = w >> 24;
}

// ---- warp / block reductions ---------------------------------------------------------------------
NQ_DEV u64 shfl_xor_u64(u64 v, int m) { return (u64)__shfl_xor_sync(0xffffffffu, (i64)v, m); }
NQ_DEV u64 word_combine(int op, u64 a, u64 b) {
    switch (op) {
        case OP_ADD_U64: return a + b;
        case OP_ADD_F64: return (u64)__double_as_longlong(__longlong_as_double((i64)a) + __longlong_as_double((i64)b));
        case OP_MIN_I64: return (i64)a < (i64)b ? a : b;
        case OP_MAX_I64: return (i64)a > (i64)b ? a : b;
        case OP_MIN_U64: return a < b ? a : b;
        case OP_MAX_U64: return a > b ? a : b;
        default: return a | b;
    }
}
NQ_DEV u64 word_identity(int op) {
    switch (op) {
        case OP_MIN_I64: return (u64)NQ_I64_MAX;
        case OP_MAX_I64: return (u64)NQ_I64_MIN;
        case OP_MIN_U64: return NQ_U64_MAX;
        default: return 0;  // ADD_U64, ADD_F64 (+0.0), MAX_U64, OR
    }
}
template <int OP> NQ_DEV u64 warp_reduce_word(u64 v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v = word_combine(OP, v, shfl_xor_u64(v, m));
    return v;
}
// Block reduce of one accumulator word in a fixed (deterministic) order; result valid in thread 0.
// scratch: u64[32] in shared memory.
template <int OP> NQ_DEV u64 block_reduce_word(u64 v, u64* scratch) {
    v = warp_reduce_word<OP>(v);
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (lane == 0) scratch[w] = v;
    __syncthreads();
    if (w == 0) {
        v = lane < nw ? scratch[lane] : word_identity(OP);
        v = warp_reduce_word<OP>(v);
    }
    return v;
}

// ---- atomic application of an accumulator word (shared or global memory) ---------------------------
template <int OP> NQ_DEV void atomic_word(u64* p, u64 x) {
    if (OP == OP_ADD_U64) atomicAdd(p, x);
    else if (OP == OP_ADD_F64) atomicAdd((double*)p, __longlong_as_double((i64)x));
    else if (OP == OP_MIN_I64) atomicMin((i64*)p, (i64)x);
    else if (OP == OP_MAX_I64) atomicMax((i64*)p, (i64)x);
    else if (OP == OP_MIN_U64) atomicMin(p, x);
    else if (OP == OP_MAX_U64) atomicMax(p, x);
    else atomicOr(p, x);
}
NQ_DEV void atomic_word_dyn(int op, u64* p, u64 x) {
    switch (op) {
        case OP_ADD_U64: atomic_word<OP_ADD_U64>(p, x); break;
        case OP_ADD_F64: atomic_word<OP_ADD_F64>(p, x); break;
        case OP_MIN_I64: atomic_word<OP_MIN_I64>(p, x); break;
        case OP_MAX_I64: atomic_word<OP_MAX_I64>(p, x); break;
        case OP_MIN_U64: atomic_word<OP_MIN_U64>(p, x); break;
        case OP_MAX_U64: atomic_word<OP_MAX_U64>(p, x); break;
        default: atomic_word<OP_OR_U64>(p, x); break;
    }
}

// ---- HBM open-addressing tables --------------------------------------------------------------------
// 64-bit keys: slot key array u64[cap], EMPTY = all ones (packed keys use at most 63 bits).
// 128-bit keys: ulonglong2[cap] claimed with one 128-bit CAS (ATOMG.E.CAS.128), EMPTY = all ones.
// returns slot, or -1 when the probe budget is exhausted (table too small -> host grows and reruns);
// *fresh (optional) reports whether this call claimed the slot.
NQ_DEV i64 table_insert64(u64* __restrict__ keys, u64 cap_mask, u64 key, bool* fresh) {
    u64 slot = mix64(key) & cap_mask;
    for (u64 probe = 0; probe <= cap_mask; ++probe) {
        u64 cur = *(volatile u64*)&keys[slot];
        if (cur == key) { if (fresh) *fresh = false; return (i64)slot; }
        if (cur == NQ_U64_MAX) {
            u64 old = atomicCAS(&keys[slot], NQ_U64_MAX, key);
            if (old == NQ_U64_MAX) { if (fresh) *fresh = true; return (i64)slot; }
            if (old == key) { if (fresh) *fresh = false; return (i64)slot; }
        }
        slot = (slot + 1) & cap_mask;
        if (probe > 4096) break;
    }
    return -1;
}
NQ_DEV i64 table_find64(const u64* __restrict__ keys, u64 cap_mask, u64 key) {
    u64 slot = mix64(key) & cap_mask;
    for (u64 probe = 0; probe <= cap_mask; ++probe) {
        u64 cur = keys[slot];
        if (cur == key) return (i64)slot;
        if (cur == NQ_U64_MAX) return -1;
        slot = (slot + 1) & cap_mask;
    }
    return -1;
}
#if !defined(__CUDA_ARCH__) || __CUDA_ARCH__ >= 900
NQ_DEV i64 table_insert128(ulonglong2* __restrict__ keys, u64 cap_mask, u64 lo, u64 hi, bool* fresh) {
    u64 slot = mix64(lo ^ mix64(hi)) & cap_mask;
    unsigned __int128 key = ((unsigned __int128)hi << 64) | lo;
    unsigned __int128 empty = ~(unsigned __int128)0;
    for (u64 probe = 0; probe <= cap_mask; ++probe) {
        ulonglong2 cur;  // one aligned 128-bit access (LDG.E.128): never observes half a key
        asm volatile("ld.relaxed.gpu.global.v2.u64 {%0,%1}, [%2];" : "=l"(cur.x), "=l"(cur.y) : "l"(&keys[slot]) : "memory");
        if (cur.x == lo && cur.y == hi) { if (fresh) *fresh = false; return (i64)slot; }
        if (cur.x == NQ_U64_MAX && cur.y == NQ_U64_MAX) {
            unsigned __int128 old = atomicCAS((unsigned __int128*)&keys[slot], empty, key);
            if (old == empty) { if (fresh) *fresh = true; return (i64)slot; }
            if (old == key) { if (fresh) *fresh = false; return (i64)slot; }
        }
        slot = (slot + 1) & cap_mask;
        if (probe > 4096) break;
    }
    return -1;
}
NQ_DEV i64 table_find128(const ulonglong2* __restrict__ keys, u64 cap_mask, u64 lo, u64 hi) {
    u64 slot = mix64(lo ^ mix64(hi)) & cap_mask;
    for (u64 probe = 0; probe <= cap_mask; ++probe) {
        ulonglong2 cur = keys[slot];
        if (cur.x == lo && cur.y == hi) return (i64)slot;
        if (cur.x == NQ_U64_MAX && cur.y == NQ_U64_MAX) return -1;
        slot = (slot + 1) & cap_mask;
    }
    return -1;
}
#endif

// 32-bit shared-state-space addresses of the front cache.  Through a generic pointer the compiler rebuilds the block's
// shared window (S2R SR_CgaCtaId + LEA) at every cache access of the row loop (config 5: 8 times per tile); the address
// made once by smem_addr is opaque to it, so it stays in a register and every access is one LDS / ATOMS [reg + imm].
NQ_DEV u32 smem_addr(const void* p) {
    u32 a;
    asm volatile("mov.b32 %0, %1;" : "=r"(a) : "r"((u32)__cvta_generic_to_shared(p)));
    return a;
}
NQ_DEV u32 lds_u32(u32 a) { u32 v; asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
NQ_DEV u32 atoms_add(u32 a, u32 x) { u32 o; asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(o) : "r"(a), "r"(x)); return o; }
NQ_DEV void reds_add(u32 a, u32 x) { asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(a), "r"(x)); }
NQ_DEV void reds_min(u32 a, u32 x) { asm volatile("red.shared.min.u32 [%0], %1;" :: "r"(a), "r"(x)); }
NQ_DEV void reds_max(u32 a, u32 x) { asm volatile("red.shared.max.u32 [%0], %1;" :: "r"(a), "r"(x)); }
NQ_DEV void reds_or(u32 a, u32 x) { asm volatile("red.shared.or.b32 [%0], %1;" :: "r"(a), "r"(x)); }
NQ_DEV u32 atoms_cas(u32 a, u32 c, u32 x) { u32 o; asm volatile("atom.shared.cas.b32 %0, [%1], %2, %3;" : "=r"(o) : "r"(a), "r"(c), "r"(x)); return o; }

// Per-block shared-memory front cache of the HBM group table (hot keys of a skewed GROUP BY are aggregated with
// shared-memory atomics and reach HBM once per block): claims or finds `key` within 4 probes, else -1 (miss).
// (any slot count, not only powers of two: the slot is the high part of hash * slots)
NQ_DEV int cache_claim_n(u64* ckeys, u32 slots, u32 hash, u64 key) {
    u32 h = __umulhi(hash, slots);
#pragma unroll
    for (int probe = 0; probe < 4; ++probe) {
        const u64 cur = ((volatile u64*)ckeys)[h];
        if (cur == key) return (int)h;
        if (cur == NQ_U64_MAX) {
            const u64 old = atomicCAS(&ckeys[h], NQ_U64_MAX, key);
            if (old == NQ_U64_MAX || old == key) return (int)h;
        }
        h = h + 1 == slots ? 0 : h + 1;
    }
    return -1;
}

// The same for packed keys of <= 31 bits: u32 keys, direct-mapped - one slot per key, one 32-bit load.  Buckets of four
// keys (one 16-byte load per lane, 4 shared-memory wavefronts at best, and a 4-way select chain for every row) miss fewer
// keys and were still slower: 6 % in tools/proto5.cu, 5.19 against 4.95 ms per 1 B config-5 rows in the generated kernel
// (profiles/r02_config5_ablation.jsonl).
// (ckeys: smem_addr of the key array)
NQ_DEV int cache_claim_1(u32 ckeys, u32 nslots, u32 hash, u32 key) {
    const u32 b = __umulhi(hash, nslots);
    const u32 k = lds_u32(ckeys + 4 * b);
    if (k == key) return (int)b;
    if (k != 0xffffffffu) return -1;
    const u32 old = atoms_cas(ckeys + 4 * b, 0xffffffffu, key);
    return (old == 0xffffffffu || old == key) ? (int)b : -1;
}
NQ_DEV int cache_claim_1(u32* ckeys, u32 nslots, u32 hash, u32 key) { return cache_claim_1(smem_addr(ckeys), nslots, hash, key); }

// Cells of the front cache.  Shared memory has native 32-bit atomics only (a 64-bit atomicAdd/Min/Max on shared
// memory compiles to a compare-and-swap loop, 3-9x slower and collapsing under same-key contention), so a cached
// accumulator word is kept in 32-bit cells wherever its per-block value provably fits or can be split:
//   row counters        one cell (a block scans far fewer than 2^32 rows)
//   integer sums        two cells, low word + high word with the carry propagated by the adding thread
//   ranged min / max    one cell holding (value - lo + 1); 0 (max) / all ones (min) = nothing seen
//   class-seen bits     one cell
// anything else (float64 sums, unranged or float min/max) keeps a 64-bit cell and checks before it swaps.
NQ_DEV void cache_add_wide(u32* lo, u32* hi, u64 x) {
    const u32 xl = (u32)x;
    const u32 old = atomicAdd(lo, xl);
    const u32 h = (u32)(x >> 32) + ((u32)(old + xl) < xl ? 1u : 0u);
    if (h) atomicAdd(hi, h);
}
// One-cell integer sum (addends within +-2^31): the low word is cached, whatever the add carries or borrows goes straight
// to the table word as a multiple of 2^32 (rare: once per 2^32 / |x| rows; a small negative addend wraps the cell and
// cancels its own sign extension).  Cell and table word are both plain sums, so the flush just adds the cell.
// (the cells of these helpers are smem_addr addresses; the u32* forms convert)
NQ_DEV void cache_add_carry(u32 lo, u64 x, u64* table_word) {
    const u32 xl = (u32)x;
    const u32 old = atoms_add(lo, xl);
    const u32 h = (u32)(x >> 32) + ((u32)(old + xl) < xl ? 1u : 0u);
    if (h) atomicAdd(table_word, (u64)h << 32);
}
NQ_DEV void cache_add_carry(u32* lo, u64 x, u64* table_word) { cache_add_carry(smem_addr(lo), x, table_word); }
// (read first: a shared-memory load costs about half an atomic, and a group's min / max settle after a few rows; a
// stale read can only cause an atomic that was not needed.  Round 1's unconditional atomic was slower: 1 520 against
// 1 497 us per 200 M config-5 rows, profiles/r01_config5_sweep.jsonl)
// the same with the cell's current value already in a register (two interleaved cells fetched by one 64-bit load)
template <int OP> NQ_DEV void cache_mm32_cur(u32 c, u64 x, u64 bias, u32 cur) {
    const u32 v = (u32)(x - bias) + 1u;
    if (OP == OP_MIN_I64 || OP == OP_MIN_U64) { if (v < cur) reds_min(c, v); } else { if (v > cur) reds_max(c, v); }
}
template <int OP> NQ_DEV void cache_mm32(u32 c, u64 x, u64 bias) { cache_mm32_cur<OP>(c, x, bias, lds_u32(c)); }
template <int OP> NQ_DEV void cache_mm32(u32* c, u64 x, u64 bias) { cache_mm32<OP>(smem_addr(c), x, bias); }
NQ_DEV void cache_or32(u32 c, u32 bits) {
    if ((lds_u32(c) & bits) != bits) reds_or(c, bits);
}
template <int OP> NQ_DEV void cache_word64(u64* c, u64 x) {
    if (OP == OP_MIN_I64) { if ((i64)x < *(volatile i64*)c) atomicMin((i64*)c, (i64)x); }
    else if (OP == OP_MAX_I64) { if ((i64)x > *(volatile i64*)c) atomicMax((i64*)c, (i64)x); }
    else if (OP == OP_MIN_U64) { if (x < *(volatile u64*)c) atomicMin(c, x); }
    else if (OP == OP_MAX_U64) { if (x > *(volatile u64*)c) atomicMax(c, x); }
    else atomic_word<OP>(c, x);
}

// bit packing of group-key / DISTINCT-entry components into a 128-bit (lo,hi) key
NQ_DEV void pack_bits(u64& lo, u64& hi, int& pos, u64 v, int nbits) {
    if (nbits == 0) return;
    if (pos < 64) {
        lo |= v << pos;
        if (pos + nbits > 64) hi |= v >> (64 - pos);
    } else {
        hi |= v << (pos - 64);
    }
    pos += nbits;
}

// ---- IN over a device-resident set ------------------------------------------------------------------
// The fold of in_arg / in_fin over a list of constants, restated over a set built on the host (codegen.cpp, build_inset):
//   STRING  bitmap over the operand column's dictionary ranks (an element absent from the dictionary sets no bit)
//   INT     open-addressing table of the INT elements (linear probing, load <= 0.25)
//   FLOAT   the same over the float64 images of the FLOAT elements and of the INT elements (v_eq compares any pair that is
//           not INT / INT as float64); -0.0 is stored and probed as +0.0, NaN never matches
// An INT row equals a FLOAT element only through rounding: integral floats below 2^63 in magnitude are INTs after
// canonicalisation, so 2^63 is the only FLOAT element an INT row can hit (INSET_P63).  NQ_U64_MAX marks an empty slot;
// an INT element of that value is the flag INSET_IEMPTY (a float key never has those bits: they are a NaN).
NQ_DEV bool inset_probe(const u64* __restrict__ keys, u32 cap, u64 key) {
    if (cap == 0) return false;
    u32 slot = inset_slot(key, cap);
    for (;;) {
        const u64 cur = __ldg(&keys[slot]);
        if (cur == key) return true;
        if (cur == NQ_U64_MAX) return false;
        slot = (slot + 1) & (cap - 1);
    }
}
NQ_DEV Val in_set(Val x, const NqInSet& d) {
    if (x.c == C_MISSING) return x;
    bool hit = false;
    if (x.c == C_INT) {
        hit = (u64)x.b == NQ_U64_MAX ? (d.flags & INSET_IEMPTY) != 0 : inset_probe(d.keys, d.icap, (u64)x.b);
        if (!hit && (d.flags & INSET_P63)) hit = (double)x.b == 9223372036854775808.0;
    } else if (x.c == C_FLOAT) {
        const double f = as_f(x.b);
        if (f == f) hit = inset_probe(d.keys + d.icap, d.fcap, f == 0.0 ? 0ULL : (u64)x.b);
    } else if (x.c == C_STRING) {
        const u64 r = (u64)x.b >> 1;
        hit = (__ldg(&d.bits[r >> 5]) >> (r & 31)) & 1u;
    } else if (x.c == C_FALSE) hit = d.flags & INSET_FALSE;
    else if (x.c == C_TRUE) hit = d.flags & INSET_TRUE;
    else return (d.flags & INSET_VALUED) ? mkv(C_NULL, 0) : ((d.flags & INSET_MISSING) ? mkv(C_MISSING, 0) : mkbool(false));  // NULL row
    return hit ? mkbool(true) : ((d.flags & INSET_NULL) ? mkv(C_NULL, 0) : ((d.flags & INSET_MISSING) ? mkv(C_MISSING, 0) : mkbool(false)));
}

NQ_DEV bool nq_cancelled(const NqParams& p, int lane) {
    int c = 0;
    if (lane == 0) c = *(volatile const int*)p.cancel;
    return __shfl_sync(0xffffffffu, c, 0) != 0;
}

// Pushes `words` final words at src to every peer's mailbox and raises the flag word behind them.
NQ_DEV void mailbox_push(const NqParams& p, const u64* src) {
    __threadfence();
    __syncthreads();
    const u64 total = p.mail_words * (u64)p.nranks;
    for (u64 i = threadIdx.x; i < total; i += blockDim.x) {
        const u64 r = i / p.mail_words, w = i % p.mail_words;
        p.peer_mail[r][p.mail_base + w] = __ldcg(&src[w]);
    }
    __threadfence_system();
    __syncthreads();
    if ((int)threadIdx.x < p.nranks) {
        u64* flag = &p.peer_mail[threadIdx.x][p.mail_base + p.mail_words];
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flag), "l"(p.mail_seq) : "memory");
    }
}

// Dynamic-op warp reduction (the final, fixed-order fold of per-block partials by the last block).
NQ_DEV u64 warp_reduce_dyn(int op, u64 v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v = word_combine(op, v, shfl_xor_u64(v, m));
    return v;
}
// Returns true in every thread of exactly one block per launch: the last one to arrive.  All global writes the
// other blocks made before their arrival are visible to it.
NQ_DEV bool last_block_arrives(unsigned* ticket) {
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned t = atomicAdd(ticket, 1u);
        s_last = (t == gridDim.x - 1);
        if (s_last) *ticket = 0;  // ready for the next launch on this stream
    }
    __syncthreads();
    if (s_last) __threadfence();
    return s_last != 0;
}
