// proto5.cu — stand-alone prototype harness for the config-5 scan (1 B rows, Zipf string keys, 20 % MISSING/NULL):
// hand-written variants of the grouped scan, timed and checked against a plain global-atomic reference, so that a
// design can be measured on the B200 before it is moved into the code generator (codegen.cpp).
//
//   nvcc -O3 -std=c++17 -lineinfo -gencode arch=compute_100a,code=sm_100a --fmad=false -Iquery_b200/csrc \
//        -o tools/_build/proto5 tools/proto5.cu && tools/_build/proto5 [rows]
//   (-DPROTO_MODE=1 / 2 builds the two experiment modes described at k_scan_q's g_match / g_pack)
//
// Variants
//   base   the kernel codegen.cpp emitted for this query when the harness was written (proto5_base.cuh: SoA table,
//          per-row phases, u32 cache keys in buckets of four)
//   q      register groups for the payload-free key classes (MISSING / NULL keys), a per-warp shared-memory queue
//          that compacts the remaining rows into full 32-lane batches for the front cache, a second queue that
//          compacts cache misses, slot-major (one 32-byte sector per group) HBM table updated by lane pairs
//          (one RED per operation class instead of one per word), 24-byte cache slots (sum carries go to HBM)
//   q+l0   the same plus a lane-replicated (bank == lane, conflict-free) L0 cache for the hottest keys
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <vector>
#include <algorithm>
#include <random>
#include <cuda_runtime.h>

#define nq_scan nq_scan_base
#include "proto5_base.cuh"
#undef nq_scan
#undef ACC
#undef ACCIF

#define CKE(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(1); } } while (0)

static const int VOCAB = 100000;
static const u64 SLOTS = 131072;  // 17-bit packed key: 0 MISSING, 1 NULL, 2 + rank

__device__ __forceinline__ u64 splitmix(u64 x) { x += 0x9e3779b97f4a7c15ULL; x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ULL; x = (x ^ (x >> 27)) * 0x94d049bb133111ebULL; return x ^ (x >> 31); }

__global__ void k_gen(u32* code, u8* ktag, i64* v, u8* vtag, i64 n, i64 npad, const double* cdf, const u32* perm, u64 seed) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < npad; i += (i64)gridDim.x * blockDim.x) {
        if (i >= n) { code[i] = 0; ktag[i] = 0; v[i] = 0; vtag[i] = 0; continue; }
        const u64 r1 = splitmix(seed ^ (u64)i * 0x2545F4914F6CDD1DULL), r2 = splitmix(r1), r3 = splitmix(r2), r4 = splitmix(r3);
        const double u = (double)(r1 >> 11) / 9007199254740992.0;
        int lo = 0, hi = VOCAB - 1;  // first index with cdf >= u
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (cdf[mid] >= u) hi = mid; else lo = mid + 1; }
        code[i] = perm[lo];
        const u64 mk = r2 % 10ULL, mv = r3 % 10ULL;
        ktag[i] = mk == 0 ? C_MISSING : (mk == 1 ? C_NULL : C_STRING);
        vtag[i] = mv == 0 ? C_MISSING : (mv == 1 ? C_NULL : C_INT);
        v[i] = (i64)(r4 % 1001000ULL) - 1000;
    }
}

// ---- reference: plain global atomics on a [6][SLOTS] table: rows, cnull, sum, nneg(unused), min, max --------------------
__global__ void k_ref(const u32* code, const u8* ktag, const i64* v, const u8* vtag, i64 n, u64* t) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        if (vtag[i] == C_MISSING) continue;
        const u64 key = ktag[i] == C_MISSING ? 0 : (ktag[i] == C_NULL ? 1 : 2 + code[i]);
        atomicAdd(&t[0 * SLOTS + key], 1ULL);
        if (vtag[i] == C_NULL) { atomicAdd(&t[1 * SLOTS + key], 1ULL); continue; }
        atomicAdd(&t[2 * SLOTS + key], (u64)v[i]);
        atomicMin((i64*)&t[4 * SLOTS + key], v[i]);
        atomicMax((i64*)&t[5 * SLOTS + key], v[i]);
    }
}
__global__ void k_fill(u64* p, u64 n, u64 v) { for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) p[i] = v; }
__global__ void k_fill4(u64* p, u64 nslots, u64 a, u64 b, u64 c, u64 d) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < nslots; i += (u64)gridDim.x * blockDim.x) { p[4 * i] = a; p[4 * i + 1] = b; p[4 * i + 2] = c; p[4 * i + 3] = d; }
}

// ---- the queued variant -------------------------------------------------------------------------------------------------------
// HBM table: slot-major, 4 words per group = one 32-byte sector:
//   W0 rows | (rows with v NULL) << 32   (add)      W1 sum of (v + 1000)            (add)
//   W2 max of ~v  (= ~min v)             (max s64)   W3 max of v                     (max s64)
#define VBIAS 1000
#define QCAP 64
#ifndef PROTO_MODE
#define PROTO_MODE 0
#endif
struct QParams { const u32* code; const u8* ktag; const i64* v; const u8* vtag; i64 nrows; u64* table; const u32* hot; int match; };

template <int NT, int NS, int K0, int QUEUES = 1>
struct Smem {
    u32 ckey[NS];
    u32 c_rows[NS], c_cnull[NS], c_sum[NS], c_nmin[NS], c_max[NS];
    u32 qkey[QUEUES ? NT / 32 : 1][QCAP], qval[QUEUES ? NT / 32 : 1][QCAP];
    u32 mkey[QUEUES ? NT / 32 : 1][QCAP], mval[QUEUES ? NT / 32 : 1][QCAP];
    u32 l0key[K0 ? K0 : 1][32], l0n[K0 ? K0 : 1][32], l0sum[K0 ? K0 : 1][32], l0nmin[K0 ? K0 : 1][32], l0max[K0 ? K0 : 1][32];
};

__device__ __forceinline__ void red_add_u64(u64* p, u64 v) { asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory"); }
__device__ __forceinline__ void red_max_s64(u64* p, i64 v) { asm volatile("red.global.max.s64 [%0], %1;" ::"l"(p), "l"(v) : "memory"); }

// probe of the block's front cache with WAYS keys per bucket (4: one LDS.128, 2: one LDS.64, 1: direct-mapped LDS.32)
template <int WAYS>
__device__ __forceinline__ int cache_claim_w(u32* ckeys, u32 nslots, u32 hash, u32 key) {
    if (WAYS == 4) return cache_claim_b4(ckeys, nslots / 4, hash, key);
    if (WAYS == 2) {
        const u32 b = __umulhi(hash, nslots / 2) * 2u;
        u32 k0, k1;
        asm volatile("ld.volatile.shared.v2.u32 {%0,%1}, [%2];" : "=r"(k0), "=r"(k1) : "r"((u32)__cvta_generic_to_shared(ckeys + b)) : "memory");
        if (k0 == key) return (int)b;
        if (k1 == key) return (int)b + 1;
        if (k1 != 0xffffffffu) return -1;  // slots fill in order: the last one taken = full
        if (k0 == 0xffffffffu) { const u32 old = atomicCAS(&ckeys[b], 0xffffffffu, key); if (old == 0xffffffffu || old == key) return (int)b; }
        const u32 old = atomicCAS(&ckeys[b + 1], 0xffffffffu, key);
        return (old == 0xffffffffu || old == key) ? (int)b + 1 : -1;
    }
    const u32 b = __umulhi(hash, nslots);
    const u32 k0 = *(volatile u32*)&ckeys[b];
    if (k0 == key) return (int)b;
    if (k0 != 0xffffffffu) return -1;
    const u32 old = atomicCAS(&ckeys[b], 0xffffffffu, key);
    return (old == 0xffffffffu || old == key) ? (int)b : -1;
}

template <int NT, int NS, int K0, int L0T, int WAYS, int CHECK, int PREF, int MNREG, int QROWS, int PAIR, int SOA>
__global__ void __launch_bounds__(NT, 1) k_scan_q(const QParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typedef Smem<NT, NS, K0, (QROWS || PAIR)> S;
    S& s = *reinterpret_cast<S*>(smem_raw);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    for (int i = threadIdx.x; i < NS; i += NT) { s.ckey[i] = p.hot ? p.hot[i] : 0xffffffffu; s.c_rows[i] = 0; s.c_cnull[i] = 0; s.c_sum[i] = 0; s.c_nmin[i] = 0; s.c_max[i] = 0; }
    if (K0) for (int i = threadIdx.x; i < K0 * 32; i += NT) { (&s.l0key[0][0])[i] = 0xffffffffu; (&s.l0n[0][0])[i] = 0; (&s.l0sum[0][0])[i] = 0; (&s.l0nmin[0][0])[i] = 0; (&s.l0max[0][0])[i] = 0; }
    __syncthreads();
    // register groups: key classes without a payload (0 MISSING, 1 NULL)
    u32 r_rows[2] = {0, 0}, r_cnull[2] = {0, 0}, r_nmin[2] = {0, 0}, r_max[2] = {0, 0};
    u64 r_sum[2] = {0, 0};
    unsigned qhead = 0, qtail = 0, mhead = 0, mtail = 0;  // warp-uniform ring cursors
    u32* const qk = s.qkey[(QROWS || PAIR) ? w : 0]; u32* const qv = s.qval[(QROWS || PAIR) ? w : 0];
    u32* const mk = s.mkey[(QROWS || PAIR) ? w : 0]; u32* const mv = s.mval[(QROWS || PAIR) ? w : 0];
    u64* const table = p.table;
    // experiment modes are compile-time (-DPROTO_MODE=1: warp-cooperative __match_any_sync pre-aggregation, 2: row counter and
    // sum packed into one shared-memory atomic) so that the plain variants keep their code and register allocation
    constexpr bool g_match = PROTO_MODE == 1;
    constexpr bool g_pack = PROTO_MODE == 2;
    // word w of group `key`: one 32-byte sector per group (slot-major), or word planes (SOA: the round-1 layout)
    auto word = [&](u32 key, int w) -> u64* { return SOA ? table + (u64)w * SLOTS + key : table + (u64)key * 4 + w; };

    auto flush_miss = [&](bool all) {
        // lane pairs: lane 2e works on word (lane & 1) of entry e's slot: one RED per operation class
        while (mtail - mhead >= 16u || (all && mtail != mhead)) {
            const unsigned n = min(16u, mtail - mhead);
            const unsigned e = lane >> 1, half = lane & 1;
            const bool valid = e < n;
            const unsigned idx = (mhead + e) & (QCAP - 1);
            const u32 key = valid ? mk[idx] : 0u, val = valid ? mv[idx] : 0u;
            const bool isnull = val >> 31;
            const u32 vb = val & 0xfffffu;
            u64* const slot = table + (u64)key * 4;
            const u64 addv = half ? (isnull ? 0ULL : (u64)vb) : (1ULL | ((u64)isnull << 32));
            if (valid && addv) red_add_u64(slot + half, addv);
            const i64 vv = (i64)vb - VBIAS;
            if (valid && !isnull) red_max_s64(slot + 2 + half, half ? vv : ~vv);
            mhead += n;
        }
    };
    auto process = [&](bool active, u32 key, u32 val) {
        int slot = -2;
        if (g_match) {
            // warp-cooperative pre-aggregation: lanes holding the same key combine their row in the lowest of them
            // (__match_any_sync), which alone probes the cache and updates it with the combined count / sum / min / max
            const bool isnull0 = val >> 31;
            const u32 vb0 = val & 0xfffffu;
            const unsigned m = __match_any_sync(0xffffffffu, active ? key : 0xffffff00u + (u32)lane);
            const int leader = __ffs(m) - 1;
            u32 a_cs = active ? (isnull0 ? (1u << 26) : vb0) : 0u;              // sum | null count << 26: both additive
            u32 a_cnt = active ? 1u : 0u;
            u32 a_mx = (active && !isnull0) ? vb0 + 1u : 0u, a_nm = (active && !isnull0) ? 0x100000u - vb0 : 0u;
            const unsigned size_max = __reduce_max_sync(0xffffffffu, (unsigned)__popc(m));
            unsigned rest = m & ~(1u << leader);
            const u32 my_cs = a_cs, my_mx = a_mx, my_nm = a_nm;
            for (unsigned r = 1; r < size_max; ++r) {
                const int src = rest ? __ffs(rest) - 1 : lane;
                rest &= rest - 1;
                const u32 o_cs = __shfl_sync(0xffffffffu, my_cs, src), o_mx = __shfl_sync(0xffffffffu, my_mx, src), o_nm = __shfl_sync(0xffffffffu, my_nm, src);
                if (src != lane) { a_cs += o_cs; a_cnt += 1u; a_mx = max(a_mx, o_mx); a_nm = max(a_nm, o_nm); }
            }
            const bool lead = active && lane == leader;
            if (lead) slot = cache_claim_w<WAYS>(s.ckey, NS, key * 0x9E3779B1u, key);
            const u32 cn = a_cs >> 26, sm = a_cs & 0x3ffffffu;
            if (slot >= 0) {
                atomicAdd(&s.c_rows[slot], a_cnt);
                if (cn) atomicAdd(&s.c_cnull[slot], cn);
                if (a_cnt > cn) {
                    const u32 so = atomicAdd(&s.c_sum[slot], sm);
                    if ((u32)(so + sm) < sm) red_add_u64(word(key, 1), 1ULL << 32);
                    if (!CHECK || a_mx > *(volatile u32*)&s.c_max[slot]) atomicMax(&s.c_max[slot], a_mx);
                    if (!CHECK || a_nm > *(volatile u32*)&s.c_nmin[slot]) atomicMax(&s.c_nmin[slot], a_nm);
                }
            } else if (slot == -1) {
                red_add_u64(word(key, 0), (u64)a_cnt | ((u64)cn << 32));
                if (a_cnt > cn) { red_add_u64(word(key, 1), (u64)sm); red_max_s64(word(key, 2), ~((i64)(0x100000u - a_nm) - VBIAS)); red_max_s64(word(key, 3), (i64)(a_mx - 1u) - VBIAS); }
            }
            return;
        }
        if (active) slot = cache_claim_w<WAYS>(s.ckey, NS, key * 0x9E3779B1u, key);
        if (slot >= 0 && g_pack) {
            // ONE shared-memory atomic for the row counter (low 8 bits) and the sum (high 24 bits): whatever a field carries
            // out is seen in the returned old value by the thread that caused it and compensated in the table
            const bool isnull = val >> 31;
            const u32 vb = val & 0xfffffu;
            const u32 addv = isnull ? 0u : vb;
            const u32 old = atomicAdd(&s.c_rows[slot], 1u | (addv << 8));
            const bool cw = (old & 0xffu) == 0xffu;  // the count wrapped: 256 rows to the table, and its carry sits in the sum field
            if (cw) { red_add_u64(word(key, 0), 256ULL); red_add_u64(word(key, 1), ~0ULL); }
            if ((old >> 8) + addv + (cw ? 1u : 0u) >= (1u << 24)) red_add_u64(word(key, 1), 1ULL << 24);
            if (isnull) atomicAdd(&s.c_cnull[slot], 1u);
            else {
                const u32 a = vb + 1u, b = 0x100000u - vb;
                if (!CHECK || a > *(volatile u32*)&s.c_max[slot]) atomicMax(&s.c_max[slot], a);
                if (!CHECK || b > *(volatile u32*)&s.c_nmin[slot]) atomicMax(&s.c_nmin[slot], b);
            }
        } else
        if (slot >= 0) {
            const bool isnull = val >> 31;
            const u32 vb = val & 0xfffffu;
            const u32 old = atomicAdd(&s.c_rows[slot], 1u);
            if (isnull) atomicAdd(&s.c_cnull[slot], 1u);
            else {
                const u32 so = atomicAdd(&s.c_sum[slot], vb);
                if ((u32)(so + vb) < vb) red_add_u64(word(key, 1), 1ULL << 32);  // carry out of the 32-bit cell (rare)
                const u32 a = vb + 1u, b = 0x100000u - vb;
                if (!CHECK || a > *(volatile u32*)&s.c_max[slot]) atomicMax(&s.c_max[slot], a);
                if (!CHECK || b > *(volatile u32*)&s.c_nmin[slot]) atomicMax(&s.c_nmin[slot], b);
            }
            if (K0 && old >= (u32)L0T) {  // hot in this block: give it a conflict-free home in this lane's L0 column
                const unsigned e = (key * 0x9E3779B1u) >> 16 & (K0 - 1);
                if (*(volatile u32*)&s.l0key[e][lane] == 0xffffffffu) atomicCAS(&s.l0key[e][lane], 0xffffffffu, key);
            }
        }
        if (!PAIR) {  // every missed lane reduces its own words, one RED per word
            if (slot == -1) {
                const bool isnull = val >> 31;
                const u32 vb = val & 0xfffffu;
                red_add_u64(word(key, 0), 1ULL | ((u64)isnull << 32));
                if (!isnull) { red_add_u64(word(key, 1), (u64)vb); const i64 vv = (i64)vb - VBIAS; red_max_s64(word(key, 2), ~vv); red_max_s64(word(key, 3), vv); }
            }
            return;
        }
        const unsigned mm = __ballot_sync(0xffffffffu, slot == -1);
        if (mm) {
            if (slot == -1) { const unsigned at = (mtail + __popc(mm & lt)) & (QCAP - 1); mk[at] = key; mv[at] = val; }
            mtail += __popc(mm);
            __syncwarp();
            flush_miss(false);
        }
    };
    auto drain = [&](unsigned n) {
        const bool active = (unsigned)lane < n;
        const unsigned idx = (qhead + lane) & (QCAP - 1);
        const u32 key = active ? qk[idx] : 0u, val = active ? qv[idx] : 0u;
        qhead += n;
        process(active, key, val);
    };

    const i64 nrows = p.nrows;
    const i64 stride = (i64)gridDim.x * (NT * 4);
    u32 n0[4]; int nt0[4]; i64 n1[4]; int nt1[4];  // next tile (software prefetch)
    i64 wbase = (i64)blockIdx.x * (NT * 4) + w * 128;
    if (PREF && wbase < nrows) { const i64 b = wbase + lane * 4; ld_rows4_b32(p.code + b, n0); ld_rows4_b8(p.ktag + b, nt0); ld_rows4_b64(p.v + b, n1); ld_rows4_b8(p.vtag + b, nt1); }
    for (; wbase < nrows; wbase += stride) {
        const i64 base = wbase + lane * 4;
        u32 c0[4]; int t0[4]; i64 c1[4]; int t1[4];
        if (PREF) {
#pragma unroll
            for (int j = 0; j < 4; ++j) { c0[j] = n0[j]; t0[j] = nt0[j]; c1[j] = n1[j]; t1[j] = nt1[j]; }
            if (wbase + stride < nrows) { const i64 b = base + stride; ld_rows4_b32(p.code + b, n0); ld_rows4_b8(p.ktag + b, nt0); ld_rows4_b64(p.v + b, n1); ld_rows4_b8(p.vtag + b, nt1); }
        } else {
            ld_rows4_b32(p.code + base, c0); ld_rows4_b8(p.ktag + base, t0); ld_rows4_b64(p.v + base, c1); ld_rows4_b8(p.vtag + base, t1);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const bool pass = base + j < nrows && t1[j] != C_MISSING;
            const bool isnull = t1[j] == C_NULL;
            const u32 vb = isnull ? 0u : (u32)(c1[j] + VBIAS);
            if (MNREG) {
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    const bool hit = pass && t0[j] == g;
                    const bool hv = hit && !isnull;
                    r_rows[g] += hit;
                    r_cnull[g] += hit && isnull;
                    r_sum[g] += hv ? vb : 0u;
                    r_max[g] = max(r_max[g], hv ? vb + 1u : 0u);
                    r_nmin[g] = max(r_nmin[g], hv ? 0x100000u - vb : 0u);
                }
            }
            bool tostr = pass && (MNREG ? t0[j] == C_STRING : true);
            const u32 key = t0[j] == C_STRING ? c0[j] + 2u : (u32)t0[j];
            if (K0) {
                const unsigned e = (key * 0x9E3779B1u) >> 16 & (K0 - 1);
                if (tostr && !isnull && s.l0key[e][lane] == key) {  // bank == lane: no conflicts inside the warp
                    tostr = false;
                    atomicAdd(&s.l0n[e][lane], 1u);
                    const u32 so = atomicAdd(&s.l0sum[e][lane], vb);
                    if ((u32)(so + vb) < vb) red_add_u64(table + (u64)key * 4 + 1, 1ULL << 32);
                    const u32 a = vb + 1u, b = 0x100000u - vb;
                    if (a > *(volatile u32*)&s.l0max[e][lane]) atomicMax(&s.l0max[e][lane], a);
                    if (b > *(volatile u32*)&s.l0nmin[e][lane]) atomicMax(&s.l0nmin[e][lane], b);
                }
            }
            if (!QROWS) {  // no compaction: the rows of this warp-row go to the cache as they are (partial warps)
                if (__ballot_sync(0xffffffffu, tostr)) process(tostr, key, vb | ((u32)isnull << 31));
                continue;
            }
            const unsigned m = __ballot_sync(0xffffffffu, tostr);
            if (tostr) { const unsigned at = (qtail + __popc(m & lt)) & (QCAP - 1); qk[at] = key; qv[at] = vb | ((u32)isnull << 31); }
            qtail += __popc(m);
            __syncwarp();
            if (qtail - qhead >= 32u) drain(32u);
        }
    }
    if (qtail != qhead) drain(qtail - qhead);
    flush_miss(true);
    // register groups -> table slots 0 and 1 (warp reduction, then one lane)
#pragma unroll
    for (int g = 0; g < 2; ++g) {
        u64 rows = r_rows[g], cn = r_cnull[g], sm = r_sum[g];
        u32 mx = r_max[g], nm = r_nmin[g];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            rows += __shfl_xor_sync(0xffffffffu, rows, o); cn += __shfl_xor_sync(0xffffffffu, cn, o); sm += __shfl_xor_sync(0xffffffffu, sm, o);
            mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o)); nm = max(nm, __shfl_xor_sync(0xffffffffu, nm, o));
        }
        if (lane == 0 && rows) {
            red_add_u64(word(g, 0), rows | (cn << 32));
            if (sm) red_add_u64(word(g, 1), sm);
            if (mx) red_max_s64(word(g, 3), (i64)(mx - 1u) - VBIAS);
            if (nm) red_max_s64(word(g, 2), ~((i64)(0x100000u - nm) - VBIAS));
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < NS; i += NT) {
        const u32 key = s.ckey[i];
        if (key == 0xffffffffu) continue;
        const u64 w0 = (u64)(g_pack ? (s.c_rows[i] & 0xffu) : s.c_rows[i]) | ((u64)s.c_cnull[i] << 32);
        if (w0) red_add_u64(word(key, 0), w0);
        const u32 fs = g_pack ? (s.c_rows[i] >> 8) : s.c_sum[i];
        if (fs) red_add_u64(word(key, 1), (u64)fs);
        if (s.c_max[i]) red_max_s64(word(key, 3), (i64)(s.c_max[i] - 1u) - VBIAS);
        if (s.c_nmin[i]) red_max_s64(word(key, 2), ~((i64)(0x100000u - s.c_nmin[i]) - VBIAS));
    }
    if (K0) for (int i = threadIdx.x; i < K0 * 32; i += NT) {
        const u32 key = (&s.l0key[0][0])[i];
        if (key == 0xffffffffu) continue;
        u64* const slot = table + (u64)key * 4;
        const u32 n = (&s.l0n[0][0])[i], sm = (&s.l0sum[0][0])[i], mx = (&s.l0max[0][0])[i], nm = (&s.l0nmin[0][0])[i];
        if (n) red_add_u64(slot, (u64)n);
        if (sm) red_add_u64(slot + 1, (u64)sm);
        if (mx) red_max_s64(slot + 3, (i64)(mx - 1u) - VBIAS);
        if (nm) red_max_s64(slot + 2, ~((i64)(0x100000u - nm) - VBIAS));
    }
}

// ---- host -------------------------------------------------------------------------------------------------------------------
struct Ref { std::vector<u64> rows, cnull, sum; std::vector<i64> mn, mx; };

static bool check(const char* name, const Ref& r, const std::vector<u64>& rows, const std::vector<u64>& cnull, const std::vector<i64>& sum,
                  const std::vector<i64>& mn, const std::vector<i64>& mx) {
    long bad = 0;
    for (u64 i = 0; i < SLOTS; ++i) {
        bool ok = rows[i] == r.rows[i] && cnull[i] == r.cnull[i] && (u64)sum[i] == r.sum[i];
        if (r.rows[i] > r.cnull[i]) ok = ok && mn[i] == r.mn[i] && mx[i] == r.mx[i];
        if (!ok && bad++ < 5)
            fprintf(stderr, "  %s slot %llu: rows %llu/%llu cnull %llu/%llu sum %lld/%lld min %lld/%lld max %lld/%lld\n", name, (unsigned long long)i,
                    (unsigned long long)rows[i], (unsigned long long)r.rows[i], (unsigned long long)cnull[i], (unsigned long long)r.cnull[i],
                    (long long)sum[i], (long long)r.sum[i], (long long)mn[i], (long long)r.mn[i], (long long)mx[i], (long long)r.mx[i]);
    }
    return bad == 0;
}

template <int NT, int NS, int K0, int L0T, int WAYS = 4, int CHECK = 1, int PREF = 0, int MNREG = 1, int QROWS = 1, int PAIR = 1, int SOA = 0>
static void run_q(const char* name, const QParams& qp0, u64* d_tab, const Ref& ref, i64 n, int sms) {
    typedef Smem<NT, NS, K0, (QROWS || PAIR)> S;
    const size_t smem = sizeof(S);
    CKE(cudaFuncSetAttribute(k_scan_q<NT, NS, K0, L0T, WAYS, CHECK, PREF, MNREG, QROWS, PAIR, SOA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaFuncAttributes fa;
    CKE(cudaFuncGetAttributes(&fa, k_scan_q<NT, NS, K0, L0T, WAYS, CHECK, PREF, MNREG, QROWS, PAIR, SOA>));
    int occ = 0;
    CKE(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_scan_q<NT, NS, K0, L0T, WAYS, CHECK, PREF, MNREG, QROWS, PAIR, SOA>, NT, smem));
    QParams qp = qp0;
    qp.table = d_tab;
    qp.hot = nullptr;
    qp.match = PROTO_MODE;
    if (getenv("HOT") && WAYS == 1) {  // most-common-values statistic: every cache slot starts out owned by the hottest key that maps to it
        std::vector<u32> hot(NS, 0xffffffffu); std::vector<u64> cnt(NS, 0);
        for (u64 key = 2; key < SLOTS; ++key) {
            if (!ref.rows[key]) continue;
            const u32 b = (u32)(((u64)((u32)key * 0x9E3779B1u) * (u64)NS) >> 32);
            if (ref.rows[key] > cnt[b]) { cnt[b] = ref.rows[key]; hot[b] = (u32)key; }
        }
        u32* d_hot; CKE(cudaMalloc(&d_hot, NS * 4)); CKE(cudaMemcpy(d_hot, hot.data(), NS * 4, cudaMemcpyHostToDevice));
        qp.hot = d_hot;
    }
    cudaEvent_t e0, e1;
    CKE(cudaEventCreate(&e0)); CKE(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
        if (SOA) { k_fill<<<592, 256>>>(d_tab, 2 * SLOTS, 0); k_fill<<<592, 256>>>(d_tab + 2 * SLOTS, 2 * SLOTS, (u64)NQ_I64_MIN); }
        else k_fill4<<<592, 256>>>(d_tab, SLOTS, 0, 0, (u64)NQ_I64_MIN, (u64)NQ_I64_MIN);
        CKE(cudaDeviceSynchronize());
        CKE(cudaEventRecord(e0));
        k_scan_q<NT, NS, K0, L0T, WAYS, CHECK, PREF, MNREG, QROWS, PAIR, SOA><<<sms * occ, NT, smem>>>(qp);
        CKE(cudaEventRecord(e1));
        CKE(cudaDeviceSynchronize());
        CKE(cudaGetLastError());
        float ms; CKE(cudaEventElapsedTime(&ms, e0, e1));
        best = std::min(best, ms);
    }
    std::vector<u64> t(SLOTS * 4);
    CKE(cudaMemcpy(t.data(), d_tab, t.size() * 8, cudaMemcpyDeviceToHost));
    std::vector<u64> rows(SLOTS), cnull(SLOTS); std::vector<i64> sum(SLOTS), mn(SLOTS), mx(SLOTS);
    for (u64 i = 0; i < SLOTS; ++i) {
        const u64 w0 = SOA ? t[i] : t[4 * i], w1 = SOA ? t[SLOTS + i] : t[4 * i + 1], w2 = SOA ? t[2 * SLOTS + i] : t[4 * i + 2], w3 = SOA ? t[3 * SLOTS + i] : t[4 * i + 3];
        rows[i] = w0 & 0xffffffffULL; cnull[i] = w0 >> 32;
        sum[i] = (i64)w1 - (i64)VBIAS * (i64)(rows[i] - cnull[i]);
        mn[i] = ~(i64)w2; mx[i] = (i64)w3;
    }
    const bool ok = check(name, ref, rows, cnull, sum, mn, mx);
    printf("{\"variant\": \"%s\", \"soa\": %d, \"qrows\": %d, \"pair\": %d, \"ways\": %d, \"check\": %d, \"prefetch\": %d, \"mnreg\": %d, \"threads\": %d, \"cache_slots\": %d, \"l0\": %d, \"smem\": %zu, \"regs\": %d, \"blocks_per_sm\": %d, \"ms\": %.4f, \"rows_per_s\": %.4g, \"gb_per_s\": %.1f, \"frac\": %.3f, \"check\": \"%s\"}\n",
           name, SOA, QROWS, PAIR, WAYS, CHECK, PREF, MNREG, NT, NS, K0, smem, fa.numRegs, occ, best, n / (best * 1e-3), 14.0 * n / (best * 1e6), 14.0 * n / (best * 1e6) / 6547.8, ok ? "ok" : "MISMATCH");
    fflush(stdout);
}

int main(int argc, char** argv) {
    const i64 n = argc > 1 ? atoll(argv[1]) : 1000000000LL;
    const i64 npad = (n + 4095) / 4096 * 4096 + 4096;
    cudaDeviceProp prop;
    CKE(cudaGetDeviceProperties(&prop, 0));
    const int sms = prop.multiProcessorCount;
    // Zipf(1.1) over the vocabulary, popularity rank -> dictionary code through a fixed permutation
    std::vector<double> cdf(VOCAB);
    { double tot = 0; for (int i = 0; i < VOCAB; ++i) tot += pow((double)(i + 1), -1.1); double acc = 0; for (int i = 0; i < VOCAB; ++i) { acc += pow((double)(i + 1), -1.1) / tot; cdf[i] = acc; } cdf[VOCAB - 1] = 1.0; }
    std::vector<u32> perm(VOCAB);
    for (int i = 0; i < VOCAB; ++i) perm[i] = i;
    { std::mt19937 g(4); std::shuffle(perm.begin(), perm.end(), g); }
    double* d_cdf; u32* d_perm;
    CKE(cudaMalloc(&d_cdf, VOCAB * 8)); CKE(cudaMalloc(&d_perm, VOCAB * 4));
    CKE(cudaMemcpy(d_cdf, cdf.data(), VOCAB * 8, cudaMemcpyHostToDevice)); CKE(cudaMemcpy(d_perm, perm.data(), VOCAB * 4, cudaMemcpyHostToDevice));
    u32* d_code; u8* d_ktag; i64* d_v; u8* d_vtag;
    CKE(cudaMalloc(&d_code, npad * 4)); CKE(cudaMalloc(&d_ktag, npad)); CKE(cudaMalloc(&d_v, npad * 8)); CKE(cudaMalloc(&d_vtag, npad));
    k_gen<<<sms * 8, 256>>>(d_code, d_ktag, d_v, d_vtag, n, npad, d_cdf, d_perm, 4);
    CKE(cudaDeviceSynchronize());
    // reference
    u64* d_ref; CKE(cudaMalloc(&d_ref, 6 * SLOTS * 8));
    k_fill<<<592, 256>>>(d_ref, 4 * SLOTS, 0);
    k_fill<<<592, 256>>>(d_ref + 4 * SLOTS, SLOTS, (u64)NQ_I64_MAX);
    k_fill<<<592, 256>>>(d_ref + 5 * SLOTS, SLOTS, (u64)NQ_I64_MIN);
    k_ref<<<sms * 8, 256>>>(d_code, d_ktag, d_v, d_vtag, n, d_ref);
    CKE(cudaDeviceSynchronize());
    std::vector<u64> hr(6 * SLOTS);
    CKE(cudaMemcpy(hr.data(), d_ref, hr.size() * 8, cudaMemcpyDeviceToHost));
    Ref ref;
    ref.rows.assign(hr.begin(), hr.begin() + SLOTS); ref.cnull.assign(hr.begin() + SLOTS, hr.begin() + 2 * SLOTS);
    ref.sum.assign(hr.begin() + 2 * SLOTS, hr.begin() + 3 * SLOTS);
    ref.mn.resize(SLOTS); ref.mx.resize(SLOTS);
    for (u64 i = 0; i < SLOTS; ++i) { ref.mn[i] = (i64)hr[4 * SLOTS + i]; ref.mx[i] = (i64)hr[5 * SLOTS + i]; }
    u64 groups = 0, total = 0;
    for (u64 i = 0; i < SLOTS; ++i) { groups += ref.rows[i] != 0; total += ref.rows[i]; }
    fprintf(stderr, "rows %lld, passing %llu, groups %llu\n", (long long)n, (unsigned long long)total, (unsigned long long)groups);

    // ---- base: the generated kernel ----
    {
        u64* d_acc; CKE(cudaMalloc(&d_acc, 5 * SLOTS * 8));
        int* d_status; CKE(cudaMalloc(&d_status, 64)); CKE(cudaMemset(d_status, 0, 64));
        NqParams p; memset(&p, 0, sizeof p);
        p.nrows = n; p.col[0] = d_code; p.tag[0] = d_ktag; p.col[1] = d_v; p.tag[1] = d_vtag; p.acc = d_acc; p.cap_mask = SLOTS - 1; p.status = d_status;
        const size_t smem = (size_t)NQ_CS * 32;
        CKE(cudaFuncSetAttribute(nq_scan_base, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cudaFuncAttributes fa; CKE(cudaFuncGetAttributes(&fa, nq_scan_base));
        cudaEvent_t e0, e1; CKE(cudaEventCreate(&e0)); CKE(cudaEventCreate(&e1));
        float best = 1e30f;
        for (int rep = 0; rep < 4; ++rep) {
            k_fill<<<592, 256>>>(d_acc, 3 * SLOTS, 0);
            k_fill<<<592, 256>>>(d_acc + 3 * SLOTS, SLOTS, (u64)NQ_I64_MAX);
            k_fill<<<592, 256>>>(d_acc + 4 * SLOTS, SLOTS, (u64)NQ_I64_MIN);
            CKE(cudaDeviceSynchronize());
            CKE(cudaEventRecord(e0));
            nq_scan_base<<<sms, NQ_BLOCK, smem>>>(p);
            CKE(cudaEventRecord(e1));
            CKE(cudaDeviceSynchronize());
            CKE(cudaGetLastError());
            float ms; CKE(cudaEventElapsedTime(&ms, e0, e1));
            best = std::min(best, ms);
        }
        std::vector<u64> t(5 * SLOTS);
        CKE(cudaMemcpy(t.data(), d_acc, t.size() * 8, cudaMemcpyDeviceToHost));
        std::vector<u64> rows(SLOTS), cnull(SLOTS); std::vector<i64> sum(SLOTS), mn(SLOTS), mx(SLOTS);
        for (u64 i = 0; i < SLOTS; ++i) { rows[i] = t[i] & 0xffffffffULL; cnull[i] = t[i] >> 32; sum[i] = (i64)t[SLOTS + i]; mn[i] = (i64)t[3 * SLOTS + i]; mx[i] = (i64)t[4 * SLOTS + i]; }
        const bool ok = check("base", ref, rows, cnull, sum, mn, mx);
        printf("{\"variant\": \"base (generated kernel, round 1)\", \"threads\": %d, \"cache_slots\": %d, \"smem\": %zu, \"regs\": %d, \"ms\": %.4f, \"rows_per_s\": %.4g, \"gb_per_s\": %.1f, \"frac\": %.3f, \"check\": \"%s\"}\n",
               NQ_BLOCK, NQ_CS, smem, fa.numRegs, best, n / (best * 1e-3), 14.0 * n / (best * 1e6), 14.0 * n / (best * 1e6) / 6547.8, ok ? "ok" : "MISMATCH");
        fflush(stdout);
        CKE(cudaFree(d_acc));
    }
    u64* d_tab; CKE(cudaMalloc(&d_tab, SLOTS * 4 * 8));
    QParams qp; qp.code = d_code; qp.ktag = d_ktag; qp.v = d_v; qp.vtag = d_vtag; qp.nrows = n; qp.table = d_tab;
    // cache slots: (budget - queues - L0) / 24 bytes, a multiple of 4
    const char* only = getenv("ONLY");
#define RUN(name, ...) if (!only || strstr(name, only)) run_q<__VA_ARGS__>(name, qp, d_tab, ref, n, sms)
    RUN("simple w1 aos", 1024, 8200, 0, 0, 1, 1, 0, 1, 0, 0, 0);
    RUN("simple w1 aos nomnreg", 1024, 8200, 0, 0, 1, 1, 0, 0, 0, 0, 0);
    RUN("simple w1 aos nomnreg 9300", 1024, 9300, 0, 0, 1, 1, 0, 0, 0, 0, 0);
    RUN("simple w1 soa", 1024, 8200, 0, 0, 1, 1, 0, 1, 0, 0, 1);
    RUN("simple w1 aos nocheck", 1024, 8200, 0, 0, 1, 0, 0, 1, 0, 0, 0);
    RUN("simple w1 aos 7040 slots", 1024, 7040, 0, 0, 1, 1, 0, 1, 0, 0, 0);
    RUN("simple w1 aos 9300 slots (no queues)", 1024, 9300, 0, 0, 1, 1, 0, 1, 0, 0, 0);
    RUN("simple w2 aos", 1024, 8200, 0, 0, 2, 1, 0, 1, 0, 0, 0);
    RUN("simple w1 soa 7040", 1024, 7040, 0, 0, 1, 1, 0, 1, 0, 0, 1);
    return 0;
}
