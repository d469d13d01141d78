// shred.cu — the device-side columnar shredder: raw JSON documents in HBM -> typed columns, one thread per
// document.  Replaces the per-document work of PrimaryScan + Fetch + lazy field access:
//   value/parsed.go:38-98   type sniff (' ', '\t', '\n' skipped), invalid JSON -> BINARY -> every field MISSING
//   value/parsed.go:159-207 Field(): first occurrence of a name wins; non-object -> MISSING
//   value/value.go:367-430  NewValue: integral float64 -> int64
// Anything the device cannot decide exactly (escape sequences in a relevant key or string value, numbers
// outside the exactly-rounded fast path, nesting deeper than the on-chip stack) is handed to the host
// shredder for that document only ("fix-up rows"); results are identical to table.cpp's host shredder,
// which tests/test_gpu_shredder.py checks row by row.
#include "shred.hpp"
#include "n1ql_device.cuh"

namespace n1 {

#define SH_MAX_DEPTH 24
#define REF_EXTRA_BIT 0x8000000000000000ULL

struct Cur { const unsigned char* p; const unsigned char* e; };

__device__ __forceinline__ void sh_ws(Cur& c) {
    while (c.p < c.e) { unsigned char ch = *c.p; if (ch == ' ' || ch == '\t' || ch == '\n' || ch == '\r') ++c.p; else break; }
}
__device__ __forceinline__ bool sh_hex(unsigned char c) { return (c >= '0' && c <= '9') || ((c | 0x20) >= 'a' && (c | 0x20) <= 'f'); }

// at the opening quote; on success c.p is past the closing quote
__device__ bool sh_string(Cur& c, const unsigned char*& rb, const unsigned char*& re, bool& esc) {
    ++c.p;
    rb = c.p;
    esc = false;
    while (c.p < c.e) {
        unsigned char ch = *c.p;
        if (ch == '"') { re = c.p; ++c.p; return true; }
        if (ch == '\\') {
            esc = true;
            ++c.p;
            if (c.p >= c.e) return false;
            unsigned char e = *c.p;
            if (e == 'u') {
                if (c.e - c.p < 5) return false;
                if (!(sh_hex(c.p[1]) && sh_hex(c.p[2]) && sh_hex(c.p[3]) && sh_hex(c.p[4]))) return false;
                c.p += 5;
            } else if (e == '"' || e == '\\' || e == '/' || e == 'b' || e == 'f' || e == 'n' || e == 'r' || e == 't') ++c.p;
            else return false;
            continue;
        }
        if (ch < 0x20) return false;
        ++c.p;
    }
    return false;
}

__constant__ double sh_pow10[23] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};

// 0 invalid, 1 int64 in iv, 2 float64 in dv (exactly rounded fast path), 3 valid but needs the host
__device__ int sh_number(Cur& c, i64& iv, double& dv) {
    bool neg = false;
    if (c.p < c.e && *c.p == '-') { neg = true; ++c.p; }
    if (c.p >= c.e) return 0;
    u64 mant = 0;
    int sig = 0;        // significant digits accumulated
    bool big = false;   // more than 19 significant digits
    int exp10 = 0;
    if (*c.p == '0') { ++c.p; if (c.p < c.e && *c.p >= '0' && *c.p <= '9') return 0; }
    else if (*c.p >= '1' && *c.p <= '9') {
        while (c.p < c.e && *c.p >= '0' && *c.p <= '9') {
            if (sig < 19) { mant = mant * 10 + (u64)(*c.p - '0'); ++sig; } else { big = true; ++exp10; }
            ++c.p;
        }
    } else return 0;
    bool frac = false;
    if (c.p < c.e && *c.p == '.') {
        frac = true;
        ++c.p;
        if (c.p >= c.e || !(*c.p >= '0' && *c.p <= '9')) return 0;
        while (c.p < c.e && *c.p >= '0' && *c.p <= '9') {
            if (sig < 19) { if (mant != 0 || *c.p != '0') { mant = mant * 10 + (u64)(*c.p - '0'); ++sig; } --exp10; }
            else if (*c.p != '0') big = true;
            ++c.p;
        }
    }
    if (c.p < c.e && (*c.p == 'e' || *c.p == 'E')) {
        frac = true;
        ++c.p;
        bool eneg = false;
        if (c.p < c.e && (*c.p == '+' || *c.p == '-')) { eneg = *c.p == '-'; ++c.p; }
        if (c.p >= c.e || !(*c.p >= '0' && *c.p <= '9')) return 0;
        int ev = 0;
        while (c.p < c.e && *c.p >= '0' && *c.p <= '9') { if (ev < 100000) ev = ev * 10 + (*c.p - '0'); ++c.p; }
        exp10 += eneg ? -ev : ev;
    }
    if (!frac) {
        if (big) return 3;  // beyond int64: float64 on the host
        if (!neg) { if (mant > 0x7fffffffffffffffULL) return 3; iv = (i64)mant; return 1; }
        if (mant > 0x8000000000000000ULL) return 3;
        iv = (i64)(0ULL - mant);
        return 1;
    }
    if (big) return 3;
    if (mant == 0) { dv = 0.0; return 2; }
    if (mant > (1ULL << 53)) return 3;
    double d = (double)mant;
    if (exp10 < 0) { if (exp10 < -22) return 3; d = d / sh_pow10[-exp10]; }
    else { if (exp10 > 22) return 3; d = d * sh_pow10[exp10]; }
    dv = neg ? -d : d;
    return 2;
}

__device__ __forceinline__ bool sh_literal(Cur& c, const char* w, int n) {
    if (c.e - c.p < n) return false;
    for (int i = 0; i < n; ++i) if (c.p[i] != (unsigned char)w[i]) return false;
    c.p += n;
    return true;
}

struct Out {
    u8* const* tags;
    i64* const* payload;
    i64 row;
    __device__ __forceinline__ void put(int col, u8 tag, i64 pay) const {
        if (tags[col][row] != C_MISSING) return;  // first occurrence wins
        tags[col][row] = tag;
        payload[col][row] = pay;
    }
};

// returns 0 ok, 1 invalid JSON (row all MISSING), 2 needs the host
__device__ int sh_document(const unsigned char* base, i64 b, i64 e, const ShredTrie& T, const Out& out) {  // T lives in global memory
    Cur c{base + b, base + e};
    while (c.p < c.e && (*c.p == ' ' || *c.p == '\t' || *c.p == '\n')) ++c.p;  // identifyType
    if (c.p >= c.e || *c.p != '{') return 1;  // non-object documents have no fields
    unsigned is_obj_bits = 0;        // bit d: frame d is an object
    short node[SH_MAX_DEPTH];        // trie node of frame d (-1: nothing below is wanted)
    int depth = 0;
    // open the root object
    ++c.p;
    is_obj_bits |= 1u;
    node[0] = 0;
    depth = 1;
    bool expect_first = true;        // just after '{' or '[': a close bracket is allowed
    for (;;) {
        const bool in_obj = (is_obj_bits >> (depth - 1)) & 1u;
        sh_ws(c);
        if (c.p >= c.e) return 1;
        unsigned char ch = *c.p;
        bool closing = false;
        if (expect_first && ch == (in_obj ? '}' : ']')) {
            ++c.p;
            closing = true;
        } else {
            int kid = -1;
            if (in_obj) {
                if (ch != '"') return 1;
                const unsigned char *rb, *re;
                bool esc;
                if (!sh_string(c, rb, re, esc)) return 1;
                const int n = node[depth - 1];
                if (n >= 0 && T.kid_end[n] > T.kid_begin[n]) {
                    if (esc) return 2;  // an escaped name could spell a wanted one: host decides
                    const int len = (int)(re - rb);
                    for (int k = T.kid_begin[n]; k < T.kid_end[n]; ++k) {
                        if (T.name_len[k] != len) continue;
                        bool eq = true;
                        for (int i = 0; i < len; ++i) if (rb[i] != (unsigned char)T.names[T.name_off[k] + i]) { eq = false; break; }
                        if (eq) { kid = T.kid_node[k]; break; }
                    }
                }
                sh_ws(c);
                if (c.p >= c.e || *c.p != ':') return 1;
                ++c.p;
                sh_ws(c);
                if (c.p >= c.e) return 1;
                ch = *c.p;
            }
            const int col = kid >= 0 ? T.col[kid] : -1;
            if (ch == '{' || ch == '[') {
                if (col >= 0) out.put(col, C_OTHER, 0);
                if (depth >= SH_MAX_DEPTH) return 2;
                const bool o = ch == '{';
                if (o) is_obj_bits |= (1u << depth); else is_obj_bits &= ~(1u << depth);
                node[depth] = (short)((o && kid >= 0 && T.kid_end[kid] > T.kid_begin[kid]) ? kid : -1);
                ++depth;
                ++c.p;
                expect_first = true;
                continue;
            }
            if (ch == '"') {
                const unsigned char *rb, *re;
                bool esc;
                if (!sh_string(c, rb, re, esc)) return 1;
                if (col >= 0) {
                    if (esc) return 2;
                    const u64 len = (u64)(re - rb);
                    if (len >= (1ULL << 24)) return 2;
                    out.put(col, C_STRING, (i64)((((u64)(rb - base)) << 24) | len));
                }
            } else if (ch == 't') { if (!sh_literal(c, "true", 4)) return 1; if (col >= 0) out.put(col, C_TRUE, 0); }
            else if (ch == 'f') { if (!sh_literal(c, "false", 5)) return 1; if (col >= 0) out.put(col, C_FALSE, 0); }
            else if (ch == 'n') { if (!sh_literal(c, "null", 4)) return 1; if (col >= 0) out.put(col, C_NULL, 0); }
            else {
                i64 iv; double dv;
                const int k = sh_number(c, iv, dv);
                if (k == 0) return 1;
                if (col >= 0) {
                    if (k == 3) return 2;
                    if (k == 1) out.put(col, C_INT, iv);
                    else if (f_is_int(dv)) out.put(col, C_INT, go_i64(dv));  // NewValue canonicalisation
                    else out.put(col, C_FLOAT, __double_as_longlong(dv));
                }
            }
        }
        // after a value (or a close): ',' continues the container, its close bracket pops it
        for (;;) {
            if (closing) {
                closing = false;
                --depth;
                if (depth == 0) {
                    sh_ws(c);
                    return c.p == c.e ? 0 : 1;  // trailing garbage -> invalid
                }
            }
            sh_ws(c);
            if (c.p >= c.e) return 1;
            const bool o = (is_obj_bits >> (depth - 1)) & 1u;
            if (*c.p == ',') { ++c.p; expect_first = false; break; }
            if (*c.p == (o ? '}' : ']')) { ++c.p; closing = true; continue; }
            return 1;
        }
    }
}

__global__ void __launch_bounds__(128) k_shred_json(const unsigned char* __restrict__ buf, const i64* __restrict__ offs, i64 first, i64 ndocs, const ShredTrie* __restrict__ Tp,
                                                    u8* const* tags, i64* const* payload, int ncols, unsigned* fix_count, i64* fix_rows, i64 fix_cap) {
    for (i64 row = first + (i64)blockIdx.x * blockDim.x + threadIdx.x; row < first + ndocs; row += (i64)gridDim.x * blockDim.x) {
        Out out{tags, payload, row};
        const int rc = sh_document(buf, offs[row], offs[row + 1], *Tp, out);
        if (rc != 0) {
            for (int c = 0; c < ncols; ++c) { tags[c][row] = C_MISSING; payload[c][row] = 0; }
            if (rc == 2) {
                const unsigned at = atomicAdd(fix_count, 1u);
                if ((i64)at < fix_cap) fix_rows[at] = row;
            }
        }
    }
}

// ---- NDJSON: document offsets computed on the device -----------------------------------------------------------------
// A document starts where a line starts (position 0 or behind a line end) unless the line is blank (only ' ', '\t', '\r'
// before its end).  One thread per 256-byte segment counts / writes the document starts of its segment; a scan over the
// segment counts in between gives every segment its first document index.  The text is read at HBM speed twice - the
// host would spend a pass of its memory bandwidth per step, and the offsets (8 bytes per document) never cross PCIe.
#define NL_SEG 256
__device__ __forceinline__ bool nl_doc_start(const unsigned char* __restrict__ t, i64 size, i64 p) {
    for (i64 a = p; a < size; ++a) {
        const unsigned char c = t[a];
        if (c == ' ' || c == '\t' || c == '\r') continue;
        return c != '\n';
    }
    return false;
}
template <bool WRITE>
__global__ void k_ndjson_lines(const unsigned char* __restrict__ t, i64 size, i64 nseg, unsigned* __restrict__ counts, const i64* __restrict__ first,
                               i64* __restrict__ offs) {
    for (i64 seg = (i64)blockIdx.x * blockDim.x + threadIdx.x; seg < nseg; seg += (i64)gridDim.x * blockDim.x) {
        const i64 lo = seg * NL_SEG, hi = lo + NL_SEG < size ? lo + NL_SEG : size;
        unsigned n = 0;
        i64 at = WRITE ? first[seg] : 0;
        if (seg == 0 && size > 0 && nl_doc_start(t, size, 0)) { if (WRITE) offs[at++] = 0; ++n; }
        for (i64 p = lo; p < hi; p += 16) {
            const uint4 v = *reinterpret_cast<const uint4*>(t + p);  // (the buffer is padded: reading past `size` is harmless)
            const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const unsigned x = w[k] ^ 0x0a0a0a0au;
                unsigned z = (x - 0x01010101u) & ~x & 0x80808080u;
                while (z) {
                    const i64 e = p + 4 * k + ((__ffs((int)z) - 1) >> 3);
                    z &= z - 1;
                    if (e < hi && t[e] == '\n' && e + 1 < size && nl_doc_start(t, size, e + 1)) { if (WRITE) offs[at++] = e + 1; ++n; }
                }
            }
        }
        if (!WRITE) counts[seg] = n;
    }
}
// exclusive scan of the segment counts: first[seg], first[nseg] = total.  Three launches - per-tile totals (a tile = 8192
// segments, one block each), the scan of those totals by one block, the tiles' own scans on top of their bases - instead of one
// block walking all tiles (10^7 segments of a 680 MB keyspace: 2 ms -> tens of microseconds).
#define NQ_SCAN_TILE (1024 * 8)
__device__ __forceinline__ i64 block_exclusive_scan_1024(i64 mine, i64* s_warp, i64& total) {
    // exclusive prefix of `mine` over the 1024 threads of the block; total = sum over the block
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    i64 incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const i64 up = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += up; }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        i64 w = s_warp[lane], wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const i64 up = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += up; }
        s_warp[lane] = wi - w;       // exclusive prefix of the warp totals
        if (lane == 31) s_warp[32] = wi;  // block total
    }
    __syncthreads();
    total = s_warp[32];
    const i64 r = s_warp[warp] + incl - mine;
    __syncthreads();
    return r;
}
__global__ void __launch_bounds__(1024) k_scan_tile_totals(const unsigned* __restrict__ counts, i64 nseg, i64* __restrict__ tile_total) {
    __shared__ i64 s_warp[33];
    const i64 mine = (i64)blockIdx.x * NQ_SCAN_TILE + (i64)threadIdx.x * 8;
    i64 sum = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) sum += mine + k < nseg ? (i64)counts[mine + k] : 0;
    i64 total;
    block_exclusive_scan_1024(sum, s_warp, total);
    if (threadIdx.x == 0) tile_total[blockIdx.x] = total;
}
// one block: tile_total[0..ntiles) -> exclusive prefix in place, grand total at tile_total[ntiles]
__global__ void __launch_bounds__(1024) k_scan_tile_bases(i64* __restrict__ tile_total, i64 ntiles) {
    __shared__ i64 s_warp[33];
    __shared__ i64 s_base;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (i64 t0 = 0; t0 < ntiles; t0 += 1024) {
        const i64 i = t0 + threadIdx.x;
        const i64 v = i < ntiles ? tile_total[i] : 0;
        i64 total;
        const i64 ex = block_exclusive_scan_1024(v, s_warp, total);
        if (i < ntiles) tile_total[i] = s_base + ex;
        __syncthreads();
        if (threadIdx.x == 0) s_base += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) tile_total[ntiles] = s_base;
}
__global__ void __launch_bounds__(1024) k_scan_counts(const unsigned* __restrict__ counts, i64 nseg, const i64* __restrict__ tile_base, i64 ntiles,
                                                      i64* __restrict__ first) {
    __shared__ i64 s_warp[33];
    // every thread owns 8 consecutive segments of its block's tile
    const i64 mine = (i64)blockIdx.x * NQ_SCAN_TILE + (i64)threadIdx.x * 8;
    i64 v[8], sum = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { v[k] = mine + k < nseg ? (i64)counts[mine + k] : 0; sum += v[k]; }
    i64 total;
    i64 run = tile_base[blockIdx.x] + block_exclusive_scan_1024(sum, s_warp, total);
#pragma unroll
    for (int k = 0; k < 8; ++k) { if (mine + k < nseg) first[mine + k] = run; run += v[k]; }
    if (blockIdx.x == 0 && threadIdx.x == 0) first[nseg] = tile_base[ntiles];
}
// device offsets of the documents `rows` (fix-up rows): out[2 * i] = offs[rows[i]], out[2 * i + 1] = offs[rows[i] + 1]
__global__ void k_gather_offsets(const i64* __restrict__ offs, const i64* __restrict__ rows, i64 n, i64* out) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) { out[2 * i] = offs[rows[i]]; out[2 * i + 1] = offs[rows[i] + 1]; }
}

// ---- dictionary encoding ------------------------------------------------------------------------------------------
__device__ __forceinline__ const unsigned char* ref_ptr(u64 ref, const unsigned char* buf, const unsigned char* extra) {
    return ((ref & REF_EXTRA_BIT) ? extra : buf) + ((ref & ~REF_EXTRA_BIT) >> 24);
}
__device__ __forceinline__ bool ref_equal(u64 a, u64 b, const unsigned char* buf, const unsigned char* extra) {
    const u64 la = a & 0xffffff, lb = b & 0xffffff;
    if (la != lb) return false;
    const unsigned char *pa = ref_ptr(a, buf, extra), *pb = ref_ptr(b, buf, extra);
    for (u64 i = 0; i < la; ++i) if (pa[i] != pb[i]) return false;
    return true;
}
// payload[row] (a string ref) -> slot of the string's representative in `keys` (EMPTY = all ones)
__global__ void k_dict_insert(const unsigned char* __restrict__ buf, const unsigned char* __restrict__ extra, const u8* __restrict__ tags,
                              const i64* __restrict__ payload, i64* __restrict__ slots, i64 nrows, u64* keys, u64 cap_mask, int* status) {
    for (i64 row = (i64)blockIdx.x * blockDim.x + threadIdx.x; row < nrows; row += (i64)gridDim.x * blockDim.x) {
        if (tags[row] != C_STRING) continue;
        if (*(volatile int*)status) return;  // the table proved too small: the host grows it and reruns, nothing here is kept
        const u64 ref = (u64)payload[row];
        const unsigned char* p = ref_ptr(ref, buf, extra);
        const u64 len = ref & 0xffffff;
        u64 h = 1469598103934665603ULL;
        for (u64 i = 0; i < len; ++i) { h ^= p[i]; h *= 1099511628211ULL; }
        u64 slot = mix64(h) & cap_mask;
        bool done = false;
        // (a probe sequence this long means the table is far too dense: every step compares string bytes)
        for (u64 probe = 0; probe <= cap_mask && probe < 128; ++probe) {
            u64 cur = *(volatile u64*)&keys[slot];
            if (cur == NQ_U64_MAX) {
                const u64 old = atomicCAS(&keys[slot], NQ_U64_MAX, ref);
                if (old == NQ_U64_MAX) { done = true; break; }
                cur = old;
            }
            if (ref_equal(cur, ref, buf, extra)) { done = true; break; }
            slot = (slot + 1) & cap_mask;
        }
        if (!done) { status[0] = 1; continue; }
        slots[row] = (i64)slot;
    }
}
// occupied slots -> (slot, ref) pairs
__global__ void k_dict_collect(const u64* __restrict__ keys, u64 cap, unsigned* count, u64* out_slots, u64* out_refs, u64 out_cap) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += (u64)gridDim.x * blockDim.x) {
        const u64 k = keys[i];
        if (k == NQ_U64_MAX) continue;
        const unsigned at = atomicAdd(count, 1u);
        if (at < out_cap) { out_slots[at] = i; out_refs[at] = k; }
    }
}
// rank[slot_of_rank[r]] = r: the ranks of the occupied dictionary slots (only those are ever read)
__global__ void k_dict_ranks(const u64* __restrict__ slot_of_rank, u64 n, u32* rank) {
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (u64)gridDim.x * blockDim.x) rank[slot_of_rank[r]] = (u32)r;
}
// slot -> rank; writes 8-byte payload in place, or the narrow 4-byte array when out32 != null
__global__ void k_dict_remap(const u8* __restrict__ tags, const i64* __restrict__ slots, i64* payload, u32* out32, i64 nrows,
                             const u32* __restrict__ rank) {
    for (i64 row = (i64)blockIdx.x * blockDim.x + threadIdx.x; row < nrows; row += (i64)gridDim.x * blockDim.x) {
        u32 r = 0;
        if (tags[row] == C_STRING) { r = rank[slots[row]]; payload[row] = (i64)r; }
        if (out32) out32[row] = r;
    }
}
// column statistics: stats[0] class mask, [1] int min, [2] int max (as i64), [3] has float, [4] MISSING / NULL rows
__global__ void k_col_stats(const u8* __restrict__ tags, const i64* __restrict__ payload, i64 nrows, u64* stats) {
    u64 mask = 0, hasf = 0, absent = 0;
    i64 mn = NQ_I64_MAX, mx = NQ_I64_MIN;
    for (i64 row = (i64)blockIdx.x * blockDim.x + threadIdx.x; row < nrows; row += (i64)gridDim.x * blockDim.x) {
        const int t = tags[row];
        mask |= 1ULL << t;
        absent += t <= C_NULL;
        if (t == C_INT && payload) { const i64 v = payload[row]; mn = v < mn ? v : mn; mx = v > mx ? v : mx; }
        else if (t == C_FLOAT) hasf = 1;
    }
    __shared__ u64 scratch[32];
    mask = block_reduce_word<OP_OR_U64>(mask, scratch);
    hasf = block_reduce_word<OP_OR_U64>(hasf, scratch);
    u64 rmn = block_reduce_word<OP_MIN_I64>((u64)mn, scratch);
    u64 rmx = block_reduce_word<OP_MAX_I64>((u64)mx, scratch);
    absent = block_reduce_word<OP_ADD_U64>(absent, scratch);
    if (threadIdx.x == 0) {
        atomicAdd(&stats[4], absent);
        atomicOr(&stats[0], mask);
        atomicMin((i64*)&stats[1], (i64)rmn);
        atomicMax((i64*)&stats[2], (i64)rmx);
        atomicOr(&stats[3], hasf);
    }
}
// pre-shredded input may hold integral floats: value.NewValue turns them into ints (value/value.go:377-382)
__global__ void k_canon_floats(u8* tags, i64* payload, i64 nrows) {
    for (i64 row = (i64)blockIdx.x * blockDim.x + threadIdx.x; row < nrows; row += (i64)gridDim.x * blockDim.x) {
        if (tags[row] != C_FLOAT) continue;
        const double d = __longlong_as_double(payload[row]);
        if (f_is_int(d)) { tags[row] = C_INT; payload[row] = go_i64(d); }
    }
}
// host fix-ups: (row, tag, payload) triples for one column
__global__ void k_patch(u8* tags, i64* payload, const i64* __restrict__ rows, const u8* __restrict__ ptags, const i64* __restrict__ ppay, i64 n) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        tags[rows[i]] = ptags[i];
        payload[rows[i]] = ppay[i];
    }
}

// ---- splice: a refreshed table's column from the old column and the re-read documents (execution.cpp, refresh) ---------
// Row r of the new table comes from run k with new_lo[k] <= r < new_lo[k + 1]: row src_lo[k] + (r - new_lo[k]) of the old
// column, or of the patch column when bit 63 of src_lo[k] is set.  A tile of SPLICE_TILE rows looks its first and last
// runs up once; its rows then search only between those two (one run in the common case).
#define SPLICE_TILE 256
#define SPLICE_PATCH_BIT 0x8000000000000000ULL
__device__ __forceinline__ i64 splice_find(const i64* __restrict__ new_lo, i64 lo, i64 hi, i64 row) {
    while (lo < hi) { const i64 m = (lo + hi + 1) >> 1; if (new_lo[m] <= row) lo = m; else hi = m - 1; }
    return lo;
}
__device__ __forceinline__ void splice_tile_runs(const i64* __restrict__ new_lo, i64 nruns, i64 t0, i64 nrows, i64* s_runs) {
    if (threadIdx.x == 0) {
        s_runs[0] = splice_find(new_lo, 0, nruns - 1, t0);
        const i64 last = t0 + SPLICE_TILE - 1 < nrows ? t0 + SPLICE_TILE - 1 : nrows - 1;
        s_runs[1] = splice_find(new_lo, s_runs[0], nruns - 1, last);
    }
    __syncthreads();
}
__device__ __forceinline__ i64 splice_payload(const i64* __restrict__ pay8, const u32* __restrict__ pay4, i64 row) {
    return pay8 ? pay8[row] : (pay4 ? (i64)pay4[row] : 0);
}
// Pre-pass over the rows kept from the old column: the dictionary ranks they still use (bitmap) and their classes.
__global__ void __launch_bounds__(SPLICE_TILE) k_splice_used(const i64* __restrict__ new_lo, const i64* __restrict__ src_lo, i64 nruns, i64 nrows,
                                                            const u8* __restrict__ tags, const i64* __restrict__ pay8, const u32* __restrict__ pay4,
                                                            u32* used, u64* class_mask) {
    __shared__ i64 s_runs[2];
    __shared__ u64 scratch[32];
    u64 mask = 0;
    for (i64 t0 = (i64)blockIdx.x * SPLICE_TILE; t0 < nrows; t0 += (i64)gridDim.x * SPLICE_TILE) {
        splice_tile_runs(new_lo, nruns, t0, nrows, s_runs);
        const i64 row = t0 + threadIdx.x;
        if (row < nrows) {
            const i64 k = splice_find(new_lo, s_runs[0], s_runs[1], row);
            const u64 src = (u64)src_lo[k];
            if (!(src & SPLICE_PATCH_BIT)) {
                const i64 at = (i64)src + (row - new_lo[k]);
                const int t = tags[at];
                mask |= 1ULL << t;
                if (t == C_STRING) { const u64 r = (u64)splice_payload(pay8, pay4, at); atomicOr(&used[r >> 5], 1u << (r & 31)); }
            }
        }
        __syncthreads();  // s_runs is rewritten by the next tile
    }
    mask = block_reduce_word<OP_OR_U64>(mask, scratch);
    if (threadIdx.x == 0 && mask) atomicOr(class_mask, mask);
}
// The new column: every padded row written once - spliced rows at the new width with ranks remapped into the new dictionary,
// rows past nrows MISSING with a zero payload (as seal() pads them).
__global__ void __launch_bounds__(SPLICE_TILE) k_splice_gather(const i64* __restrict__ new_lo, const i64* __restrict__ src_lo, i64 nruns, i64 nrows, i64 padded,
                                                              const u8* __restrict__ o_tags, const i64* __restrict__ o_pay8, const u32* __restrict__ o_pay4,
                                                              const u32* __restrict__ o_remap,
                                                              const u8* __restrict__ p_tags, const i64* __restrict__ p_pay8, const u32* __restrict__ p_pay4,
                                                              const u32* __restrict__ p_remap,
                                                              u8* __restrict__ tags, i64* __restrict__ pay8, u32* __restrict__ pay4) {
    __shared__ i64 s_runs[2];
    for (i64 t0 = (i64)blockIdx.x * SPLICE_TILE; t0 < padded; t0 += (i64)gridDim.x * SPLICE_TILE) {
        if (t0 < nrows) splice_tile_runs(new_lo, nruns, t0, nrows, s_runs);
        const i64 row = t0 + threadIdx.x;
        u8 t = C_MISSING;
        i64 v = 0;
        if (row < nrows) {
            const i64 k = splice_find(new_lo, s_runs[0], s_runs[1], row);
            const u64 src = (u64)src_lo[k];
            const bool patch = (src & SPLICE_PATCH_BIT) != 0;
            const i64 at = (i64)(src & ~SPLICE_PATCH_BIT) + (row - new_lo[k]);
            t = patch ? p_tags[at] : o_tags[at];
            v = patch ? splice_payload(p_pay8, p_pay4, at) : splice_payload(o_pay8, o_pay4, at);
            if (t == C_STRING) v = (i64)(patch ? p_remap : o_remap)[v];
        }
        if (row < padded) {
            tags[row] = t;
            if (pay8) pay8[row] = v;
            else if (pay4) pay4[row] = (u32)v;
        }
        if (t0 < nrows) __syncthreads();
    }
}

static int sgrid(i64 n, int block) {
    i64 g = (n + block - 1) / block;
    if (g < 1) g = 1;
    if (g > 148 * 32) g = 148 * 32;
    return (int)g;
}

void launch_shred_json(const unsigned char* buf, const i64* offs, i64 first, i64 ndocs, const ShredTrie* T, u8* const* tags, i64* const* payload,
                       int ncols, unsigned* fix_count, i64* fix_rows, i64 fix_cap, cudaStream_t s) {
    if (ndocs <= 0) return;
    k_shred_json<<<sgrid(ndocs, 128), 128, 0, s>>>(buf, offs, first, ndocs, T, tags, payload, ncols, fix_count, fix_rows, fix_cap);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
i64 ndjson_segments(i64 size) { return (size + NL_SEG - 1) / NL_SEG; }
i64 ndjson_scan_tiles(i64 nseg) { return std::max<i64>(1, (nseg + NQ_SCAN_TILE - 1) / NQ_SCAN_TILE); }
void launch_ndjson_count(const unsigned char* text, i64 size, unsigned* counts, cudaStream_t s) {
    const i64 nseg = ndjson_segments(size);
    if (!nseg) return;
    k_ndjson_lines<false><<<sgrid(nseg, 128), 128, 0, s>>>(text, size, nseg, counts, nullptr, nullptr);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_ndjson_scan(const unsigned* counts, i64 nseg, i64* first, i64* tile_scratch, cudaStream_t s) {
    const i64 ntiles = ndjson_scan_tiles(nseg);
    k_scan_tile_totals<<<(unsigned)ntiles, 1024, 0, s>>>(counts, nseg, tile_scratch);
    k_scan_tile_bases<<<1, 1024, 0, s>>>(tile_scratch, ntiles);
    k_scan_counts<<<(unsigned)ntiles, 1024, 0, s>>>(counts, nseg, tile_scratch, ntiles, first);
    g_launches.fetch_add(3);
    CK(cudaGetLastError());
}
void launch_ndjson_write(const unsigned char* text, i64 size, const i64* first, i64* offs, cudaStream_t s) {
    const i64 nseg = ndjson_segments(size);
    if (!nseg) return;
    k_ndjson_lines<true><<<sgrid(nseg, 128), 128, 0, s>>>(text, size, nseg, nullptr, first, offs);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_gather_offsets(const i64* offs, const i64* rows, i64 n, i64* out, cudaStream_t s) {
    if (n == 0) return;
    k_gather_offsets<<<sgrid(n, 256), 256, 0, s>>>(offs, rows, n, out);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_dict_insert(const unsigned char* buf, const unsigned char* extra, const u8* tags, const i64* payload, i64* slots, i64 nrows,
                        u64* keys, u64 cap, int* status, cudaStream_t s) {
    k_dict_insert<<<sgrid(nrows, 256), 256, 0, s>>>(buf, extra, tags, payload, slots, nrows, keys, cap - 1, status);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_dict_collect(const u64* keys, u64 cap, unsigned* count, u64* out_slots, u64* out_refs, u64 out_cap, cudaStream_t s) {
    k_dict_collect<<<sgrid((i64)cap, 256), 256, 0, s>>>(keys, cap, count, out_slots, out_refs, out_cap);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
// ranks of one dictionary -> ranks of a sorted superset (multi-GPU dictionary agreement on columns that live in HBM)
__global__ void k_rank_remap(const u8* __restrict__ tags, i64* pay8, u32* pay4, i64 nrows, const u32* __restrict__ remap, u32 n) {
    for (i64 row = (i64)blockIdx.x * blockDim.x + threadIdx.x; row < nrows; row += (i64)gridDim.x * blockDim.x) {
        if (tags[row] != C_STRING) continue;
        if (pay4) { const u32 r = pay4[row]; if (r < n) pay4[row] = remap[r]; }
        else { const u64 r = (u64)pay8[row]; if (r < n) pay8[row] = (i64)remap[r]; }
    }
}
void launch_rank_remap(const u8* tags, i64* pay8, u32* pay4, i64 nrows, const u32* remap, u32 n, cudaStream_t s) {
    if (nrows == 0 || n == 0) return;
    k_rank_remap<<<sgrid(nrows, 256), 256, 0, s>>>(tags, pay8, pay4, nrows, remap, n);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
__global__ void k_widen_ranks(const u32* __restrict__ pay4, i64* __restrict__ pay8, i64 nrows) {
    for (i64 row = (i64)blockIdx.x * blockDim.x + threadIdx.x; row < nrows; row += (i64)gridDim.x * blockDim.x) pay8[row] = (i64)pay4[row];
}
void launch_widen_ranks(const u32* pay4, i64* pay8, i64 nrows, cudaStream_t s) {
    if (nrows == 0) return;
    k_widen_ranks<<<sgrid(nrows, 256), 256, 0, s>>>(pay4, pay8, nrows);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_dict_ranks(const u64* slot_of_rank, u64 n, u32* rank, cudaStream_t s) {
    if (n == 0) return;
    k_dict_ranks<<<sgrid((i64)n, 256), 256, 0, s>>>(slot_of_rank, n, rank);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_dict_remap(const u8* tags, const i64* slots, i64* payload, u32* out32, i64 nrows, const u32* rank, cudaStream_t s) {
    k_dict_remap<<<sgrid(nrows, 256), 256, 0, s>>>(tags, slots, payload, out32, nrows, rank);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_col_stats(const u8* tags, const i64* payload, i64 nrows, u64* stats, cudaStream_t s) {
    k_col_stats<<<sgrid(nrows, 256) > 592 ? 592 : sgrid(nrows, 256), 256, 0, s>>>(tags, payload, nrows, stats);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_canon_floats(u8* tags, i64* payload, i64 nrows, cudaStream_t s) {
    if (nrows == 0) return;
    k_canon_floats<<<sgrid(nrows, 256), 256, 0, s>>>(tags, payload, nrows);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_splice_used(const SpliceRuns& r, const u8* tags, const i64* pay8, const u32* pay4, u32* used, u64* class_mask, cudaStream_t s) {
    if (r.nrows == 0) return;
    k_splice_used<<<sgrid(r.nrows, SPLICE_TILE), SPLICE_TILE, 0, s>>>(r.new_lo, r.src_lo, r.nruns, r.nrows, tags, pay8, pay4, used, class_mask);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_splice_gather(const SpliceRuns& r, i64 padded, const u8* o_tags, const i64* o_pay8, const u32* o_pay4, const u32* o_remap,
                          const u8* p_tags, const i64* p_pay8, const u32* p_pay4, const u32* p_remap, u8* tags, i64* pay8, u32* pay4, cudaStream_t s) {
    k_splice_gather<<<sgrid(padded, SPLICE_TILE), SPLICE_TILE, 0, s>>>(r.new_lo, r.src_lo, r.nruns, r.nrows, padded, o_tags, o_pay8, o_pay4, o_remap,
                                                                      p_tags, p_pay8, p_pay4, p_remap, tags, pay8, pay4);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}
void launch_patch(u8* tags, i64* payload, const i64* rows, const u8* ptags, const i64* ppay, i64 n, cudaStream_t s) {
    if (n == 0) return;
    k_patch<<<sgrid(n, 256), 256, 0, s>>>(tags, payload, rows, ptags, ppay, n);
    g_launches.fetch_add(1);
    CK(cudaGetLastError());
}

}  // namespace n1
