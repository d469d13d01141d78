// n1ql_value.cuh — the N1QL value model and the scan-kernel parameter block, defined once for the host code (g++), the
// static kernels (nvcc) and every generated scan kernel (NVRTC, embedded next to n1ql_device.cuh):
//   value classes and accumulator word operations; Val, one value as class + 64-bit payload
//   number semantics (int64 -> float64 promotion, NewValue canonicalisation), collation, 4-valued logic and the
//   MISSING / NULL folds of the expression operators
//   NqParams, the argument of every scan kernel, with its IN-set descriptors (NqInSet)
// Strings are the one place where the evaluators differ: the kernel holds 2 * dictionary rank as the payload and tests
// truth against the rank of "", the host tail (group_tail.cpp) compares bytes and tests emptiness.
// Everything here is global-scope and host + device; no host or std includes on the NVRTC path.
//
// Reference semantics restated here (reference file:line):
//   value/value.go:69-79 (type order)        value/integer.go:100-130,266-348 (int collate/arith)
//   value/float.go:106-172,331-381            value/string.go:116-142  value/boolean.go:100-114
//   expression/comp_lt.go:57-65 comp_le.go:57-65 comp_eq.go:76-78 comp_between.go:58-78
//   expression/coll_in.go:61-91 logic_and.go:64-88 logic_or.go:98-122 logic_not.go:57-68
//   expression/arith_add.go:51-70 arith_mult.go:51-70 arith_sub.go:53-61 arith_div.go:46-64
//   expression/arith_mod.go:48-66 arith_neg.go:51-59 comp_null.go comp_missing.go comp_valued.go
#pragma once
#ifndef __CUDACC_RTC__
#include <cmath>
#include <cstring>
#endif

#ifdef __CUDACC__
#define N1_HD __host__ __device__ __forceinline__
#else
#define N1_HD inline
#endif

typedef long long i64;
typedef unsigned long long u64;
typedef unsigned int u32;
typedef unsigned char u8;

// value classes: the per-row tag byte of a column.  Ordered so that the N1QL type order
// MISSING < NULL < BOOLEAN(false<true) < NUMBER < STRING is monotone in the class.
enum : int {
    C_MISSING = 0,
    C_NULL = 1,
    C_FALSE = 2,
    C_TRUE = 3,
    C_INT = 4,
    C_FLOAT = 5,
    C_STRING = 6,
    C_OTHER = 7  // array / object / binary: never reaches a kernel (plan is ineligible)
};

#define NQ_I64_MIN ((i64)0x8000000000000000LL)
#define NQ_I64_MAX ((i64)0x7fffffffffffffffLL)
#define NQ_U64_MAX (~(u64)0)

// accumulator word operations (also the merge operation of IntermediateGroup)
enum : int { OP_ADD_U64 = 0, OP_ADD_F64 = 1, OP_MIN_I64 = 2, OP_MAX_I64 = 3, OP_MIN_U64 = 4, OP_MAX_U64 = 5, OP_OR_U64 = 6 };

struct Val {
    int c;  // class
    i64 b;  // payload: int64 | float64 bits | string: 2*dictionary-rank in a kernel (odd = absent constant),
            // dictionary column << 40 | rank in a finalised group
};

N1_HD double as_f(i64 b) {
#ifdef __CUDA_ARCH__
    return __longlong_as_double(b);
#else
    double d;
    memcpy(&d, &b, 8);
    return d;
#endif
}
N1_HD i64 f_bits(double d) {
#ifdef __CUDA_ARCH__
    return __double_as_longlong(d);
#else
    i64 b;
    memcpy(&b, &d, 8);
    return b;
#endif
}

N1_HD Val mkv(int c, i64 b) { Val v; v.c = c; v.b = b; return v; }
N1_HD Val mkbool(bool t) { return mkv(t ? C_TRUE : C_FALSE, 0); }
N1_HD Val mkint(i64 x) { return mkv(C_INT, x); }
N1_HD Val mkflt(double d) { return mkv(C_FLOAT, f_bits(d)); }
N1_HD bool is_num(int c) { return c == C_INT || c == C_FLOAT; }
N1_HD int type_rank(int c) { return c <= C_NULL ? c : (c <= C_TRUE ? 2 : (c <= C_FLOAT ? 3 : 4)); }
N1_HD double num_f(Val v) { return v.c == C_INT ? (double)v.b : as_f(v.b); }

// Go's int64(float64) on amd64 (out of range -> MinInt64) and value.IsInt (integer.go:354-356)
N1_HD i64 go_i64(double d) {
    if (!(d >= -9223372036854775808.0 && d < 9223372036854775808.0)) return NQ_I64_MIN;
    return (i64)d;
}
N1_HD bool f_is_int(double d) { return d == (double)go_i64(d); }
// value.NewValue(float64): integral -> intValue (value/value.go:377-382)
N1_HD Val new_num(double d) { return f_is_int(d) ? mkint(go_i64(d)) : mkflt(d); }
// canonical number identity used by group keys / DISTINCT / MIN / MAX: an integral floatValue
// (only arithmetic can make one) is the equal int (group_util.go:18-35 text form, set.go:83-99)
N1_HD Val canon_num(Val v) {
    if (v.c == C_FLOAT) { double d = as_f(v.b); if (f_is_int(d)) return mkint(go_i64(d)); }
    return v;
}

// ---- collation -------------------------------------------------------------------------------
N1_HD int collate_f(double t, double o) {  // value/float.go:123-172
    bool tn = t != t, on = o != o;
    if (tn) return on ? 0 : -1;
    if (on) return 1;
    return t < o ? -1 : (t > o ? 1 : 0);  // +-Inf order falls out of IEEE compare
}
// same-or-different type collation sign for values > NULL
N1_HD int collate(Val a, Val b) {
    int ra = type_rank(a.c), rb = type_rank(b.c);
    if (ra != rb) return ra - rb;
    if (ra == 3) {
        if (a.c == C_INT && b.c == C_INT) return a.b < b.b ? -1 : (a.b > b.b ? 1 : 0);
        return collate_f(num_f(a), num_f(b));
    }
    if (ra == 2) return a.c - b.c;
    if (ra == 4) return a.b < b.b ? -1 : (a.b > b.b ? 1 : 0);
    return 0;
}
enum : int { CMP_NULL = 8, CMP_MISSING = 9 };
N1_HD int v_compare(Val a, Val b) {  // Value.Compare
    if (a.c == C_MISSING || b.c == C_MISSING) return CMP_MISSING;
    if (a.c == C_NULL || b.c == C_NULL) return CMP_NULL;
    int c = collate(a, b);
    return c < 0 ? -1 : (c > 0 ? 1 : 0);
}
N1_HD Val cmp_result(int cmp, bool t) { return cmp == CMP_MISSING ? mkv(C_MISSING, 0) : (cmp == CMP_NULL ? mkv(C_NULL, 0) : mkbool(t)); }
N1_HD Val v_lt(Val a, Val b) { int c = v_compare(a, b); return cmp_result(c, c < 0); }
N1_HD Val v_le(Val a, Val b) { int c = v_compare(a, b); return cmp_result(c, c <= 0); }
N1_HD Val v_eq(Val a, Val b) {  // Value.Equals
    if (a.c == C_MISSING || b.c == C_MISSING) return mkv(C_MISSING, 0);
    if (a.c == C_NULL || b.c == C_NULL) return mkv(C_NULL, 0);
    int ra = type_rank(a.c), rb = type_rank(b.c);
    if (ra != rb) return mkbool(false);
    if (ra == 3) {
        if (a.c == C_INT && b.c == C_INT) return mkbool(a.b == b.b);
        return mkbool(num_f(a) == num_f(b));
    }
    if (ra == 2) return mkbool(a.c == b.c);
    return mkbool(a.b == b.b);
}
N1_HD Val v_between(Val x, Val lo, Val hi) {  // comp_between.go:58-78
    int lc = v_compare(x, lo);
    if (lc == CMP_MISSING) return mkv(C_MISSING, 0);
    int hc = v_compare(x, hi);
    if (hc == CMP_MISSING) return mkv(C_MISSING, 0);
    if (lc == CMP_NULL || hc == CMP_NULL) return mkv(C_NULL, 0);
    return mkbool(lc >= 0 && hc <= 0);
}
// Value.Truth; empty2 = the payload of "" (kernel: 2*rank of "" in the string operand's dictionary, or -1)
N1_HD bool v_truth(Val v, i64 empty2) {
    if (v.c == C_TRUE) return true;
    if (v.c == C_INT) return v.b != 0;
    if (v.c == C_FLOAT) { double d = as_f(v.b); return d == d && d != 0.0; }
    if (v.c == C_STRING) return v.b != empty2;
    return false;
}
N1_HD Val v_not(Val a, i64 empty2) {
    if (a.c <= C_NULL) return a;
    return mkbool(!v_truth(a, empty2));
}
// n-ary AND / OR folded one argument at a time: flags f(alse seen) / t(rue seen), m(issing), n(ull)
N1_HD void and_arg(Val a, i64 empty2, bool& f, bool& m, bool& n) {
    if (a.c == C_NULL) n = true; else if (a.c == C_MISSING) m = true; else if (!v_truth(a, empty2)) f = true;
}
N1_HD Val and_fin(bool f, bool m, bool n) { return f ? mkbool(false) : (m ? mkv(C_MISSING, 0) : (n ? mkv(C_NULL, 0) : mkbool(true))); }
N1_HD void or_arg(Val a, i64 empty2, bool& t, bool& m, bool& n) {
    if (a.c == C_NULL) n = true; else if (a.c == C_MISSING) m = true; else if (v_truth(a, empty2)) t = true;
}
N1_HD Val or_fin(bool t, bool m, bool n) { return t ? mkbool(true) : (n ? mkv(C_NULL, 0) : (m ? mkv(C_MISSING, 0) : mkbool(false))); }
N1_HD Val v_is_null(Val a) { return a.c == C_NULL ? mkbool(true) : (a.c == C_MISSING ? a : mkbool(false)); }
N1_HD Val v_is_not_null(Val a) { return a.c == C_NULL ? mkbool(false) : (a.c == C_MISSING ? a : mkbool(true)); }
N1_HD Val v_is_missing(Val a) { return mkbool(a.c == C_MISSING); }
N1_HD Val v_is_not_missing(Val a) { return mkbool(a.c != C_MISSING); }
N1_HD Val v_is_valued(Val a) { return mkbool(a.c > C_NULL); }
N1_HD Val v_is_not_valued(Val a) { return mkbool(a.c <= C_NULL); }
// one element of `x IN [..]` (coll_in.go:69-82)
N1_HD void in_arg(Val x, Val e, bool& hit, bool& m, bool& n) {
    if (x.c > C_NULL && e.c > C_NULL) { if (v_eq(x, e).c == C_TRUE) hit = true; }
    else if (e.c == C_MISSING) m = true;
    else n = true;
}
N1_HD Val in_fin(Val x, bool hit, bool m, bool n) {
    if (x.c == C_MISSING) return x;
    return hit ? mkbool(true) : (n ? mkv(C_NULL, 0) : (m ? mkv(C_MISSING, 0) : mkbool(false)));
}

// ---- NumberValue arithmetic ----------------------------------------------------------------------
N1_HD Val num_add(Val a, Val b) {  // integer.go:266-277, float.go:331-333
    if (a.c == C_INT && b.c == C_INT) {
        i64 rv = (i64)((u64)a.b + (u64)b.b);
        if ((a.b >= 0 && b.b >= 0 && rv >= 0) || (a.b < 0 && b.b < 0 && rv < 0)) return mkint(rv);
    }
    return mkflt(num_f(a) + num_f(b));
}
N1_HD Val num_mult(Val a, Val b) {  // integer.go:319-329 (rv/this == n  <=>  no overflow, bar MinInt64 * -1)
    if (a.c == C_INT && b.c == C_INT) {
        i64 lo = (i64)((u64)a.b * (u64)b.b);
#ifdef __CUDA_ARCH__
        i64 hi = __mul64hi(a.b, b.b);
#else
        i64 hi = (i64)(((__int128)a.b * (__int128)b.b) >> 64);
#endif
        bool ok = (hi == (lo >> 63)) || (a.b == -1 && b.b == NQ_I64_MIN);
        if (a.b == NQ_I64_MIN && b.b == -1) ok = false;
        if (ok) return mkint(lo);
    }
    return mkflt(num_f(a) * num_f(b));
}
N1_HD Val num_neg(Val a) {  // integer.go:331-337
    if (a.c == C_INT) { if (a.b == NQ_I64_MIN) return mkflt(-(double)a.b); return mkint(-a.b); }
    return mkflt(-as_f(a.b));
}
N1_HD Val num_sub(Val a, Val b) {  // integer.go:339-348, float.go:375-377
    if (a.c == C_INT && b.c == C_INT && b.b > NQ_I64_MIN) return num_add(a, mkint(-b.b));
    return mkflt(num_f(a) - num_f(b));
}
// n-ary + and * fold (arith_add.go:51-70, arith_mult.go:51-70)
N1_HD void add_arg(Val a, Val& acc, bool& m, bool& n) {
    if (!n && is_num(a.c)) acc = num_add(acc, a); else if (a.c == C_MISSING) m = true; else n = true;
}
N1_HD void mult_arg(Val a, Val& acc, bool& m, bool& n) {
    if (!n && is_num(a.c)) acc = num_mult(acc, a); else if (a.c == C_MISSING) m = true; else n = true;
}
N1_HD Val arith_fin(Val acc, bool m, bool n) { return m ? mkv(C_MISSING, 0) : (n ? mkv(C_NULL, 0) : acc); }
N1_HD Val v_sub(Val a, Val b) {
    if (is_num(a.c) && is_num(b.c)) return num_sub(a, b);
    if (a.c == C_MISSING || b.c == C_MISSING) return mkv(C_MISSING, 0);
    return mkv(C_NULL, 0);
}
N1_HD Val v_neg(Val a) { return is_num(a.c) ? num_neg(a) : (a.c == C_MISSING ? a : mkv(C_NULL, 0)); }
N1_HD Val v_div(Val a, Val b) {  // arith_div.go:46-64
    if (a.c == C_MISSING || b.c == C_MISSING) return mkv(C_MISSING, 0);
    if (is_num(b.c)) {
        double s = num_f(b);
        if (s == 0.0) return mkv(C_NULL, 0);
        if (is_num(a.c)) return new_num(num_f(a) / s);
    }
    return mkv(C_NULL, 0);
}
N1_HD Val v_mod(Val a, Val b) {  // arith_mod.go:48-66 (math.Mod == C fmod)
    if (a.c == C_MISSING || b.c == C_MISSING) return mkv(C_MISSING, 0);
    if (is_num(b.c)) {
        double s = num_f(b);
        if (s == 0.0) return mkv(C_NULL, 0);
        if (is_num(a.c)) return new_num(fmod(num_f(a), s));
    }
    return mkv(C_NULL, 0);
}

// order-preserving u64 image of a float64 (for MIN/MAX through integer atomics)
N1_HD u64 f64_ordered(double d) { u64 u = (u64)f_bits(d); return (u >> 63) ? ~u : (u | 0x8000000000000000ULL); }
N1_HD double f64_unordered(u64 k) { u64 u = (k >> 63) ? (k & 0x7fffffffffffffffULL) : ~k; return as_f((i64)u); }

N1_HD u64 mix64(u64 x) {  // splitmix64 finaliser
    x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ULL; x ^= x >> 27; x *= 0x94d049bb133111ebULL; x ^= x >> 31; return x;
}

// ---- IN over a device-resident set (in_set, n1ql_device.cuh; built by build_inset, codegen.cpp) ---------------------
#define NQ_MAX_INSETS 8
enum : u32 {
    INSET_MISSING = 1,  // some element is MISSING
    INSET_NULL = 2,     // some element is NULL
    INSET_VALUED = 4,   // some element is not MISSING
    INSET_FALSE = 8,
    INSET_TRUE = 16,
    INSET_IEMPTY = 32,  // the INT element -1 (the empty-slot marker)
    INSET_P63 = 64      // the FLOAT element 2^63
};
struct NqInSet {
    const u32* bits;  // STRING: bit r <=> dictionary rank r is an element
    const u64* keys;  // INT table [icap], then FLOAT table [fcap]
    u32 icap, fcap;   // powers of two, 0: no table
    u32 flags;
    u32 pad;
};
// home slot: Fibonacci hashing of the key folded to 32 bits (one 32-bit multiply; mix64 costs two 64-bit ones per row)
N1_HD u32 inset_slot(u64 key, u32 cap) {
#ifdef __CUDA_ARCH__
    return (((u32)key ^ (u32)(key >> 32)) * 0x9E3779B1u) >> (1 + __clz(cap));
#else
    return (((u32)key ^ (u32)(key >> 32)) * 0x9E3779B1u) >> (1 + __builtin_clz(cap));
#endif
}

// status[1] of a wide-key table (MODE_HASHW) whose slot stayed claimed but unpublished past the wait bound: a defect,
// reported as an error (never a hang, never a silently lost row)
#define NQ_WIDE_STUCK 5

// kernel parameter block shared by every generated scan kernel
struct NqParams {
    i64 nrows;             // rows in this partition
    const void* col[16];   // payload arrays (i64* or u32*), 32-byte aligned, padded to a multiple of 4096 rows
    const u8* tag[16];     // class byte per row
    u64* acc;              // UNGROUPED: per-block partials [grid][nwords]; DENSE/HASH: table words [nwords][cap]
    u64* keys;             // HASH: slot keys (u64[cap], ulonglong2[cap], or u64[cap][1 + key words] for wide keys)
    u64 cap_mask;          // HASH: capacity-1
    u64* set_keys;         // DISTINCT entry set (ulonglong2[set_cap] or u64[set_cap])
    u64 set_mask;
    int* status;           // [0] != 0: a table overflowed (host grows it and reruns); [1]: NQ_WIDE_STUCK
    u64 dense_groups;      // DENSE: number of dense slots
    u64* final_dev;        // UNGROUPED: final words [nwords] in HBM (written by the last block to finish)
    u64* final_host;       // UNGROUPED/DENSE: the same words in mapped pinned host memory (zero-copy result)
    unsigned* ticket;      // blocks-done counter for the last-block pattern (self-resetting)
    u64* partials;         // UNGROUPED: per-block partials of the float64-sum words [nfloat][grid]
    // multi-GPU small-state merge fused into the scan: the last block pushes this rank's final words straight into
    // every peer's mailbox over NVLink (peer stores), then publishes a sequence flag (release, system scope)
    u64* const* peer_mail; // [nranks] mailbox base of every rank (peer-mapped; own entry = local pointer), or null
    int nranks, rank;
    u64 mail_base;         // word offset of (slot, this rank) inside a mailbox
    u64 mail_words;        // words pushed per step (accumulator words x slots of the dense table)
    u64 mail_seq;          // sequence number of this step (never 0)
    // DISTINCT bitmap larger than the L2 keeps: the scan runs in passes, pass k sets the bits of entries whose high
    // bits (entry >> set_shift) equal k - a slice of the bitmap that stays L2-resident - and only pass 0 feeds the
    // group table
    int set_pass, set_shift;
    // payloads of the chain's constants and bound parameters (int64 / float64 bits / 2 * dictionary rank): the kernel text
    // only fixes their CLASS, so statements that differ in a bound - or bindings of one prepared statement - share a cubin
    i64 cst[32];
    // execution.Operator.SendStop while the scan runs: a word in HBM that n1gpu_query_cancel sets with an asynchronous copy;
    // lane 0 of every warp polls it once per 32 tiles and the warp leaves the loop
    const int* cancel;
    // `x IN $list` and IN over long literal lists: the list's contents as kernel data (NqInSet), never kernel text
    NqInSet inset[NQ_MAX_INSETS];
};
