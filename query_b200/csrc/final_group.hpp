// final_group.hpp — FinalGroup of one group: the bit-packed group key decoded into (class, payload) per component and
// ComputeFinal applied to every aggregate.  One restatement, compiled by g++ for the host finalisation (Query::finalize)
// and by nvcc for the device one (k_finalize_groups), so that a group finalises alike whichever path a chain takes.
//
// Reference behaviour restated here:
//   algebra/agg_count.go:95-149, agg_countn.go:77-129   counts are int64
//   algebra/agg_sum.go:77-136 + value/integer.go:266-277  int64 sum stays int while every operand shares a
//       sign class and the total fits, otherwise float64
//   algebra/agg_avg.go:117-131   float64(sum)/float64(count), then value.NewValue (integral -> int)
//   algebra/agg_min.go:76-127, agg_max.go:76-127   collation winner over any type, NULL when nothing counted
//   algebra/agg_*_distinct.go + value/set.go:65-110  DISTINCT sets; SUM starts from int 0 (0 + negative -> float)
//   execution/group_final.go:55-118   one item per group
#pragma once
#include <cstdint>

#include "n1ql_value.cuh"

namespace n1 {

enum class AggKind : signed char { COUNT, COUNTN, SUM, AVG, MIN, MAX };

// One bit-packed component (PackComp as plain data): a group-key value or the value of a DISTINCT entry
struct FinalComp {
    int cbits, pbits, nfree, biased, dict_col, nclasses;
    i64 bias;
    int classes[8];
};

// What finalises one aggregate; AggPlan (codegen.hpp) adds what only the code generator needs.  Word indices are LOGICAL
// words (< 64, -1 = absent); the fields are small because the descriptor of a chain's aggregates is a kernel argument.
struct FinalAgg {
    AggKind kind = AggKind::COUNT;
    bool distinct = false;
    signed char w_cnt = -1;
    signed char w_isum = -1;              // exact single-word int sum (range proves no overflow)
    signed char w_ilo = -1, w_ihi = -1;   // split int sum: sum of low 32 bits / sum of (x >> 32)
    signed char w_nint = -1, w_neg = -1;  // ints summed / negative ints among them (intValue.Add: mixed signs -> float64)
    signed char w_fsum = -1, w_nflt = -1;
    // the sign mix of the summed ints read off MIN / MAX of the same operand (any negative <=> min < 0, any non-negative
    // <=> max >= 0) instead of a counter of negatives: one accumulator word (and one cache cell) less
    signed char w_sgn_min = -1, w_sgn_max = -1;
    // "float-carried" sum of an operand that mixes INT and FLOAT values whose ints are provably small (|x| * rows < 2^53):
    // every number is added to ONE float64 word (integers that small add exactly in float64, so an all-INT group still
    // gets its exact int64 sum), w_nnum counts the numbers, and three bits of a shared OR word remember whether a float,
    // a negative int or a non-negative int was seen (the int / float class of the result: value/integer.go:266-277).
    bool fcarry = false;
    signed char w_nnum = -1, w_flags = -1, flag_shift = 0;
    signed char w_seen = -1, w_mi = -1, w_mf = -1, w_ms = -1;
    signed char w_seen_cnt = -1, seen_class = -1;  // single-class operand: "seen" = (this count word > 0) ? bit(seen_class) : 0
    signed char dict_col = -1;                     // MIN / MAX string: the operand's column (a table has at most 16)
};

// A chain's finalisation: how logical words sit in the physical words of the table, and its key components / aggregates.
struct FinalDesc {
    int nkeys, naggs, LW, PW;
    unsigned char phys_of[64], shift_of[64], bits_of[64], complement[64];
    FinalComp keys[16];  // device finalisation only (Query::device_final_ok); the host passes its components separately
    FinalAgg aggs[24];
};

// the next n bits of v (low bits first)
N1_HD u64 take_bits(unsigned __int128& v, int n) {
    if (n == 0) return 0;
    const u64 r = n >= 64 ? (u64)v : ((u64)v & ((1ULL << n) - 1));
    v >>= n;
    return r;
}

// the next component of a packed key or DISTINCT entry
N1_HD Val decode_comp(const FinalComp& pc, unsigned __int128& bits) {
    u64 ci = take_bits(bits, pc.cbits);
    u64 pv = take_bits(bits, pc.pbits);
    if (pc.nfree >= 0) {  // offset packing: one field
        ci = pv < (u64)pc.nfree ? pv : (u64)pc.nfree;
        pv = pv < (u64)pc.nfree ? 0 : pv - (u64)pc.nfree;
    }
    const int cls = ci < (u64)pc.nclasses ? pc.classes[ci] : C_MISSING;
    switch (cls) {
        case C_INT: return {C_INT, pc.biased ? (i64)(pv + (u64)pc.bias) : (i64)pv};
        case C_FLOAT: return {C_FLOAT, (i64)pv};
        case C_STRING: return {C_STRING, (i64)(((u64)pc.dict_col << 40) | (pv & 0xffffffffffULL))};
        case C_NULL: case C_FALSE: case C_TRUE: return {cls, 0};
        default: return {C_MISSING, 0};
    }
}

// The logical words of a group from its physical words pw: packed counter fields extracted, complemented counters
// (KernelPlan::word_complement) restored from logical word 0, the group's row count
N1_HD void logical_words(const FinalDesc& D, const u64* pw, u64* w) {
    for (int l = 0; l < D.LW; ++l) {
        const u64 v = pw[D.phys_of[l]];
        w[l] = D.bits_of[l] == 64 ? v : (v >> D.shift_of[l]) & 0xffffffffULL;
    }
    for (int l = 0; l < D.LW; ++l) if (D.complement[l]) w[l] = w[0] - w[l];
}

// the SUM value as the reference's NumberValue chain would leave it (see the header comment)
N1_HD Val sum_value(__int128 itotal, u64 n_nonneg, u64 n_neg, u64 n_flt, double fsum, bool from_zero) {
    const u64 nI = n_nonneg + n_neg;
    if (nI + n_flt == 0) return {C_NULL, 0};
    if (n_flt == 0) {
        const bool same_sign = from_zero ? (n_neg == 0) : (n_neg == 0 || n_nonneg == 0);
        if (same_sign && itotal >= (__int128)INT64_MIN && itotal <= (__int128)INT64_MAX) return {C_INT, (i64)itotal};
        return mkflt((double)itotal);
    }
    if (nI == 0) return mkflt(fsum);
    return mkflt((double)itotal + fsum);
}

// ComputeFinal of one aggregate from the group's logical words
N1_HD Val final_agg(const FinalAgg& ap, const u64* w) {
    if (ap.distinct) {
        const u64 count = w[ap.w_cnt];
        if (ap.kind == AggKind::COUNT || ap.kind == AggKind::COUNTN) return {C_INT, (i64)count};
        if (count == 0) return {C_NULL, 0};
        __int128 itotal = 0;  // entries of SUM / AVG DISTINCT are numbers only
        u64 n_neg = 0, n_flt = 0;
        double fsum = 0;
        if (ap.w_ilo >= 0) itotal = (((__int128)(i64)w[ap.w_ihi]) << 32) + (__int128)w[ap.w_ilo];
        if (ap.w_neg >= 0) n_neg = w[ap.w_neg];
        if (ap.w_nflt >= 0) n_flt = w[ap.w_nflt];
        if (ap.w_fsum >= 0) fsum = as_f((i64)w[ap.w_fsum]);
        const Val sv = sum_value(itotal, count - n_neg - n_flt, n_neg, n_flt, fsum, true);
        return ap.kind == AggKind::SUM ? sv : new_num(num_f(sv) / (double)count);
    }
    if (ap.kind == AggKind::COUNT || ap.kind == AggKind::COUNTN) return {C_INT, (i64)w[ap.w_cnt]};
    if (ap.fcarry) {
        const u64 count = w[ap.w_nnum], flags = (w[ap.w_flags] >> ap.flag_shift) & 7;
        const double fs = as_f((i64)w[ap.w_fsum]);
        if (count == 0) return {C_NULL, 0};
        // a float, or ints of both signs (intValue.Add went float): float; else the exact int total
        const Val sv = ((flags & 1) || ((flags & 2) && (flags & 4))) ? mkflt(fs) : Val{C_INT, (i64)fs};
        return ap.kind == AggKind::SUM ? sv : new_num(num_f(sv) / (double)count);
    }
    if (ap.kind == AggKind::SUM || ap.kind == AggKind::AVG) {
        __int128 itotal = 0;
        u64 n_neg = 0, n_nonneg = 0, n_flt = 0;
        double fsum = 0;
        if (ap.w_isum >= 0) itotal = (i64)w[ap.w_isum];
        else if (ap.w_ilo >= 0) itotal = (((__int128)(i64)w[ap.w_ihi]) << 32) + (__int128)w[ap.w_ilo];
        if (ap.w_neg >= 0) n_neg = w[ap.w_neg];
        if (ap.w_nint >= 0) n_nonneg = w[ap.w_nint] - n_neg;
        if (ap.w_sgn_min >= 0 && ap.w_nint >= 0 && w[ap.w_nint]) {  // the sign mix from MIN / MAX of the operand
            const bool any_neg = (i64)w[ap.w_sgn_min] < 0, any_nonneg = (i64)w[ap.w_sgn_max] >= 0;
            n_neg = any_neg ? (any_nonneg ? 1 : w[ap.w_nint]) : 0;
            n_nonneg = w[ap.w_nint] - n_neg;
        }
        if (ap.w_nflt >= 0) n_flt = w[ap.w_nflt];
        if (ap.w_fsum >= 0) fsum = as_f((i64)w[ap.w_fsum]);
        const Val sv = sum_value(itotal, n_nonneg, n_neg, n_flt, fsum, false);
        if (ap.kind == AggKind::SUM || sv.c == C_NULL) return sv;
        return new_num(num_f(sv) / (double)(n_nonneg + n_neg + n_flt));
    }
    // MIN / MAX: the collation winner over the classes seen
    const bool mn = ap.kind == AggKind::MIN;
    const u64 seen = ap.w_seen >= 0 ? w[ap.w_seen] : (w[ap.w_seen_cnt] ? (1ULL << ap.seen_class) : 0);
    const bool hi = seen & (1ULL << C_INT), hf = seen & (1ULL << C_FLOAT);
    const i64 iv = ap.w_mi >= 0 ? (i64)w[ap.w_mi] : 0;
    const double fv = ap.w_mf >= 0 ? f64_unordered(w[ap.w_mf]) : 0;
    Val number;
    if (hi && hf) {  // intValue.Collate(floatValue): float64 compare (value/integer.go:100-118)
        const double ad = (double)iv;
        number = (mn ? (ad <= fv) : (ad >= fv)) ? Val{C_INT, iv} : mkflt(fv);
    } else number = hi ? Val{C_INT, iv} : mkflt(fv);
    const Val str{C_STRING, ap.w_ms >= 0 ? (i64)(((u64)ap.dict_col << 40) | (w[ap.w_ms] & 0xffffffffffULL)) : 0};
    const u64 M_NUMB = (1ULL << C_INT) | (1ULL << C_FLOAT);
    if (seen == 0) return {C_NULL, 0};
    if (mn) {
        if (seen & (1ULL << C_FALSE)) return {C_FALSE, 0};
        if (seen & (1ULL << C_TRUE)) return {C_TRUE, 0};
        return (seen & M_NUMB) ? number : str;
    }
    if (seen & (1ULL << C_STRING)) return str;
    if (seen & M_NUMB) return number;
    return {(seen & (1ULL << C_TRUE)) ? C_TRUE : C_FALSE, 0};
}

// FinalGroup of one group: its nkeys key components decoded from the packed key (khi:klo), its aggregates finalised from
// its physical words pw, into key_cls / key_val [nkeys] and agg_cls / agg_val [D.naggs]
N1_HD void final_group(const FinalDesc& D, const FinalComp* keys, int nkeys, u64 klo, u64 khi, const u64* pw, u8* key_cls,
                       i64* key_val, u8* agg_cls, i64* agg_val) {
    u64 w[64];
    logical_words(D, pw, w);
    unsigned __int128 kb = ((unsigned __int128)khi << 64) | klo;
    for (int k = 0; k < nkeys; ++k) {
        const Val v = decode_comp(keys[k], kb);
        key_cls[k] = (u8)v.c;
        key_val[k] = v.b;
    }
    for (int a = 0; a < D.naggs; ++a) {
        const Val v = final_agg(D.aggs[a], w);
        agg_cls[a] = (u8)v.c;
        agg_val[a] = v.b;
    }
}

}  // namespace n1
