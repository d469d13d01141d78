// codegen.cpp — emits the specialised scan kernel for one Filter + Group chain.
//
// The kernel is straight-line CUDA over the hand-written device library n1ql_device.cuh: per thread and
// iteration 4 consecutive rows are fetched with one 256-bit (8-byte columns), 128-bit (4-byte dictionary
// ranks) or 32-bit (class bytes) coalesced load per referenced column, the Filter condition is evaluated
// with N1QL's 4-valued logic, a warp ballot of the selection skips the aggregation when no lane passes,
// and the aggregates are folded into
//   MODE_UNGROUPED  per-thread registers -> block reduction -> persistent accumulators / ordered float partials,
//                   folded and published by the last block (one launch per step, programmatic dependent launch)
//   MODE_DENSE      a table indexed by the bit-packed group key: in shared memory when it fits (thread-private
//                   copies for a handful of groups), else direct-indexed in HBM (dense_global) behind the
//                   shared-memory front cache
//   MODE_HASH64/128 an HBM open-addressing table claimed with 64-/128-bit CAS (64: behind the front cache)
//   MODE_HASHW      the same for keys wider than 127 bits: a tag word claimed with a CAS, then the key words
// DISTINCT aggregates add bit-packed (set, group, value) entries to a bitmap or an HBM hash set.
// The planner (plan_layout and its stages) turns static type analysis (expr.cpp), column statistics and the N1GPU_*
// knobs into the KernelPlan: which accumulator words exist, how wide keys and entries are, which layout above is
// generated.  It writes no text; the emitters turn the plan and the bound expressions into text and decide nothing.
#include "codegen.hpp"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <set>

namespace n1 {

namespace {

struct StrCtx {
    int dict_col = -1;
    std::vector<std::string> locals;  // sorted constants when no dictionary is involved
};

std::string lit_i64(i64 v) { return strf("((i64)0x%016llxULL)", (unsigned long long)(u64)v); }
const char* op_name(int op) {
    static const char* n[] = {"OP_ADD_U64", "OP_ADD_F64", "OP_MIN_I64", "OP_MAX_I64", "OP_MIN_U64", "OP_MAX_U64", "OP_OR_U64"};
    return n[op];
}
const char* cls_name(int c) {
    static const char* n[] = {"C_MISSING", "C_NULL", "C_FALSE", "C_TRUE", "C_INT", "C_FLOAT", "C_STRING", "C_OTHER"};
    return n[c];
}

// open-addressing table of `keys` at load <= 0.25 (short clusters: a warp waits for its longest probe), probed like
// inset_probe (n1ql_device.cuh)
std::vector<u64> inset_table(std::vector<u64> keys) {
    std::sort(keys.begin(), keys.end());
    keys.erase(std::unique(keys.begin(), keys.end()), keys.end());
    if (keys.empty()) return {};
    u64 cap = 2;
    while (cap < 4 * keys.size()) cap <<= 1;
    if (cap > ((u64)1 << 31)) N1_THROW(N1GPU_E_INELIGIBLE, "IN list of %zu numbers", keys.size());
    std::vector<u64> tab(cap, ~(u64)0);
    for (u64 k : keys) {
        u64 s = inset_slot(k, (u32)cap);
        while (tab[s] != ~(u64)0) s = (s + 1) & (cap - 1);
        tab[s] = k;
    }
    return tab;
}

// the set of `x IN [constants]`; string elements are looked up in the dictionary of the operand column `dict_col`
InSet build_inset(const Table& t, const Expr& list, int dict_col) {
    InSet s;
    std::vector<u64> ik, fk;
    if (dict_col >= 0) s.bits.assign((t.cols[dict_col].dict.size() + 31) / 32 + 1, 0u);
    for (auto& el : list.ops) {
        const HValue& v = el->cval;
        s.flags |= v.cls == C_MISSING ? INSET_MISSING : INSET_VALUED;
        switch (v.cls) {
            case C_NULL: s.flags |= INSET_NULL; break;
            case C_FALSE: s.flags |= INSET_FALSE; break;
            case C_TRUE: s.flags |= INSET_TRUE; break;
            case C_INT: {
                if ((u64)v.bits == ~(u64)0) s.flags |= INSET_IEMPTY; else ik.push_back((u64)v.bits);
                const double d = (double)v.bits;  // float64 image for FLOAT rows (v_eq: float64(a) == float64(b))
                u64 b;
                memcpy(&b, &d, 8);
                fk.push_back(d == 0.0 ? 0 : b);
                break;
            }
            case C_FLOAT: {
                const double d = v.f();
                if (d != d) break;  // NaN equals nothing
                if (d == 9223372036854775808.0) s.flags |= INSET_P63;
                fk.push_back(d == 0.0 ? 0 : (u64)v.bits);
                break;
            }
            case C_STRING: {
                if (dict_col < 0) break;  // the operand is never a string
                const auto& d = t.cols[dict_col].dict;
                auto it = std::lower_bound(d.begin(), d.end(), v.s);
                if (it != d.end() && *it == v.s) { const size_t r = (size_t)(it - d.begin()); s.bits[r >> 5] |= 1u << (r & 31); }
                break;
            }
            default: break;
        }
    }
    s.ikeys = inset_table(ik);
    s.fkeys = inset_table(fk);
    return s;
}

struct Gen {
    const Table& t;
    std::string body;
    std::string decls;  // column Val declarations, hoisted to the top of the row body
    int tmp = 0;
    std::string ind = "                ";
    std::map<int, std::string> colvar;  // per-row cache of column Val variables
    std::vector<i64> consts;            // payloads handed to the kernel as p.cst[k] (at most 32; more stay literals)
    std::vector<InSet> in_sets;         // handed to the kernel as p.inset[k]
    std::map<const Expr*, int> in_set_of;  // an IN emitted twice (operand of two aggregates) uses one set
    explicit Gen(const Table& tt) : t(tt) {}
    // the payload of a constant as an expression: a kernel argument slot of its own (numbered by occurrence, never by
    // value: the text must not depend on the payloads), else a literal
    std::string payload_ref(i64 bits) {
        if (consts.size() < 32) { consts.push_back(bits); return strf("p.cst[%d]", (int)consts.size() - 1); }
        return lit_i64(bits);
    }

    std::string nv(const char* p = "v") { return strf("%s%d", p, tmp++); }
    void line(const std::string& s) { body += ind + s + "\n"; }
    // `const Val r = f(args);`: a new value r, numbered after the arguments
    std::string call(const char* f, const std::vector<std::string>& args) {
        std::string r = nv(), list;
        for (auto& a : args) list += (list.empty() ? "" : ", ") + a;
        line(strf("const Val %s = %s(%s);", r.c_str(), f, list.c_str()));
        return r;
    }
    void open(const std::string& head) { line(head); ind += "    "; }  // a block: `head` ... close()
    void close() { ind.resize(ind.size() - 4); line("}"); }

    i64 const_code(const std::string& s, const StrCtx* cx) {
        if (cx && cx->dict_col >= 0) {
            const auto& d = t.cols[cx->dict_col].dict;
            auto it = std::lower_bound(d.begin(), d.end(), s);
            i64 lb = it - d.begin();
            if (it != d.end() && *it == s) return 2 * lb;
            return 2 * lb - 1;  // absent: sorts strictly between its neighbours, equals nothing
        }
        if (cx) {
            auto it = std::lower_bound(cx->locals.begin(), cx->locals.end(), s);
            return 2 * (i64)(it - cx->locals.begin()) + 2;
        }
        return s.empty() ? 0 : 2;
    }
    // 2*rank of "" for the truth value of a string-capable operand (-1: cannot be empty)
    i64 empty2_of(const Expr& e) {
        if (!(e.ti.mask & bit(C_STRING))) return -1;
        if (e.kind == EK::CONST) return 0;
        if (e.ti.plain_col) { i64 r = t.cols[e.ti.dict_col].stats.empty_rank; return r < 0 ? -1 : 2 * r; }
        N1_THROW(N1GPU_E_INELIGIBLE, "truth value of a computed string");
    }

    std::string colval(int c) {
        auto it = colvar.find(c);
        if (it != colvar.end()) return it->second;
        const Column& col = t.cols[c];
        u32 mask = col.stats.class_mask ? col.stats.class_mask : bit(C_MISSING);
        std::string cls;
        if (col.stats.uniform_tag() || col.stats.class_mask == 0) {
            int only = 0;
            for (int k = 0; k < 8; ++k) if (mask & bit(k)) only = k;
            cls = cls_name(only);
        } else {
            // normalise the tag to the classes that occur so the compiler can prune the others
            std::vector<int> cs;
            for (int k = 0; k < 8; ++k) if (mask & bit(k)) cs.push_back(k);
            std::string e = cls_name(cs.back());
            for (int k = (int)cs.size() - 2; k >= 0; --k) e = strf("(t%d[j] == %s ? %s : %s)", c, cls_name(cs[k]), cls_name(cs[k]), e.c_str());
            cls = e;
        }
        std::string pay;
        bool has_str = mask & bit(C_STRING);
        if (col.width == 8) {
            if (has_str) pay = strf("(t%d[j] == C_STRING ? c%d[j] * 2 : c%d[j])", c, c, c);
            else pay = strf("c%d[j]", c);
        } else if (col.width == 4) pay = strf("((i64)c%d[j] * 2)", c);
        else pay = "0";
        std::string v = nv("col");
        decls += strf("            const Val %s = mkv(%s, %s);\n", v.c_str(), cls.c_str(), pay.c_str());
        colvar[c] = v;
        return v;
    }

    StrCtx make_ctx(const Expr& e) {
        StrCtx cx;
        cx.dict_col = e.ti.dict_col;
        if (cx.dict_col < 0) {
            std::vector<const Expr*> flat;
            for (auto& o : e.ops) {
                if (o->kind == EK::ARRAY) for (auto& el : o->ops) flat.push_back(el.get()); else flat.push_back(o.get());
            }
            for (auto* x : flat) if (x->kind == EK::CONST && x->cval.cls == C_STRING) cx.locals.push_back(x->cval.s);
            std::sort(cx.locals.begin(), cx.locals.end());
            cx.locals.erase(std::unique(cx.locals.begin(), cx.locals.end()), cx.locals.end());
        }
        return cx;
    }

    std::string emit(const Expr& e, const StrCtx* cx) {
        switch (e.kind) {
            case EK::CONST: {
                std::string v = nv();
                const HValue& c = e.cval;
                if (c.cls == C_STRING) line(strf("const Val %s = mkv(C_STRING, %s);", v.c_str(), payload_ref(const_code(c.s, cx)).c_str()));
                else if (c.cls == C_INT || c.cls == C_FLOAT) line(strf("const Val %s = mkv(%s, %s);", v.c_str(), cls_name(c.cls), payload_ref(c.bits).c_str()));
                else line(strf("const Val %s = mkv(%s, 0);", v.c_str(), cls_name(c.cls)));
                return v;
            }
            case EK::FIELD: return colval(e.col);
            case EK::ADD: case EK::MULT: {
                std::string acc = nv("acc"), m = nv("m"), n = nv("n"), r = nv();
                std::vector<std::string> args;
                for (auto& o : e.ops) args.push_back(emit(*o, nullptr));
                line(strf("Val %s = mkint(%d); bool %s = false, %s = false;", acc.c_str(), e.kind == EK::ADD ? 0 : 1, m.c_str(), n.c_str()));
                for (auto& a : args) line(strf("%s(%s, %s, %s, %s);", e.kind == EK::ADD ? "add_arg" : "mult_arg", a.c_str(), acc.c_str(), m.c_str(), n.c_str()));
                line(strf("const Val %s = arith_fin(%s, %s, %s);", r.c_str(), acc.c_str(), m.c_str(), n.c_str()));
                return r;
            }
            case EK::SUB: case EK::DIV: case EK::MOD:
                return call(e.kind == EK::SUB ? "v_sub" : (e.kind == EK::DIV ? "v_div" : "v_mod"), {emit(*e.ops[0], nullptr), emit(*e.ops[1], nullptr)});
            case EK::NEG: return call("v_neg", {emit(*e.ops[0], nullptr)});
            case EK::EQ: case EK::LT: case EK::LE: {
                StrCtx c2 = make_ctx(e);
                return call(e.kind == EK::EQ ? "v_eq" : (e.kind == EK::LT ? "v_lt" : "v_le"), {emit(*e.ops[0], &c2), emit(*e.ops[1], &c2)});
            }
            case EK::BETWEEN: {
                StrCtx c2 = make_ctx(e);
                return call("v_between", {emit(*e.ops[0], &c2), emit(*e.ops[1], &c2), emit(*e.ops[2], &c2)});
            }
            case EK::IN: {
                const Expr& list = *e.ops[1];
                const bool str_opnd = e.ops[0]->ti.mask & bit(C_STRING);
                if (in_takes_set(e)) {
                    if (str_opnd && !e.ops[0]->ti.plain_col) N1_THROW(N1GPU_E_INELIGIBLE, "IN over an array parameter with a constant string operand");
                    const std::string x = emit(*e.ops[0], nullptr);
                    auto it = in_set_of.find(&e);
                    int k;
                    if (it != in_set_of.end()) k = it->second;
                    else {
                        if ((int)in_sets.size() >= NQ_MAX_INSETS) N1_THROW(N1GPU_E_INELIGIBLE, "more than %d IN sets in one chain", NQ_MAX_INSETS);
                        k = (int)in_sets.size();
                        in_sets.push_back(build_inset(t, list, str_opnd ? e.ops[0]->ti.dict_col : -1));
                        in_set_of[&e] = k;
                    }
                    return call("in_set", {x, strf("p.inset[%d]", k)});
                }
                StrCtx c2 = make_ctx(e);
                std::string x = emit(*e.ops[0], &c2);
                std::string h = nv("h"), m = nv("m"), n = nv("n"), r = nv();
                line(strf("bool %s = false, %s = false, %s = false;", h.c_str(), m.c_str(), n.c_str()));
                for (auto& el : e.ops[1]->ops) {
                    std::string ev = emit(*el, &c2);
                    line(strf("in_arg(%s, %s, %s, %s, %s);", x.c_str(), ev.c_str(), h.c_str(), m.c_str(), n.c_str()));
                }
                line(strf("const Val %s = in_fin(%s, %s, %s, %s);", r.c_str(), x.c_str(), h.c_str(), m.c_str(), n.c_str()));
                return r;
            }
            case EK::AND: case EK::OR: {
                std::string f = nv("f"), m = nv("m"), n = nv("n"), r = nv();
                std::vector<std::pair<std::string, i64>> args;
                for (auto& o : e.ops) { std::string a = emit(*o, nullptr); args.emplace_back(a, empty2_of(*o)); }
                line(strf("bool %s = false, %s = false, %s = false;", f.c_str(), m.c_str(), n.c_str()));
                for (auto& a : args)
                    line(strf("%s(%s, %lldLL, %s, %s, %s);", e.kind == EK::AND ? "and_arg" : "or_arg", a.first.c_str(), (long long)a.second, f.c_str(), m.c_str(), n.c_str()));
                line(strf("const Val %s = %s(%s, %s, %s);", r.c_str(), e.kind == EK::AND ? "and_fin" : "or_fin", f.c_str(), m.c_str(), n.c_str()));
                return r;
            }
            case EK::NOT: return call("v_not", {emit(*e.ops[0], nullptr), strf("%lldLL", (long long)empty2_of(*e.ops[0]))});
            case EK::IS_NULL: case EK::IS_NOT_NULL: case EK::IS_MISSING: case EK::IS_NOT_MISSING: case EK::IS_VALUED: case EK::IS_NOT_VALUED:
                return call(e.kind == EK::IS_NULL ? "v_is_null" : e.kind == EK::IS_NOT_NULL ? "v_is_not_null" : e.kind == EK::IS_MISSING ? "v_is_missing"
                            : e.kind == EK::IS_NOT_MISSING ? "v_is_not_missing" : e.kind == EK::IS_VALUED ? "v_is_valued" : "v_is_not_valued",
                            {emit(*e.ops[0], nullptr)});
            case EK::ARRAY: N1_THROW(N1GPU_E_INELIGIBLE, "array value outside IN");
            case EK::AGG: N1_THROW(N1GPU_E_INELIGIBLE, "nested aggregate");
            case EK::IDENT: N1_THROW(N1GPU_E_INELIGIBLE, "bare identifier");
            case EK::ROUND: N1_THROW(N1GPU_E_INELIGIBLE, "round() on the GPU path");
            case EK::PARAM: N1_THROW(N1GPU_E_INVALID, "No value for parameter $%s.", e.name.c_str());
        }
        N1_THROW(N1GPU_E_INVALID, "unhandled expression kind");
    }
};

// Packed component for a value with TypeInfo ti (after canon_num when it is not a plain column).
PackComp make_comp(const Table& t, const Expr& e, const char* what, bool offset_pack) {
    PackComp pc;
    TypeInfo ti = e.ti;
    if (ti.mask & bit(C_STRING)) {
        if (!ti.plain_col) N1_THROW(N1GPU_E_INELIGIBLE, "%s over a constant or computed string", what);
        pc.dict_col = ti.dict_col;
    }
    if (!ti.plain_col && (ti.mask & bit(C_FLOAT))) { ti.mask |= bit(C_INT); ti.ranged = false; }  // canon_num
    pc.mask = ti.mask;
    for (int k = 0; k < 7; ++k) if (ti.mask & bit(k)) pc.classes.push_back(k);
    pc.cbits = bits_for(pc.classes.size());
    int pb = 0;
    if (ti.mask & bit(C_INT)) {
        if (ti.ranged && (u64)ti.hi - (u64)ti.lo < ((u64)1 << 62)) {
            pc.biased = true; pc.bias = ti.lo;
            pb = std::max(pb, bits_for((u64)ti.hi - (u64)ti.lo + 1));
        } else pb = 64;
    }
    if (ti.mask & bit(C_FLOAT)) pb = 64;
    if (ti.mask & bit(C_STRING)) pb = std::max(pb, bits_for((u64)std::max<i64>(1, t.cols[pc.dict_col].stats.ndict)));
    pc.pbits = pb;
    // offset packing: exactly one payload class, bounded
    {
        const bool has_i = ti.mask & bit(C_INT), has_f = ti.mask & bit(C_FLOAT), has_s = ti.mask & bit(C_STRING);
        if (offset_pack && pc.classes.size() > 1 && !has_f && (has_i != has_s) && (!has_i || pc.biased) && pb < 62) {
            const int pcls = has_i ? C_INT : C_STRING;
            const u64 range = has_i ? (u64)ti.hi - (u64)ti.lo + 1 : (u64)std::max<i64>(1, t.cols[pc.dict_col].stats.ndict);
            const int nfree = (int)pc.classes.size() - 1;
            const int nb = bits_for((u64)nfree + range);
            if (nb < pc.cbits + pc.pbits) {
                std::vector<int> order;
                for (int c : pc.classes) if (c != pcls) order.push_back(c);
                order.push_back(pcls);
                pc.classes = order;
                pc.nfree = nfree;
                pc.range = range;
                pc.cbits = 0;
                pc.pbits = nb;
            }
        }
    }
    return pc;
}

// number of distinct packed values of a component (0: too many to matter)
u64 comp_values(const Table& t, const PackComp& pc) {
    if (pc.bits() > 20) return 0;
    if (pc.nfree >= 0) return (u64)pc.nfree + pc.range;
    if (pc.cbits == 0 && pc.classes.size() == 1) {
        if (pc.classes[0] == C_STRING) return (u64)std::max<i64>(1, t.cols[pc.dict_col].stats.ndict);
        if (pc.classes[0] != C_INT && pc.classes[0] != C_FLOAT) return 1;
    }
    return (u64)1 << pc.bits();
}

// The fields of Val `v` packed as component pc: the whole offset-packed value (nfree >= 0), else the class index (integer
// literals with suffix `sfx`) and the payload
std::string offset_field(const PackComp& pc, const std::string& v) {
    const int pcls = pc.classes.back();
    std::string pay = pcls == C_STRING ? strf("((u64)%s.b >> 1)", v.c_str()) : strf("((u64)%s.b - (u64)%s)", v.c_str(), lit_i64(pc.bias).c_str());
    std::string e = strf("(%dULL + %s)", pc.nfree, pay.c_str());
    for (int k = pc.nfree - 1; k >= 0; --k) e = strf("(%s.c == %s ? %dULL : %s)", v.c_str(), cls_name(pc.classes[k]), k, e.c_str());
    return e;
}
std::string class_field(const PackComp& pc, const std::string& v, const char* sfx) {
    std::string e = strf("%d%s", (int)pc.classes.size() - 1, sfx);
    for (int k = (int)pc.classes.size() - 2; k >= 0; --k) e = strf("(%s.c == %s ? %d%s : %s)", v.c_str(), cls_name(pc.classes[k]), k, sfx, e.c_str());
    return e;
}
std::string payload_field(const PackComp& pc, const std::string& v) {
    std::string e = "0ULL";
    if (pc.mask & bit(C_STRING)) e = strf("(%s.c == C_STRING ? ((u64)%s.b >> 1) : %s)", v.c_str(), v.c_str(), e.c_str());
    if (pc.mask & bit(C_FLOAT)) e = strf("(%s.c == C_FLOAT ? (u64)%s.b : %s)", v.c_str(), v.c_str(), e.c_str());
    if (pc.mask & bit(C_INT)) {
        std::string iv = pc.biased ? strf("((u64)%s.b - (u64)%s)", v.c_str(), lit_i64(pc.bias).c_str()) : strf("(u64)%s.b", v.c_str());
        e = strf("(%s.c == C_INT ? %s : %s)", v.c_str(), iv.c_str(), e.c_str());
    }
    return e;
}

// Emits code packing Val `v` as component pc into (lo,hi,pos) variables, or with hi == nullptr into the u64 array `lo`
// (MODE_HASHW keys); with `radix` also adds the component's packed value times `radix_stride` to the variable of that
// name (mixed-radix slot of a dense shared-memory table).
void emit_pack(Gen& g, const PackComp& pc, const std::string& v, const char* lo, const char* hi, const char* pos,
               const char* radix = nullptr, u64 radix_stride = 0) {
    const std::string dst = hi ? strf("%s, %s, %s", lo, hi, pos) : strf("%s, %s", lo, pos);
    if (radix && pc.bits() > 0) {
        // the whole component as one value: class index in the low cbits, payload above
        std::string cv = g.nv("cv");
        if (pc.nfree >= 0) g.line(strf("const u64 %s = %s;", cv.c_str(), offset_field(pc, v).c_str()));
        else g.line(strf("const u64 %s = %s | (%s << %d);", cv.c_str(), pc.cbits ? class_field(pc, v, "ULL").c_str() : "0ULL",
                         pc.pbits ? payload_field(pc, v).c_str() : "0ULL", pc.cbits));
        g.line(strf("pack_bits(%s, %s, %d);", dst.c_str(), cv.c_str(), pc.bits()));
        g.line(strf("%s += %s * %lluULL;", radix, cv.c_str(), (unsigned long long)radix_stride));
        return;
    }
    if (pc.nfree >= 0) { g.line(strf("pack_bits(%s, %s, %d);", dst.c_str(), offset_field(pc, v).c_str(), pc.pbits)); return; }
    if (pc.cbits) g.line(strf("pack_bits(%s, (u64)%s, %d);", dst.c_str(), class_field(pc, v, "").c_str(), pc.cbits));
    if (pc.pbits) g.line(strf("pack_bits(%s, %s, %d);", dst.c_str(), payload_field(pc, v).c_str(), pc.pbits));
}

double comp_domain(const Table& t, const PackComp& pc) {
    double d = 0;
    for (int c : pc.classes) {
        if (c == C_INT) d += pc.nfree >= 0 ? (double)pc.range : (pc.biased ? std::ldexp(1.0, std::min(pc.pbits, 62)) : 1e18);
        else if (c == C_FLOAT) d += 1e18;
        else if (c == C_STRING) d += (double)std::max<i64>(1, t.cols[pc.dict_col].stats.ndict);
        else d += 1;
    }
    return d;
}

// ---- planner: every layout decision of a chain and every N1GPU_* knob of the generator; writes no CUDA text ----------

// N1GPU_* tuning and test knobs, read when a query is compiled: a flag is on when its value starts with '1'; a number
// is the value's atoi, `fallback` when the variable is not set (each call site checks the range it accepts)
bool env_flag(const char* name) { const char* v = getenv(name); return v && *v == '1'; }
int env_int(const char* name, int fallback) { const char* v = getenv(name); return v ? atoi(v) : fallback; }

// Group key packing and the accumulator words.  Returns the sharing key of every word (see add_word).
std::map<std::string, int> plan_words(KernelPlan& kp, const Table& t, const std::vector<ExprP>& keys, const std::vector<ExprP>& aggs,
                                      const std::vector<std::string>& agg_texts, double total_rows_bound) {
    const bool offset_pack = !env_flag("N1GPU_NO_OFFSET_PACK"), sign_from_minmax = !env_flag("N1GPU_NO_SIGN_FROM_MINMAX");
    const bool fcarry = !env_flag("N1GPU_NO_FCARRY");
    for (auto& k : keys) {
        kp.keys.push_back(make_comp(t, *k, "GROUP BY", offset_pack));
        kp.key_bits += kp.keys.back().bits();
    }
    // Accumulator words are shared between aggregates wherever they would hold the same value: SUM(x), AVG(x),
    // COUNT(x), COUNTN(x) over the same operand text use one sum word / one count word, and a count that provably
    // equals the number of selected rows (operand never MISSING/NULL/non-number) is the rows word itself.
    std::map<std::string, int> shared;
    auto add_word = [&](int op, const std::string& key, bool counter = false, i64 lo = 1, i64 hi = 0) {
        auto it = shared.find(key);
        if (it != shared.end()) return it->second;
        // checked here, before any index is stored: FinalAgg keeps word indices in a signed char
        if (kp.word_ops.size() == 64) N1_THROW(N1GPU_E_INELIGIBLE, "more than 64 accumulator words per group");
        kp.word_ops.push_back(op);
        kp.word_count.push_back(counter);
        kp.word_lo.push_back(lo);
        kp.word_hi.push_back(hi);
        shared[key] = (int)kp.word_ops.size() - 1;
        return (int)kp.word_ops.size() - 1;
    };
    const u32 M_ABSENT = bit(C_MISSING) | bit(C_NULL);
    std::map<std::string, int> dset_of;  // DISTINCT operand text -> entry-set id
    int ndistinct_aggs = 0;
    std::map<std::string, std::pair<int, int>> flag_of;  // float-carried operand text -> (OR word, first of its three bits)
    int flag_word = -1, flag_next = 0;
    if (!keys.empty()) kp.w_rows = add_word(OP_ADD_U64, "rows", true);  // word 0: rows per group (group existence)
    auto rows_word = [&]() { if (kp.w_rows < 0) kp.w_rows = add_word(OP_ADD_U64, "rows", true); return kp.w_rows; };

    // does the chain also compute plain MIN and MAX of this (INT-or-absent) operand?  Then a SUM over it reads the sign mix
    // of its ints off them (value/integer.go:266-277 only asks whether both signs occurred)
    auto int_minmax_of = [&](const std::string& ot) {
        if (!sign_from_minmax) return false;
        bool mn = false, mx = false;
        for (auto& x : aggs) {
            if (x->kind != EK::AGG || x->distinct || x->star || x->ops.empty() || x->ops[0]->str() != ot) continue;
            if ((x->ops[0]->ti.mask & ~(bit(C_INT) | bit(C_MISSING) | bit(C_NULL))) != 0) continue;
            mn = mn || x->agg == AggKind::MIN;
            mx = mx || x->agg == AggKind::MAX;
        }
        return mn && mx;
    };
    for (size_t a = 0; a < aggs.size(); ++a) {
        const Expr& e = *aggs[a];
        if (e.kind != EK::AGG) N1_THROW(N1GPU_E_INELIGIBLE, "%s is not an aggregate", agg_texts[a].c_str());
        AggPlan ap;
        ap.kind = e.agg; ap.distinct = e.distinct; ap.star = e.star; ap.text = agg_texts[a];
        const Expr* opnd = e.star ? nullptr : e.ops[0].get();
        if (opnd && opnd->kind == EK::AGG) N1_THROW(N1GPU_E_INELIGIBLE, "nested aggregate");
        ap.opmask = opnd ? opnd->ti.mask : 0;
        if (opnd && (ap.opmask & bit(C_STRING)) && opnd->ti.plain_col) ap.dict_col = opnd->ti.dict_col;
        if (ap.distinct) {
            // result words, filled at finalisation by k_distinct_finalize from the set entries (never during the scan)
            // DISTINCT aggregates over the same operand share one entry set: COUNT(DISTINCT x) and SUM(DISTINCT x)
            // insert x once; the set holds every non-NULL value when one of them is a COUNT, numbers only otherwise
            const std::string ot = opnd->str();
            if (!dset_of.count(ot)) { dset_of[ot] = kp.ndistinct++; kp.set_any.push_back(false); }
            ap.distinct_id = dset_of[ot];
            if (ap.kind == AggKind::COUNT) kp.set_any[ap.distinct_id] = true;
            if (++ndistinct_aggs > 16) N1_THROW(N1GPU_E_INELIGIBLE, "more than 16 DISTINCT aggregates");
            ap.dcomp = make_comp(t, *opnd, "DISTINCT", offset_pack);
            const std::string dk = strf("d%d:", ndistinct_aggs);
            ap.w_cnt = add_word(OP_ADD_U64, dk + "cnt", true);
            if (ap.kind == AggKind::SUM || ap.kind == AggKind::AVG) {
                if (ap.dcomp.mask & bit(C_INT)) {
                    ap.w_ilo = add_word(OP_ADD_U64, dk + "ilo");
                    ap.w_ihi = add_word(OP_ADD_U64, dk + "ihi");
                    ap.w_neg = add_word(OP_ADD_U64, dk + "neg");
                }
                if (ap.dcomp.mask & bit(C_FLOAT)) { ap.w_fsum = add_word(OP_ADD_F64, dk + "fsum"); ap.w_nflt = add_word(OP_ADD_U64, dk + "nflt"); }
            }
        } else if (ap.kind == AggKind::COUNT || ap.kind == AggKind::COUNTN) {
            const std::string ot = opnd ? opnd->str() : std::string("*");
            const u32 counted = ap.kind == AggKind::COUNT ? ~(bit(C_MISSING) | bit(C_NULL)) : M_NUM;
            if (ap.star || (ap.opmask & ~counted) == 0) ap.w_cnt = rows_word();  // every selected row counts
            else ap.w_cnt = add_word(OP_ADD_U64, (ap.kind == AggKind::COUNT ? "cnt:" : "cntn:") + ot, true);
        } else if ((ap.kind == AggKind::SUM || ap.kind == AggKind::AVG) && (ap.opmask & bit(C_INT)) && (ap.opmask & bit(C_FLOAT)) &&
                   opnd->ti.imax * std::max(1.0, total_rows_bound) < 9.0e15 && fcarry) {
            // INT and FLOAT values mixed, ints provably small: one float64 word carries both (see AggPlan::fcarry)
            const std::string ot = opnd->str();
            ap.fcarry = true;
            ap.w_fsum = add_word(OP_ADD_F64, "fsum:" + ot);
            ap.w_nnum = (ap.opmask & ~M_NUM) == 0 ? rows_word() : add_word(OP_ADD_U64, "cntn:" + ot, true);
            if (!flag_of.count(ot)) {
                if (flag_word < 0 || flag_next + 3 > 30) { flag_word = add_word(OP_OR_U64, strf("flags:%d", (int)flag_of.size())); flag_next = 0; }
                flag_of[ot] = {flag_word, flag_next};
                flag_next += 3;
            }
            ap.w_flags = flag_of[ot].first;
            ap.flag_shift = flag_of[ot].second;
        } else if (ap.kind == AggKind::SUM || ap.kind == AggKind::AVG) {
            const std::string ot = opnd->str();
            if (ap.opmask & bit(C_INT)) {
                const TypeInfo& ti = opnd->ti;
                bool exact1 = false;
                if (ti.ranged) {
                    double mx = std::max(std::fabs((double)ti.lo), std::fabs((double)ti.hi));
                    exact1 = mx * std::max(1.0, total_rows_bound) < 2.3e18;  // < 2^61: no int64 overflow possible
                }
                if (exact1) ap.w_isum = add_word(OP_ADD_U64, "isum:" + ot, false, ti.lo, ti.hi);
                else { ap.w_ilo = add_word(OP_ADD_U64, "ilo:" + ot); ap.w_ihi = add_word(OP_ADD_U64, "ihi:" + ot); }
                // how many ints were summed, and how many of them were negative; the int counter is whichever existing
                // counter provably counts the same rows (every selected row / rows > NULL / numbers), else its own word
                bool can_neg = !ti.ranged || ti.lo < 0, can_nonneg = !ti.ranged || ti.hi >= 0;
                if (ap.opmask == bit(C_INT)) ap.w_nint = rows_word();
                else if ((ap.opmask & ~(M_ABSENT | bit(C_INT))) == 0) ap.w_nint = add_word(OP_ADD_U64, "cnt:" + ot, true);
                else if ((ap.opmask & bit(C_FLOAT)) == 0) ap.w_nint = add_word(OP_ADD_U64, "cntn:" + ot, true);
                else ap.w_nint = add_word(OP_ADD_U64, "nint:" + ot, true);
                if (can_neg && can_nonneg && int_minmax_of(ot)) ap.w_sgn_min = -2;  // resolved below: MIN / MAX of this operand exist
                else if (can_neg) ap.w_neg = can_nonneg ? add_word(OP_ADD_U64, "nneg:" + ot, true) : ap.w_nint;
            }
            if (ap.opmask & bit(C_FLOAT)) {
                ap.w_fsum = add_word(OP_ADD_F64, "fsum:" + ot);
                ap.w_nflt = ap.opmask == bit(C_FLOAT) ? rows_word() : add_word(OP_ADD_U64, "nflt:" + ot, true);
            }
        } else {  // MIN / MAX
            bool mn = ap.kind == AggKind::MIN;
            const std::string ot = (mn ? "min:" : "max:") + opnd->str();
            u32 m = ap.opmask;
            if (m & bit(C_STRING)) { if (ap.dict_col < 0) N1_THROW(N1GPU_E_INELIGIBLE, "MIN/MAX over a constant or computed string"); }
            if (opnd && !opnd->ti.plain_col && (m & bit(C_FLOAT))) m |= bit(C_INT);  // canon_num
            ap.opmask = m;
            // which classes were seen: MIN and MAX of one operand share the word; an operand with a single class above
            // NULL needs no class bits at all, only "was there any" = a counter other aggregates usually keep anyway
            const u32 above = m & ~M_ABSENT;
            if (above && (above & (above - 1)) == 0) {
                for (int c = 0; c < 8; ++c) if (above == bit(c)) ap.seen_class = c;
                ap.w_seen_cnt = (m & M_ABSENT) == 0 ? rows_word() : add_word(OP_ADD_U64, "cnt:" + opnd->str(), true);
            } else ap.w_seen = add_word(OP_OR_U64, "seen:" + opnd->str());
            const TypeInfo& ti = opnd->ti;
            const bool r = ti.ranged;
            if (m & bit(C_INT)) ap.w_mi = add_word(mn ? OP_MIN_I64 : OP_MAX_I64, "i:" + ot, false, r ? ti.lo : 1, r ? ti.hi : 0);
            if (m & bit(C_FLOAT)) ap.w_mf = add_word(mn ? OP_MIN_U64 : OP_MAX_U64, "f:" + ot);
            if (m & bit(C_STRING)) ap.w_ms = add_word(mn ? OP_MIN_U64 : OP_MAX_U64, "s:" + ot, false, 0,
                                                    std::max<i64>(t.cols[ap.dict_col].stats.ndict, (i64)t.cols[ap.dict_col].dict.size()));
        }
        kp.aggs.push_back(ap);
    }
    if (kp.word_ops.empty()) rows_word();  // keep at least one word (only DISTINCT aggregates)
    for (auto& ap : kp.aggs) {
        if (ap.w_sgn_min != -2) continue;
        ap.w_sgn_min = ap.w_sgn_max = -1;
        const std::string ot = aggs[(size_t)(&ap - &kp.aggs[0])]->ops[0]->str();
        for (size_t b = 0; b < kp.aggs.size(); ++b) {
            const AggPlan& o = kp.aggs[b];
            if (o.distinct || o.star || aggs[b]->ops.empty() || aggs[b]->ops[0]->str() != ot || o.w_mi < 0) continue;
            if (o.kind == AggKind::MIN) ap.w_sgn_min = o.w_mi;
            if (o.kind == AggKind::MAX) ap.w_sgn_max = o.w_mi;
        }
        if (ap.w_sgn_min < 0 || ap.w_sgn_max < 0) N1_THROW(N1GPU_E_INVALID, "internal: MIN / MAX words of %s not found", ot.c_str());
    }
    return shared;
}

// The table mode: shared-memory dense (thread-private block shape), direct-indexed or hashed HBM with the front cache's
// cells, pairs, key width, block and slots, or the 128-bit hash table.
void plan_mode(KernelPlan& kp, const Table& t, i64 layout_rows) {
    const int W = (int)kp.word_ops.size();
    const int min_blocks = env_int("N1GPU_MIN_BLOCKS", 0);  // resident blocks per SM (0: compiler's choice / the cache's)
    double est = 1;
    for (auto& pc : kp.keys) est *= comp_domain(t, pc);
    int cache_blocks = 0;  // resident blocks per SM the front cache is sized for
    if (kp.keys.empty()) kp.mode = MODE_UNGROUPED;
    else if (kp.key_bits <= 13 && ((i64)1 << kp.key_bits) * W * 8 <= 40 * 1024) {
        kp.mode = MODE_DENSE;
        kp.dense_slots = (i64)1 << kp.key_bits;
        {   // slots numbered by the mixed-radix value of the components when that is tighter than the bit-packed key
            u64 tight = 1;
            std::vector<u64> dom;
            for (auto& pc : kp.keys) { const u64 d = comp_values(t, pc); dom.push_back(d); tight = d ? tight * d : 0; }
            if (tight > 0 && (i64)tight < kp.dense_slots && kp.ndistinct == 0 && !env_flag("N1GPU_NO_TIGHT")) { kp.dense_dom = dom; kp.dense_slots = (i64)tight; }
        }
        // A handful of groups (TPC-H Q1: 6) would serialise every row on the same few shared-memory words.  When the
        // whole table is <= 48 words, every thread keeps its own copy in shared memory (bank = thread: conflict-free
        // plain read-modify-write, no atomics) and the copies are folded once per block.
        if (kp.dense_slots * W <= 48 && !env_flag("N1GPU_NO_PRIV")) {
            kp.dense_priv = true;
            // Block shape: cells x 8 bytes per thread decide how many threads an SM holds (config 3: 42 cells = 336 bytes ->
            // 2 blocks x 256 threads = 16 warps, a quarter of the SM: ncu shows the scan latency-bound, issue 53 %, DRAM 48 %).
            // When fewer than four 256-thread blocks fit, the block size that packs the most warps into 227 KiB is taken
            // instead (config 3: 1 x 640 threads = 20 warps; 718 -> 645 us per 60 M rows).  The private cells stay conflict-free
            // for any multiple of 32.
            const i64 cells = kp.dense_slots * W;
            const int pb = env_int("N1GPU_PRIV_BLOCK", 0);
            auto blocks_of = [&](int block) {  // private cells + the per-warp fold buffer + the reserved KiB of every block
                return (int)std::min<i64>((i64)(227 * 1024) / (cells * 8 * block + cells * 8 * (block / 32) + 1536), 2048 / block);
            };
            int best_block = 256;
            if (pb >= 32 && pb <= 1024 && pb % 32 == 0) best_block = pb;
            else if (blocks_of(256) < 4) {
                int best_warps = blocks_of(256) * 8;
                for (int block = 128; block <= 1024; block += 32) {
                    const int warps = blocks_of(block) * (block / 32);
                    if (warps >= best_warps && warps > 0) { best_warps = warps; best_block = block; }  // ties: the larger block (fewer folds; measured 645 vs 665 us)
                }
            }
            kp.block = best_block;
            kp.dyn_smem = (int)(cells * kp.block * 8);
        }
    }
    else if (kp.key_bits <= 63) {
        // A packed key of few bits indexes the HBM table directly: no key array, no hash probe, no insert race, the
        // table (config 5: 2^19 slots x 6 words = 25 MB) stays in L2, and because slot == key on every rank the
        // multi-GPU merge is element-wise (all_gather + k_merge_words, stream-ordered) instead of a record exchange.
        const double slots = kp.key_bits <= 22 ? (double)((i64)1 << kp.key_bits) : 1e30;
        // (every partition must take the same decision - their states are merged slot by slot - so it is based on the rows
        // of the whole keyspace when they are declared, never on this partition's own share)
        if (!env_flag("N1GPU_NO_DIRECT") && slots * W * 8 <= 256.0 * 1024 * 1024 && slots <= 8.0 * std::max<double>((double)layout_rows, 131072.0)) {
            kp.mode = MODE_DENSE;
            kp.dense_global = true;
            kp.dense_slots = (i64)1 << kp.key_bits;
        } else kp.mode = MODE_HASH64;
        // shared-memory front cache for hot keys (Zipf-skewed GROUP BY)
        if (!env_flag("N1GPU_NO_CACHE")) {
            // cell layout (see n1ql_device.cuh "Cells of the front cache")
            const bool wide1 = kp.dense_global && !env_flag("N1GPU_NO_WIDE1");
            for (int w = 0; w < W; ++w) {
                const int op = kp.word_ops[w];
                int kind = CK_64;
                // an integer sum whose addends are within +-2^31: ONE 32-bit cell, the (rare) carries go straight to the table word
                const bool small_addends = kp.word_lo[w] <= kp.word_hi[w] && kp.word_lo[w] > -((i64)1 << 31) && kp.word_hi[w] < ((i64)1 << 31);
                if (op == OP_ADD_U64) kind = kp.word_count[w] ? CK_CNT : ((small_addends && wide1) ? CK_WIDE1 : CK_WIDE);
                else if (op == OP_OR_U64) kind = CK_OR32;
                else if (op != OP_ADD_F64 && kp.word_lo[w] <= kp.word_hi[w] && (u64)kp.word_hi[w] - (u64)kp.word_lo[w] <= 0xfffffffcULL) kind = CK_MM32;
                kp.cell_kind.push_back(kind);
                if (kind == CK_64) kp.cell_idx.push_back(kp.cache_n64++);
                else { kp.cell_idx.push_back(kp.cache_n32); kp.cache_n32 += kind == CK_WIDE ? 2 : 1; }
            }
            kp.cell_pair.assign((size_t)W, 0);
            if (!env_flag("N1GPU_NO_MM_PAIR"))
                for (int w = 0; w + 1 < W; ++w)
                    if (kp.cell_kind[w] == CK_MM32 && kp.cell_kind[w + 1] == CK_MM32 && kp.cell_idx[w + 1] == kp.cell_idx[w] + 1 && kp.cell_pair[w] == 0) {
                        kp.cell_pair[w] = 1; kp.cell_pair[w + 1] = 2; ++w;
                    }
            // u32 keys, direct-mapped (cache_claim_1).  Buckets of four keys were removed: 5.19 against 4.95 ms per 1 B
            // config-5 rows (profiles/r02_config5_ablation.jsonl)
            kp.cache_key32 = kp.key_bits <= 31 && !env_flag("N1GPU_NO_KEY32");
            const int slot_bytes = (kp.cache_key32 ? 4 : 8) + 8 * kp.cache_n64 + 4 * kp.cache_n32;
            // The five 256-thread blocks of an SM each cache the same hot keys in their own 44 KiB; one 1024-thread block
            // caches five times as many distinct keys in the SM's 220 KiB.  Measured on config 5 (Zipf over 100 k keys,
            // tools/sweep_config5.py, 200 M rows): 5 x 256 1 242 us, 2 x 512 1 201 us, 1 x 1024 1 161 us - every miss is
            // 3-4 scattered L2 reductions, one LSU wavefront each, and LSU wavefronts are what the kernel runs out of.
            // So: the small block when its cache holds every group anyway or the key domain is far beyond any cache
            // (uniform high-cardinality keys: occupancy matters more), the large block in between.
            const int kb = env_int("N1GPU_CACHE_KB", 0);     // shared memory per block spent on the cache
            const int bt = env_int("N1GPU_CACHE_BLOCK", 0);  // threads per block
            const double slots_small = 44.0 * 1024 / slot_bytes, slots_large = 220.0 * 1024 / slot_bytes;
            kp.block = bt >= 64 ? bt / 32 * 32 : (est > 0.8 * slots_small && est <= 64.0 * slots_large ? 1024 : 256);
            cache_blocks = min_blocks > 0 ? min_blocks : std::max(1, 1280 / kp.block);
            // the resident blocks of an SM share 220 of its 227 KiB (each block also pays 1 KiB of system shared memory)
            const i64 budget = (kb > 0 ? kb : 220 / cache_blocks) * 1024;
            i64 cs = budget / slot_bytes / 64 * 64;
            const i64 need = (i64)std::min(4.0 * std::max(est, 1.0), 1e9);  // never more than the groups need
            if (cs > need) cs = std::max<i64>(64, (need + 63) / 64 * 64);
            kp.cache_slots = (int)cs;
            kp.dyn_smem = (int)cs * slot_bytes;
        }
    }
    else if (kp.key_bits <= 127) kp.mode = MODE_HASH128;
    else if (kp.keys.size() <= 16) {
        // Two mixed INT / FLOAT columns already pack into 130 bits.  No front cache: its cells are keyed by one word, and
        // without it there are neither packed nor complemented counters.  A DISTINCT entry would embed the whole key:
        // plan_distinct refuses it (entry > 127 bits).
        kp.mode = MODE_HASHW;
        kp.key_words = (kp.key_bits + 63) / 64;
    }
    else N1_THROW(N1GPU_E_INELIGIBLE, "group key of %zu components needs %d bits (> 127) after packing", kp.keys.size(), kp.key_bits);
    kp.est_groups = (i64)std::min(est, 4e18);
    kp.min_blocks = min_blocks != 0 ? min_blocks : (kp.cache_slots > 0 ? cache_blocks : 0);
}

// Complemented counters.  Behind the front cache every accumulator update of a cached row is a shared-memory atomic, the
// unit the kernel runs out of first.  "cnt:x" (rows where x > NULL) over a plain column counts the other rows when the
// column statistics say those are the minority.  Every partition must decide alike, so the decision only uses agreed
// numbers: the declared keyspace rows with exchanged statistics, this table's own rows otherwise.
void plan_complement(KernelPlan& kp, const Table& t, const std::vector<ExprP>& aggs, const std::map<std::string, int>& word_of) {
    kp.word_complement.assign(kp.word_ops.size(), false);
    kp.complement_agg.assign(kp.word_ops.size(), -1);
    if (kp.cache_slots == 0 || kp.w_rows != 0 || env_flag("N1GPU_NO_COMPLEMENT")) return;
    bool forced = false;
    for (auto& c : t.cols) forced = forced || c.stats_forced;
    const i64 denom = t.global_rows > 0 ? std::max(t.global_rows, t.nrows) : (forced ? 0 : t.nrows);
    for (size_t a = 0; a < aggs.size() && denom > 0; ++a) {
        const Expr& e = *aggs[a];
        if (e.star || e.distinct || e.ops.empty()) continue;
        const Expr* opnd = e.ops[0].get();
        if (opnd->kind != EK::FIELD || opnd->col < 0) continue;
        auto it = word_of.find("cnt:" + opnd->str());
        if (it == word_of.end() || it->second == kp.w_rows) continue;
        if (t.cols[opnd->col].stats.absent_rows * 2 < denom) { kp.word_complement[it->second] = true; kp.complement_agg[it->second] = (int)a; }
    }
}

// Physical words.  Behind the front cache a miss pays one L2 reduction per word it touches, and the request path SM -> L2
// is what bounds a skewed GROUP BY (profiles/r01_atomic_probe.txt: 190 G scattered RED/s whatever their width).  Row
// counters are therefore packed two per 64-bit word (32-bit fields) when no counter can reach 2^32 over all ranks.
void plan_physical(KernelPlan& kp, double total_rows_bound) {
    const int W = (int)kp.word_ops.size();
    const bool pack = kp.cache_slots > 0 && kp.ndistinct == 0 && !env_flag("N1GPU_NO_PACK") && total_rows_bound < 4294967295.0;
    kp.phys_of.assign(W, -1); kp.shift_of.assign(W, 0); kp.bits_of.assign(W, 64);
    int pending = -1;  // counter waiting for a partner
    for (int w = 0; w < W; ++w) {
        if (pack && kp.word_count[w] && kp.word_ops[w] == OP_ADD_U64) {
            if (pending >= 0) {
                kp.phys_of[w] = kp.phys_of[pending]; kp.shift_of[w] = 32; kp.bits_of[w] = 32; kp.bits_of[pending] = 32;
                pending = -1;
                continue;
            }
            pending = w;
        }
        kp.phys_of[w] = (int)kp.phys_ops.size();
        kp.phys_ops.push_back(kp.word_ops[w]);
    }
}

// DISTINCT entry layout: (set, group key, value) bits, hash set or bitmap, and the bitmap's passes
void plan_distinct(KernelPlan& kp, i64 layout_rows) {
    if (!kp.ndistinct) return;
    kp.abits = bits_for((u64)kp.ndistinct);
    int mx = 0;
    for (auto& ap : kp.aggs) if (ap.distinct) mx = std::max(mx, ap.dcomp.bits());
    kp.entry_bits = kp.abits + kp.key_bits + mx;
    if (kp.entry_bits > 127) N1_THROW(N1GPU_E_INELIGIBLE, "DISTINCT entry needs %d bits (> 127)", kp.entry_bits);
    kp.set128 = kp.entry_bits > 63;
    // An entry of few bits indexes a bitmap directly: one fire-and-forget atomicOr per row instead of a hash probe
    // with a dependent compare-and-swap, and 2^bits / 8 bytes instead of 16 bytes per row - config 4's 2^30
    // entries are 128 MiB, about the size of the L2, where the hash set is 4 GiB of random DRAM sectors.
    // Chosen when the bitmap is no larger than the hash set would be.
    const double bitmap_bytes = kp.entry_bits <= 36 ? (double)((u64)1 << kp.entry_bits) / 8.0 : 1e30;
    kp.set_bitmap = !env_flag("N1GPU_NO_BITMAP") && bitmap_bytes <= std::max(65536.0, 16.0 * (double)std::max<i64>(layout_rows, 1) * kp.ndistinct);
    // A bitmap the size of the L2 (config 4: 128 MiB) turns every row into a random DRAM sector read-modify-write.
    // The scan then runs in passes over slices of the entry range small enough to stay L2-resident: the columns
    // are streamed once per pass (cheap next to random DRAM), the bits land in L2.
    if (!kp.set_bitmap) return;
    const int sp = env_int("N1GPU_SET_PASSES", 0);
    int passes = 1;
    if (sp >= 1) passes = sp;
    // measured (config 4, 200 M rows, 128 MiB bitmap; profiles/r01_config4_bitmap_passes.jsonl): 1 pass 5.58 ms,
    // 2 passes 3.23 ms, 4 passes 3.45 ms, 8 passes 5.41 ms - a pass costs ~0.65 ms of streaming and key work, so
    // the slices are made just small enough (<= 64 MiB) for most of their sectors to stay in the 126 MB L2
    else if (bitmap_bytes > 96.0 * 1024 * 1024) while (passes < 8 && bitmap_bytes / passes > 64.0 * 1024 * 1024) passes *= 2;
    while (passes & (passes - 1)) passes &= passes - 1;                          // a power of two ...
    while (passes > 1 && bits_for((u64)passes) > kp.entry_bits - 6) passes /= 2;  // ... of slices of >= 64 bits
    // only where the kernel has no epilogue that publishes and re-arms state (the HBM table modes)
    const bool hbm_table = kp.mode == MODE_HASH64 || kp.mode == MODE_HASH128 || (kp.mode == MODE_DENSE && kp.dense_global);
    kp.set_passes = hbm_table ? passes : 1;
}

// Partitioned DISTINCT aggregation (see KernelPlan::part): eligibility and the record layout
void plan_partition(KernelPlan& kp, i64 layout_rows) {
    const bool force = env_flag("N1GPU_PART");  // also for keyspaces too small to profit (tests)
    if (env_flag("N1GPU_NO_PART") || !(kp.mode == MODE_DENSE && kp.dense_global && kp.ndistinct == 1 && kp.cache_slots > 0 && kp.w_rows == 0)) return;
    const AggPlan* da = nullptr;
    for (auto& ap : kp.aggs) {
        if (ap.distinct) { if (!da) da = &ap; continue; }
        // every other aggregate must be the group's row count
        if (!((ap.kind == AggKind::COUNT || ap.kind == AggKind::COUNTN) && ap.w_cnt == kp.w_rows)) return;
    }
    // the value component must be one class with a small payload: a ranged INT (sums from popcounts) or a STRING rank
    if (!(da->dcomp.classes.size() == 1 && da->dcomp.cbits == 0 && da->dcomp.nfree < 0 &&
          ((da->dcomp.classes[0] == C_INT && da->dcomp.biased) || (da->dcomp.classes[0] == C_STRING && da->w_ilo < 0)))) return;
    for (auto& ap : kp.aggs) if (ap.distinct && (ap.w_fsum >= 0 || ap.w_nflt >= 0)) return;
    const int KB = kp.key_bits, VB = da->dcomp.bits();
    const int PB = std::max(1, std::max(KB + VB - 20, KB - 12));  // a partition's bitmap <= 2^20 bits, <= 4096 groups
    if (!(VB >= 1 && VB <= 12 && PB <= 10 && PB < KB && (KB - PB) + 1 + VB <= 32 && (force || layout_rows >= ((i64)1 << (PB + 12))))) return;
    kp.part = true;
    kp.part_bits = PB; kp.part_gbits = KB - PB; kp.part_vbits = VB;
    kp.part_bincap = std::max(8, std::min(48, 192 * 1024 / (4 << PB)));
    kp.part_smem = (4 << PB) * (1 + kp.part_bincap);
}

KernelPlan plan_layout(const Table& t, const std::vector<ExprP>& keys, const std::vector<ExprP>& aggs,
                       const std::vector<std::string>& agg_texts, double total_rows_bound) {
    KernelPlan kp;
    // rows that layout decisions shared by all partitions are based on: the declared keyspace rows, else this table's
    const i64 layout_rows = t.global_rows > 0 ? std::max(t.global_rows, t.nrows) : t.nrows;
    const std::map<std::string, int> word_of = plan_words(kp, t, keys, aggs, agg_texts, total_rows_bound);
    plan_mode(kp, t, layout_rows);
    plan_complement(kp, t, aggs, word_of);
    plan_physical(kp, total_rows_bound);
    plan_distinct(kp, layout_rows);
    plan_partition(kp, layout_rows);
    // An ungrouped scan consumes nothing that a stream-preceding kernel produces (its table was sealed with a device
    // synchronisation, its state belongs to this query handle alone), so the next kernel of the stream may be scheduled
    // as soon as SMs free up: programmatic dependent launch.
    kp.pdl = kp.mode == MODE_UNGROUPED;
    return kp;
}

// ---- emitters: the CUDA text of a planned chain; they make no decision -----------------------------------------------

// Row code through Gen, in the order Gen numbers constant slots, IN sets, temporaries and column values: WHERE, keys,
// aggregates, the partition kernel's value operand.
struct RowCode {
    std::string filter;      // sets w_true (empty without WHERE)
    std::string key;         // the cached modes: packs the group key into klo (the other modes: part of `agg`)
    std::string agg;         // executed under `if (pass)`
    std::string part_value;  // the partition kernel: hasv and the packed DISTINCT value vlo
};

// the value of computed FLOAT operand `e` with integral floats as INT (canon_num), as packed or compared
std::string canon(Gen& g, const Expr& e, const std::string& v, const char* prefix) {
    if (e.ti.plain_col || !(e.ti.mask & bit(C_FLOAT))) return v;
    const std::string cv = g.nv(prefix);
    g.line(strf("const Val %s = canon_num(%s);", cv.c_str(), v.c_str()));
    return cv;
}

// does `v` go into DISTINCT entry set `set`: every value above NULL, or numbers only
std::string has_value(const KernelPlan& kp, int set, const std::string& v) {
    return kp.set_any[(size_t)set] ? strf("%s.c > C_NULL", v.c_str()) : strf("is_num(%s.c)", v.c_str());
}

RowCode emit_row_code(Gen& g, const KernelPlan& kp, const Expr* where, const std::vector<ExprP>& keys, const std::vector<ExprP>& aggs) {
    RowCode rc;
    if (where) {
        std::string wv = g.emit(*where, nullptr);
        g.line(strf("const bool w_true = v_truth(%s, %lldLL);", wv.c_str(), (long long)g.empty2_of(*where)));
    }
    rc.filter = g.body;
    g.body.clear();
    const bool cached = kp.cache_slots > 0;
    g.ind = "                    ";
    if (kp.mode == MODE_HASHW) {
        // the key words stay in registers: every pack_bits index is a constant once the row code is unrolled
        g.line(strf("u64 kwd[%d] = {}; int kpos = 0;", kp.key_words));
        for (size_t k = 0; k < keys.size(); ++k) emit_pack(g, kp.keys[k], canon(g, *keys[k], g.emit(*keys[k], nullptr), "k"), "kwd", nullptr, "kpos");
        g.line(strf("const i64 slot = table_insert_wide<%d>(p.keys, p.cap_mask, kwd);", kp.key_words));
        g.line("if (slot < 0) { if (slot == -1) p.status[0] = 1; else p.status[1] = NQ_WIDE_STUCK; continue; }");
    } else if (kp.mode != MODE_UNGROUPED) {
        g.line("u64 klo = 0, khi = 0; int kpos = 0;");
        const bool radix = !kp.dense_dom.empty();
        if (radix) g.line("u64 kslot = 0;");
        u64 radix_stride = 1;
        for (size_t k = 0; k < keys.size(); ++k) {
            const std::string kv = canon(g, *keys[k], g.emit(*keys[k], nullptr), "k");
            emit_pack(g, kp.keys[k], kv, "klo", "khi", "kpos", radix ? "kslot" : nullptr, radix_stride);
            if (radix) radix_stride *= kp.dense_dom[k];
        }
        if (kp.mode == MODE_DENSE && !cached) g.line(radix ? "const i64 slot = (i64)kslot;" : "const i64 slot = (i64)klo;");
        else if (cached) {
            // the kernel is assembled in phases (keys + cache probe / cached updates / table updates, see cached_rows):
            // the key code ends here, the update code starts from an empty body
            rc.key = g.body;
            g.body.clear();
        }
        else if (kp.mode == MODE_HASH64) g.line("const i64 slot = table_insert64(p.keys, p.cap_mask, klo, nullptr);");
        else g.line("const i64 slot = table_insert128((ulonglong2*)p.keys, p.cap_mask, klo, khi, nullptr);");
        if (kp.mode != MODE_DENSE && !cached) g.line("if (slot < 0) { p.status[0] = 1; continue; }");
    }
    std::set<int> emitted_sets;
    std::set<int> emitted;  // a shared word is updated once per row, by the first aggregate that owns it
    if (kp.w_rows >= 0) { g.line(strf("ACC(%d, OP_ADD_U64, 1);  // rows", kp.w_rows)); emitted.insert(kp.w_rows); }
    for (int w = 0; w < (int)kp.word_ops.size(); ++w) {
        if (!kp.word_complement[w]) continue;
        const Expr& opnd = *aggs[(size_t)kp.complement_agg[w]]->ops[0];
        const std::string o = g.emit(opnd, nullptr);
        g.line(strf("ACCIF(%d, OP_ADD_U64, 1, %s.c <= C_NULL);  // rows NOT counted by count(%s)", w, o.c_str(), opnd.str().c_str()));
        emitted.insert(w);
    }
    for (size_t a = 0; a < kp.aggs.size(); ++a) {
        const AggPlan& ap = kp.aggs[a];
        const Expr& e = *aggs[a];
        g.open(strf("{ // %s", ap.text.c_str()));
        std::string o;
        if (!ap.star) o = g.emit(*e.ops[0], nullptr);
        auto ACC = [&](int w, int op, const std::string& x) {
            if (!emitted.insert(w).second) return;  // another aggregate over the same operand already feeds this word
            g.line(strf("ACC(%d, %s, %s);", w, op_name(op), x.c_str()));
        };
        auto ACCIF = [&](const std::string& cond, int w, int op, const std::string& x) {
            if (!emitted.insert(w).second) return;
            g.line(strf("ACCIF(%d, %s, %s, %s);", w, op_name(op), x.c_str(), cond.c_str()));
        };
        if (ap.distinct && !emitted_sets.insert(ap.distinct_id).second) {
            // the entry set of this operand is already fed by an earlier aggregate
        } else if (ap.distinct) {
            g.open(strf("if (%s) {", has_value(kp, ap.distinct_id, o).c_str()));
            const std::string cv = canon(g, *e.ops[0], o, "d");
            g.line("u64 elo = 0, ehi = 0; int epos = 0;");
            if (kp.abits) g.line(strf("pack_bits(elo, ehi, epos, %dULL, %d);", ap.distinct_id, kp.abits));
            if (kp.key_bits) {
                g.line(strf("pack_bits(elo, ehi, epos, klo, %d);", std::min(64, kp.key_bits)));
                if (kp.key_bits > 64) g.line(strf("pack_bits(elo, ehi, epos, khi, %d);", kp.key_bits - 64));
            }
            emit_pack(g, ap.dcomp, cv, "elo", "ehi", "epos");
            if (kp.set_bitmap && kp.set_passes > 1)
                g.line("if ((int)(elo >> p.set_shift) == p.set_pass) atomicOr(&((u32*)p.set_keys)[elo >> 5], 1u << (elo & 31));  // DISTINCT bitmap, this pass's slice");
            else if (kp.set_bitmap) g.line("atomicOr(&((u32*)p.set_keys)[elo >> 5], 1u << (elo & 31));  // DISTINCT bitmap");
            else if (kp.set128) g.line("if (table_insert128((ulonglong2*)p.set_keys, p.set_mask, elo, ehi, nullptr) < 0) p.status[0] = 2;");
            else g.line("if (table_insert64(p.set_keys, p.set_mask, elo, nullptr) < 0) p.status[0] = 2;");
            g.close();
        } else if (ap.kind == AggKind::COUNT) {
            if (ap.star) ACC(ap.w_cnt, OP_ADD_U64, "1");
            else ACCIF(strf("%s.c > C_NULL", o.c_str()), ap.w_cnt, OP_ADD_U64, "1");
        } else if (ap.kind == AggKind::COUNTN) {
            ACCIF(strf("is_num(%s.c)", o.c_str()), ap.w_cnt, OP_ADD_U64, "1");
        } else if (ap.fcarry) {
            if (!emitted.count(ap.w_fsum)) {  // SUM(x) and AVG(x) share the words: fed once
                g.open(strf("if (is_num(%s.c)) {", o.c_str()));
                ACC(ap.w_fsum, OP_ADD_F64, strf("(u64)__double_as_longlong(num_f(%s))", o.c_str()));
                g.line(strf("ACC(%d, OP_OR_U64, (%s.c == C_FLOAT ? 1ULL : (%s.b < 0 ? 2ULL : 4ULL)) << %d);", ap.w_flags, o.c_str(), o.c_str(), ap.flag_shift));
                ACC(ap.w_nnum, OP_ADD_U64, "1");
                g.close();
            }
        } else if (ap.kind == AggKind::SUM || ap.kind == AggKind::AVG) {
            if (ap.opmask & bit(C_INT)) {
                g.open(strf("if (%s.c == C_INT) {", o.c_str()));
                if (ap.w_isum >= 0) ACC(ap.w_isum, OP_ADD_U64, strf("(u64)%s.b", o.c_str()));
                else {
                    ACC(ap.w_ilo, OP_ADD_U64, strf("((u64)%s.b & 0xffffffffULL)", o.c_str()));
                    ACC(ap.w_ihi, OP_ADD_U64, strf("(u64)(%s.b >> 32)", o.c_str()));
                }
                ACC(ap.w_nint, OP_ADD_U64, "1");
                if (ap.w_neg >= 0 && ap.w_neg != ap.w_nint) ACCIF(strf("%s.b < 0", o.c_str()), ap.w_neg, OP_ADD_U64, "1");
                g.close();
            }
            if (ap.opmask & bit(C_FLOAT)) {
                g.open(strf("if (%s.c == C_FLOAT) {", o.c_str()));
                ACC(ap.w_fsum, OP_ADD_F64, strf("(u64)%s.b", o.c_str()));
                ACC(ap.w_nflt, OP_ADD_U64, "1");
                g.close();
            }
        } else {  // MIN / MAX
            bool mn = ap.kind == AggKind::MIN;
            const std::string cv = canon(g, *e.ops[0], o, "mm");
            g.open(strf("if (%s.c > C_NULL) {", cv.c_str()));
            if (ap.w_seen >= 0) ACC(ap.w_seen, OP_OR_U64, strf("(1ULL << %s.c)", cv.c_str()));
            else ACC(ap.w_seen_cnt, OP_ADD_U64, "1");
            if (ap.w_mi >= 0) ACCIF(strf("%s.c == C_INT", cv.c_str()), ap.w_mi, mn ? OP_MIN_I64 : OP_MAX_I64, strf("(u64)%s.b", cv.c_str()));
            if (ap.w_mf >= 0) ACCIF(strf("%s.c == C_FLOAT", cv.c_str()), ap.w_mf, mn ? OP_MIN_U64 : OP_MAX_U64, strf("f64_ordered(as_f(%s.b))", cv.c_str()));
            if (ap.w_ms >= 0) ACCIF(strf("%s.c == C_STRING", cv.c_str()), ap.w_ms, mn ? OP_MIN_U64 : OP_MAX_U64, strf("((u64)%s.b >> 1)", cv.c_str()));
            g.close();
        }
        g.close();
    }
    rc.agg = g.body;
    g.body.clear();
    if (kp.part) {
        size_t a = 0;
        while (!kp.aggs[a].distinct) ++a;
        const std::string cv = canon(g, *aggs[a]->ops[0], g.emit(*aggs[a]->ops[0], nullptr), "d");
        g.line(strf("const bool hasv = %s;", has_value(kp, kp.aggs[a].distinct_id, cv).c_str()));
        g.line("u64 vlo = 0, vhi = 0; int vpos = 0;");
        g.open("if (hasv) {");
        emit_pack(g, kp.aggs[a].dcomp, cv, "vlo", "vhi", "vpos");
        g.close();
        rc.part_value = g.body;
    }
    return rc;
}

// the loop over the thread's 4 rows, up to `pass` = in range and selected by WHERE (after the row's column values)
std::string select_row(const RowCode& rc, const std::string& decls, const char* in_range) {
    std::string s = strf("#pragma unroll\n        for (int j = 0; j < 4; ++j) {\n            bool pass = %s;\n", in_range) + decls;
    if (!rc.filter.empty()) s += rc.filter + "                pass = pass && w_true;\n";
    return s;
}

// the HBM table slot of packed key `key` behind the front cache: the key itself (direct-indexed), else its insert
std::string hbm_slot(const KernelPlan& kp, const std::string& ind, const char* key, const char* direct_note) {
    if (kp.dense_global) return ind + strf("const i64 slot = (i64)%s;%s\n", key, direct_note);
    return ind + strf("const i64 slot = table_insert64(p.keys, p.cap_mask, %s, nullptr);\n", key) + ind + "if (slot < 0) { p.status[0] = 1; continue; }\n";
}

// the empty value of a 32-bit MIN / MAX cell (CK_MM32: cells hold value - lo + 1)
const char* mm32_empty(int op) { return op == OP_MIN_I64 || op == OP_MIN_U64 ? "0xffffffffu" : "0u"; }

// index of word w's 32-bit cache cell of slot `slot` inside s_c32 (see KernelPlan::cell_pair)
std::string cell32(const KernelPlan& kp, int w, const char* slot) {
    if (kp.cell_pair[(size_t)w] == 1) return strf("%d * NQ_CS + 2 * (%s)", kp.cell_idx[(size_t)w], slot);
    if (kp.cell_pair[(size_t)w] == 2) return strf("%d * NQ_CS + 2 * (%s) + 1", kp.cell_idx[(size_t)w - 1], slot);
    return strf("%d * NQ_CS + %s", kp.cell_idx[(size_t)w], slot);
}

// #defines, accumulator macros and the signature of nq_scan
std::string scan_prologue(const KernelPlan& kp) {
    const int W = (int)kp.word_ops.size();
    const bool cached = kp.cache_slots > 0, smem_dense = kp.mode == MODE_DENSE && !kp.dense_global;
    std::string s;
    s += "// generated by libn1gpu codegen: one specialised scan kernel for this Filter + Group chain\n";
    s += "#include \"n1ql_device.cuh\"\n";
    s += strf("#define NQ_W %d\n", W);
    s += "#define ACCIF(k, OP, x, c) if (c) { ACC(k, OP, x); }\n";
    if (smem_dense) s += strf("#define NQ_G %lld\n", (long long)kp.dense_slots);
    s += "__constant__ int nq_ops[NQ_W] = {";
    for (int w = 0; w < W; ++w) s += strf("%s%d", w ? ", " : "", kp.word_ops[w]);
    s += "};\n";
    s += "__constant__ int nq_fidx[NQ_W] = {";  // float64-sum words keep per-block partials: their partial row
    for (int w = 0, fi = 0; w < W; ++w) s += strf("%s%d", w ? ", " : "", kp.word_ops[w] == OP_ADD_F64 ? fi++ : -1);
    s += "};\n";
    if (kp.mode == MODE_UNGROUPED) s += "#define ACC(k, OP, x) a##k = word_combine(OP, a##k, (u64)(x))\n";
    else if (smem_dense && kp.dense_priv)
        s += "#define ACC(k, OP, val_) { u64* c_ = &s_priv[((k) * NQ_G + slot) * NQ_BLOCK + threadIdx.x]; *c_ = word_combine(OP, *c_, (u64)(val_)); }\n";
    else if (smem_dense) s += "#define ACC(k, OP, x) atomic_word<OP>(&s_tab[(k) * NQ_G + slot], (u64)(x))\n";
    else if (cached) {
        s += strf("#define NQ_CS %d\n", kp.cache_slots);
        // table update of a cache miss, per logical word: packed counters gather in a register (one RED per physical
        // word and row, issued after the row's aggregate code), every other word is one reduction.  The table's min / max /
        // or word is not read before its reduction: on config 5 reading first lost 20 % (1 277 -> 1 563 us per 200 M rows,
        // reading ahead for all four rows 1 766 us) and 43 % per 1 B rows (profiles/r02_config5_ablation.jsonl) - the
        // kernel is bound by LSU wavefronts, and a scattered load costs as many as the reduction it saves.
        for (int w = 0; w < W; ++w) {
            const int P = kp.phys_of[w];
            if (kp.bits_of[w] != 64) s += strf("#define ACCM_%d(OP, val_) pk%d += (u64)(val_) << %d\n", w, P, kp.shift_of[w]);
            else s += strf("#define ACCM_%d(OP, val_) atomic_word<OP>(&p.acc[%dULL * cap + (u64)slot], (u64)(val_))\n", w, P);
        }
        for (int w = 0; w < W; ++w) {
            std::string hit;
            const int ci = kp.cell_idx[w];
            switch (kp.cell_kind[w]) {
                case CK_CNT: hit = strf("reds_add(a_c32 + 4 * (%d * NQ_CS + cslot), (u32)(val_))", ci); break;
                case CK_WIDE: hit = strf("cache_add_wide(&s_c32[%d * NQ_CS + cslot], &s_c32[%d * NQ_CS + cslot], (u64)(val_))", ci, ci + 1); break;
                case CK_WIDE1: hit = strf("cache_add_carry(a_c32 + 4 * (%d * NQ_CS + cslot), (u64)(val_), &p.acc[%dULL * cap + klo])", ci, kp.phys_of[w]); break;
                case CK_MM32:
                    // interleaved with its neighbour: the hit phase has loaded both cells of the slot with one 64-bit load (mmpN)
                    if (kp.cell_pair[w]) hit = strf("cache_mm32_cur<OP>(a_c32 + 4 * (%s), (u64)(val_), %lluULL, (u32)(mmp%d%s))", cell32(kp, w, "cslot").c_str(),
                                                    (unsigned long long)kp.word_lo[w], kp.cell_pair[w] == 1 ? w : w - 1, kp.cell_pair[w] == 1 ? "" : " >> 32");
                    else hit = strf("cache_mm32<OP>(a_c32 + 4 * (%d * NQ_CS + cslot), (u64)(val_), %lluULL)", ci, (unsigned long long)kp.word_lo[w]);
                    break;
                case CK_OR32: hit = strf("cache_or32(a_c32 + 4 * (%d * NQ_CS + cslot), (u32)(val_))", ci); break;
                default: hit = strf("cache_word64<OP>(&s_c64[%d * NQ_CS + cslot], (u64)(val_))", ci); break;
            }
            s += strf("#define ACCH_%d(OP, val_) %s\n", w, hit.c_str());
        }
    }
    else s += "#define ACC(k, OP, x) if (nq_first) atomic_word<OP>(&p.acc[(u64)(k) * cap + (u64)slot], (u64)(x))\n";
    s += strf("#define NQ_BLOCK %d\n", kp.block);
    // One 1024-thread block per SM at 64 registers per thread owns the whole register file: no other kernel - the next
    // step's table re-arm, the flag wait and the finalisation of the step before - can start on that SM until the scan
    // ends.  Capped at 56 registers the scan leaves 8 K registers per SM, enough for a 256-thread block of those, so a
    // second step in flight overlaps its merge and finalisation with this scan.  (__maxnreg__ replaces
    // __launch_bounds__: the two cannot be combined.)
    const int cap_regs = cached && kp.block == 1024 ? 56 : 0;
    if (cap_regs > 0 && cap_regs * kp.block <= 65536) s += strf("extern \"C\" __global__ void __maxnreg__(%d) nq_scan(const NqParams p) {\n", cap_regs);
    else if (kp.min_blocks > 0) s += strf("extern \"C\" __global__ void __launch_bounds__(NQ_BLOCK, %d) nq_scan(const NqParams p) {\n", kp.min_blocks);
    else s += "extern \"C\" __global__ void __launch_bounds__(NQ_BLOCK) nq_scan(const NqParams p) {\n";
    if (kp.pdl) s += "    asm volatile(\"griddepcontrol.launch_dependents;\");\n";
    // later passes over a sliced DISTINCT bitmap only set bits: the group table was fed by pass 0
    s += kp.set_passes > 1 ? "    const bool nq_first = p.set_pass == 0;\n" : "    const bool nq_first = true; (void)nq_first;\n";
    return s;
}

// per-mode state: accumulator registers, the (private) shared-memory table, or the front cache
std::string scan_state(const KernelPlan& kp) {
    const int W = (int)kp.word_ops.size();
    std::string s;
    if (kp.mode == MODE_UNGROUPED) {
        for (int w = 0; w < W; ++w) s += strf("    u64 a%d = word_identity(%s);\n", w, op_name(kp.word_ops[w]));
    } else if (kp.mode == MODE_DENSE && !kp.dense_global && kp.dense_priv) {
        s += "    extern __shared__ u64 s_priv[];  // [NQ_W * NQ_G cells][NQ_BLOCK threads]: cell c of thread t at c * NQ_BLOCK + t\n";
        s += "#pragma unroll\n";
        s += "    for (int c = 0; c < NQ_W * NQ_G; ++c) s_priv[c * NQ_BLOCK + threadIdx.x] = word_identity(nq_ops[c / NQ_G]);\n";
    } else if (kp.mode == MODE_DENSE && !kp.dense_global) {
        s += "    __shared__ u64 s_tab[NQ_W * NQ_G];\n";
        s += "    for (int i = threadIdx.x; i < NQ_W * NQ_G; i += 256) s_tab[i] = word_identity(nq_ops[i / NQ_G]);\n";
        s += "    __syncthreads();\n";
    } else {
        s += "    const u64 cap = p.cap_mask + 1;\n";
        if (kp.cache_slots) {
            s += "    extern __shared__ u64 s_dyn[];\n";
            if (kp.cache_key32) {
                s += strf("    u64* const s_c64 = s_dyn;             // [%d][NQ_CS] 64-bit cells\n", kp.cache_n64);
                s += strf("    u32* const s_ckey = (u32*)(s_dyn + %d * NQ_CS);  // [NQ_CS] cached group keys, direct-mapped (all ones = empty)\n", kp.cache_n64);
                s += strf("    u32* const s_c32 = s_ckey + NQ_CS;    // [%d][NQ_CS] 32-bit cells\n", kp.cache_n32);
            } else {
                s += "    u64* const s_ckey = s_dyn;            // [NQ_CS] cached group keys (all ones = empty)\n";
                s += strf("    u64* const s_c64 = s_dyn + NQ_CS;     // [%d][NQ_CS] 64-bit cells\n", kp.cache_n64);
                s += strf("    u32* const s_c32 = (u32*)(s_dyn + %d * NQ_CS);  // [%d][NQ_CS] 32-bit cells\n", 1 + kp.cache_n64, kp.cache_n32);
            }
            s += "    (void)s_c64; (void)s_c32;\n";
            // 32-bit shared addresses made once: the row loop's 32-bit cells and u32 keys are accessed through them
            s += "    const u32 a_ckey = smem_addr(s_ckey), a_c32 = smem_addr(s_c32); (void)a_ckey; (void)a_c32;\n";
            s += "    for (int i = threadIdx.x; i < NQ_CS; i += NQ_BLOCK) {\n";
            s += kp.cache_key32 ? "        s_ckey[i] = 0xffffffffu;\n" : "        s_ckey[i] = NQ_U64_MAX;\n";
            for (int w = 0; w < W; ++w) {
                const int ci = kp.cell_idx[w], op = kp.word_ops[w];
                switch (kp.cell_kind[w]) {
                    case CK_WIDE: s += strf("        s_c32[%d * NQ_CS + i] = 0; s_c32[%d * NQ_CS + i] = 0;\n", ci, ci + 1); break;
                    case CK_MM32: s += strf("        s_c32[%s] = %s;\n", cell32(kp, w, "i").c_str(), mm32_empty(op)); break;
                    case CK_64: s += strf("        s_c64[%d * NQ_CS + i] = word_identity(%s);\n", ci, op_name(op)); break;
                    default: s += strf("        s_c32[%d * NQ_CS + i] = 0;\n", ci); break;
                }
            }
            s += "    }\n";
            s += "    __syncthreads();\n";
            s += "    bool cache_on = nq_first;  // per warp: switched off after 4 tiles when fewer than 1 in 4 rows hit\n";
            s += "    unsigned nlook = 0, nhit = 0; int tiles = 0;\n";
        }
    }
    return s;
}

// The cached modes' rows, three phases per 4 rows, so that the lanes of a warp diverge once per phase instead of once per
// accumulator word: (1) filter, group key and front-cache probe of all four rows (the four probes are independent: their
// shared-memory latencies overlap); (2) rows whose key is cached update shared-memory cells; (3) the others insert into
// the HBM table and update it with L2 atomics.
std::string cached_rows(const KernelPlan& kp, const RowCode& rc, const std::string& decls) {
    const int W = (int)kp.word_ops.size();
    std::string s;
    s += "        u64 kk[4]; int cs[4];  // group key / cache slot (-1: not cached, -2: row not selected)\n";
    s += "        __syncwarp();\n";
    // only the grid's last tile can hold rows at or beyond nrows: phase (1) is emitted twice, and full tiles run the
    // copy without the per-row 64-bit bounds check
    std::string p1;
    p1 += select_row(rc, decls, "NQ_IN_RANGE(j)");
    p1 += "            cs[j] = -2; kk[j] = 0;\n";
    // MISSING / NULL keys (one row in five of config 5, two slots) are cached like any other key.  Register
    // accumulators for them were removed: -16 % per 1 B config-5 rows (4.95 -> 5.72 ms, profiles/r02_config5_ablation.jsonl),
    // ~55 extra instructions per row on a kernel whose issue slots are already 68 % busy.
    p1 += "            if (pass) {\n";
    p1 += rc.key;
    p1 += "                    kk[j] = klo;\n";
    p1 += "                    ++nlook;\n";
    if (kp.cache_key32) p1 += "                    cs[j] = cache_on ? cache_claim_1(a_ckey, NQ_CS, (u32)klo * 0x9E3779B1u, (u32)klo) : -1;\n";
    else if (kp.key_bits <= 32) p1 += "                    cs[j] = cache_on ? cache_claim_n(s_ckey, NQ_CS, (u32)klo * 0x9E3779B1u, klo) : -1;\n";
    else p1 += "                    cs[j] = cache_on ? cache_claim_n(s_ckey, NQ_CS, (u32)(mix64(klo) >> 32), klo) : -1;\n";
    p1 += "                    nhit += cs[j] >= 0;\n";
    p1 += "            }\n";
    p1 += "        }\n";
    s += "        if (wbase + 128 <= nrows) {\n";
    s += "#define NQ_IN_RANGE(j) true\n";
    s += p1;
    s += "#undef NQ_IN_RANGE\n";
    s += "        } else {\n";
    s += "#define NQ_IN_RANGE(j) (base + (j) < nrows)\n";
    s += p1;
    s += "#undef NQ_IN_RANGE\n";
    s += "        }\n";
    s += "#define ACC(k, OP, val_) if (nq_first) ACCH_##k(OP, val_)\n";
    s += "#pragma unroll\n";
    s += "        for (int j = 0; j < 4; ++j) {\n";
    s += "            // warp-ballot selection mask (also the point where the lanes of the warp reconverge)\n";
    s += "            if (__ballot_sync(0xffffffffu, cs[j] >= 0) == 0) continue;\n";
    s += "            if (cs[j] >= 0) {\n";
    s += "                    const int cslot = cs[j]; const u64 klo = kk[j]; (void)klo;\n";
    for (int w = 0; w < W; ++w)
        if (kp.cell_pair[w] == 1)
            s += strf("                    const u64 mmp%d = *(volatile u64*)__cvta_shared_to_generic(a_c32 + 4 * (%d * NQ_CS + 2 * cslot));  // both cells of the slot: one LDS.64\n", w, kp.cell_idx[w]);
    s += decls;
    s += rc.agg;
    s += "            }\n";
    s += "        }\n";
    s += "#undef ACC\n";
    s += "#define ACC(k, OP, val_) if (nq_first) ACCM_##k(OP, val_)\n";
    s += "#pragma unroll\n";
    s += "        for (int j = 0; j < 4; ++j) {\n";
    s += "            if (__ballot_sync(0xffffffffu, cs[j] == -1) == 0) continue;\n";
    s += "            if (cs[j] == -1) {\n";
    s += "                    const u64 klo = kk[j];\n";
    s += hbm_slot(kp, "                    ", "klo", "  // direct-indexed table");
    std::set<int> packed_phys;
    for (int w = 0; w < W; ++w) if (kp.bits_of[w] != 64) packed_phys.insert(kp.phys_of[w]);
    for (int P : packed_phys) s += strf("                    u64 pk%d = 0;\n", P);
    s += decls;
    s += rc.agg;
    for (int P : packed_phys) s += strf("                    if (pk%d) atomicAdd(&p.acc[%dULL * cap + (u64)slot], pk%d);\n", P, P, P);
    s += "            }\n";
    s += "        }\n";
    s += "#undef ACC\n";
    s += "        if (cache_on && ++tiles == 4) {  // warp-uniform: is the front cache earning its probes?\n";
    s += "            const unsigned L = __reduce_add_sync(0xffffffffu, nlook), H = __reduce_add_sync(0xffffffffu, nhit);\n";
    s += "            if (H * 4 < L) cache_on = false;\n";
    s += "        }\n";
    return s;
}

// the grid-stride loop over warp tiles of 4 rows per lane
std::string scan_rows(const KernelPlan& kp, const Table& t, const RowCode& rc, const std::string& decls) {
    std::string s;
    s += "    const i64 nrows = p.nrows;\n";
    s += "    const int lane = threadIdx.x & 31;\n";
    s += "    const i64 stride = (i64)gridDim.x * (NQ_BLOCK * 4);\n";
    s += "    // warp-uniform trip count: every lane of a warp stays in the loop while the warp has rows\n";
    s += "    int nq_tile = 0;\n";
    s += "    for (i64 wbase = (i64)blockIdx.x * (NQ_BLOCK * 4) + (threadIdx.x >> 5) * 128; wbase < nrows; wbase += stride) {\n";
    s += "        if ((++nq_tile & 31) == 0 && nq_cancelled(p, lane)) break;  // SendStop: the host discards whatever was aggregated\n";
    s += "        const i64 base = wbase + lane * 4;\n";
    for (int c : kp.used_cols) {
        const Column& col = t.cols[c];
        if (col.width == 8) s += strf("        i64 c%d[4]; ld_rows4_b64((const i64*)p.col[%d] + base, c%d);\n", c, c, c);
        else if (col.width == 4) s += strf("        u32 c%d[4]; ld_rows4_b32((const u32*)p.col[%d] + base, c%d);\n", c, c, c);
        if (!col.stats.uniform_tag() && col.stats.class_mask) s += strf("        int t%d[4]; ld_rows4_b8(p.tag[%d] + base, t%d);\n", c, c, c);
    }
    if (kp.cache_slots > 0) s += cached_rows(kp, rc, decls);
    else {
        s += select_row(rc, decls, "base + j < nrows");
        s += "            // warp-ballot selection mask: skip the aggregation when no lane selected its row\n";
        s += "            const unsigned sel = __ballot_sync(0xffffffffu, pass);\n";
        s += "            if (sel == 0) continue;\n";
        s += "            if (pass) {\n";
        s += rc.agg;
        s += "            }\n";
        s += "        }\n";
    }
    s += "    }\n";
    return s;
}

// flush the block's cached groups into the HBM table: one insert + one atomic per word per cached key
std::string cache_flush(const KernelPlan& kp) {
    const int W = (int)kp.word_ops.size();
    std::string s;
    s += "    __syncthreads();\n";
    s += "    for (int i = threadIdx.x; i < NQ_CS; i += NQ_BLOCK) {\n";
    s += "        const u64 key = s_ckey[i];\n";
    s += kp.cache_key32 ? "        if (key == 0xffffffffULL) continue;\n" : "        if (key == NQ_U64_MAX) continue;\n";
    s += hbm_slot(kp, "        ", "key", "");
    for (int P = 0; P < (int)kp.phys_ops.size(); ++P) {  // packed counters: both fields leave in one reduction
        std::string v;
        for (int w = 0; w < W; ++w)
            if (kp.phys_of[w] == P && kp.bits_of[w] != 64)
                v += strf("%s((u64)s_c32[%d * NQ_CS + i] << %d)", v.empty() ? "" : " | ", kp.cell_idx[w], kp.shift_of[w]);
        if (!v.empty()) s += strf("        { const u64 v = %s; if (v) atomicAdd(&p.acc[%dULL * cap + (u64)slot], v); }\n", v.c_str(), P);
    }
    for (int w = 0; w < W; ++w) {
        if (kp.bits_of[w] != 64) continue;
        const int ci = kp.cell_idx[w], op = kp.word_ops[w];
        const std::string dst = strf("&p.acc[%dULL * cap + (u64)slot]", kp.phys_of[w]);
        switch (kp.cell_kind[w]) {
            case CK_WIDE:
                s += strf("        { const u64 v = ((u64)s_c32[%d * NQ_CS + i] << 32) + (u64)s_c32[%d * NQ_CS + i]; if (v) atomic_word<%s>(%s, v); }\n",
                          ci + 1, ci, op_name(op), dst.c_str());
                break;
            case CK_MM32:
                s += strf("        { const u32 c = s_c32[%s]; if (c != %s) atomic_word<%s>(%s, (u64)(c - 1u) + %lluULL); }\n", cell32(kp, w, "i").c_str(),
                          mm32_empty(op), op_name(op), dst.c_str(), (unsigned long long)kp.word_lo[w]);
                break;
            case CK_64:
                s += strf("        { const u64 v = s_c64[%d * NQ_CS + i]; if (v != word_identity(%s)) atomic_word<%s>(%s, v); }\n", ci, op_name(op),
                          op_name(op), dst.c_str());
                break;
            default:
                s += strf("        { const u64 v = s_c32[%d * NQ_CS + i]; if (v) atomic_word<%s>(%s, v); }\n", ci, op_name(op), dst.c_str());
                break;
        }
    }
    s += "    }\n";
    return s;
}

// the block epilogue: fold the block's accumulators into the persistent state; the last block publishes it
std::string scan_epilogue(const KernelPlan& kp) {
    const int W = (int)kp.word_ops.size();
    std::string s;
    if (kp.mode == MODE_UNGROUPED) {
        // Block epilogue: warp-shuffle reduce every word, one barrier, then thread w folds word w's 8 warp values in
        // order.  Order-independent words (integer add / min / max / or) go straight into persistent accumulators
        // with one atomic per block; float64 sums are kept as per-block partials and folded in a fixed order by the
        // last block to finish, so float results are run-to-run identical.  That block also publishes the final
        // words to HBM and, zero-copy, to mapped pinned host memory, and re-arms the accumulators.
        s += "    __shared__ u64 s_part[NQ_W][8];\n";
        s += "    __shared__ u64 scratch[32];\n";
        s += "    {\n        const int warp = threadIdx.x >> 5;\n";
        for (int w = 0; w < W; ++w)
            s += strf("        { const u64 r = warp_reduce_word<%s>(a%d); if (lane == 0) s_part[%d][warp] = r; }\n", op_name(kp.word_ops[w]), w, w);
        s += "    }\n";
        s += "    __syncthreads();\n";
        s += "    if (threadIdx.x < NQ_W) {\n";
        s += "        const int w = threadIdx.x, op = nq_ops[w];\n";
        s += "        u64 r = s_part[w][0];\n";
        s += "        for (int k = 1; k < 8; ++k) r = word_combine(op, r, s_part[w][k]);\n";
        s += "        if (op == OP_ADD_F64) p.partials[(u64)nq_fidx[w] * gridDim.x + blockIdx.x] = r;\n";
        s += "        else if (r != word_identity(op)) atomic_word_dyn(op, &p.acc[w], r);\n";
        s += "    }\n";
        s += "    if (last_block_arrives(p.ticket)) {\n";
        s += "        if (threadIdx.x < NQ_W && nq_ops[threadIdx.x] != OP_ADD_F64) {\n";
        s += "            const u64 v = atomicExch(&p.acc[threadIdx.x], word_identity(nq_ops[threadIdx.x]));\n";
        s += "            p.final_dev[threadIdx.x] = v; p.final_host[threadIdx.x] = v;\n";
        s += "        }\n";
        for (int w = 0, fi = 0; w < W; ++w) {
            if (kp.word_ops[w] != OP_ADD_F64) continue;
            s += "        {\n";
            s += "            u64 t[5];\n";
            s += "#pragma unroll\n";
            s += strf("            for (int k = 0; k < 5; ++k) { const unsigned b = threadIdx.x + k * 256; t[k] = b < gridDim.x ? __ldcg(&p.partials[(u64)%d * gridDim.x + b]) : 0ULL; }\n", fi);
            s += "            u64 v = t[0];\n";
            s += "#pragma unroll\n";
            s += "            for (int k = 1; k < 5; ++k) v = word_combine(OP_ADD_F64, v, t[k]);\n";
            s += "            v = block_reduce_word<OP_ADD_F64>(v, scratch);\n";
            s += strf("            if (threadIdx.x == 0) { p.final_dev[%d] = v; p.final_host[%d] = v; }\n", w, w);
            s += "        }\n";
            ++fi;
        }
        s += "        if (p.peer_mail) mailbox_push(p, p.final_dev);  // fused all-gather: peer stores over NVLink\n";
        s += "    }\n";
    } else if (kp.mode == MODE_DENSE && !kp.dense_global) {
        if (kp.dense_priv) {
            // fold the private copies of every cell: one warp-shuffle reduction per warp and cell, then thread c folds cell c's
            // warp values in order and applies one global atomic per (block, cell)
            s += "    __shared__ u64 s_wpart[NQ_W * NQ_G][NQ_BLOCK / 32];\n";
            s += "    for (int c = 0; c < NQ_W * NQ_G; ++c) {\n";
            s += "        const u64 r = warp_reduce_dyn(nq_ops[c / NQ_G], s_priv[c * NQ_BLOCK + threadIdx.x]);\n";
            s += "        if (lane == 0) s_wpart[c][threadIdx.x >> 5] = r;\n";
            s += "    }\n";
            s += "    __syncthreads();\n";
            s += "    if (threadIdx.x < NQ_W * NQ_G) {\n";
            s += "        const int op = nq_ops[threadIdx.x / NQ_G];\n";
            s += "        u64 v = s_wpart[threadIdx.x][0];\n";
            s += "        for (int k = 1; k < NQ_BLOCK / 32; ++k) v = word_combine(op, v, s_wpart[threadIdx.x][k]);\n";
            s += "        if (v != word_identity(op)) atomic_word_dyn(op, &p.acc[threadIdx.x], v);\n";
            s += "    }\n";
        } else {
            s += "    __syncthreads();\n";
            s += "    for (int i = threadIdx.x; i < NQ_W * NQ_G; i += 256) {\n";
            s += "        const int op = nq_ops[i / NQ_G];\n";
            s += "        const u64 v = s_tab[i];\n";
            s += "        if (v != word_identity(op)) atomic_word_dyn(op, &p.acc[i], v);\n";
            s += "    }\n";
        }
        s += "    if (last_block_arrives(p.ticket)) {\n";
        s += "        for (int i = threadIdx.x; i < NQ_W * NQ_G; i += NQ_BLOCK) p.final_host[i] = __ldcg(&p.acc[i]);\n";
        s += "        if (p.peer_mail) mailbox_push(p, p.acc);\n";
        s += "    }\n";
    }
    if (kp.pdl) s += "    asm volatile(\"griddepcontrol.wait;\" ::: \"memory\");  // complete in stream order\n";
    s += "}\n";
    return s;
}

// the partitioning kernel of the partitioned DISTINCT aggregation (see KernelPlan::part)
std::string emit_partition(const KernelPlan& kp, const Table& t, const RowCode& rc, const std::string& decls) {
    std::string q;
    q += "// generated by libn1gpu codegen: the partitioning kernel of this chain's partitioned DISTINCT aggregation\n";
    q += "#include \"n1ql_device.cuh\"\n";
    q += strf("#define NQ_BLOCK %d\n", PART_THREADS);
    q += strf("#define NP %d\n#define BINCAP %d\n#define GBITS %d\n#define ROUND_TILES 8\n", 1 << kp.part_bits, kp.part_bincap, kp.part_gbits);
    q += "extern \"C\" __global__ void __launch_bounds__(NQ_BLOCK, 1) nq_scan(const NqParams p) {\n";
    q += "    extern __shared__ u32 s_part[];\n";
    q += "    __shared__ int s_stop;\n";
    q += "    u32* const s_cnt = s_part;        // [NP] records staged per partition in this round\n";
    q += "    u32* const s_bin = s_part + NP;   // [NP][BINCAP]\n";
    q += "    u32* const g_recs = (u32*)p.set_keys;  // [NP][part_cap] partitioned records\n";
    q += "    u32* const g_cur = (u32*)p.keys;       // [NP] records written per partition\n";
    q += "    const u64 part_cap = p.set_mask;\n";
    q += "    const i64 nrows = p.nrows;\n";
    q += "    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;\n";
    q += "    const i64 tile = NQ_BLOCK * 4;\n";
    q += "    const i64 ntiles = (nrows + tile - 1) / tile;\n";
    // columns of the tile being processed (c*, t*) and of the next tile this block will process (nc*, nt*): the next
    // tile's loads are in flight while this one is partitioned - also across the flush at the end of a round
    std::string load_next, take_next;
    for (int c : kp.used_cols) {
        const Column& col = t.cols[c];
        const bool tags = !col.stats.uniform_tag() && col.stats.class_mask;
        if (col.width == 8) { q += strf("    i64 c%d[4], nc%d[4];\n", c, c); load_next += strf("ld_rows4_b64((const i64*)p.col[%d] + nb, nc%d); ", c, c); }
        else if (col.width == 4) { q += strf("    u32 c%d[4], nc%d[4];\n", c, c); load_next += strf("ld_rows4_b32((const u32*)p.col[%d] + nb, nc%d); ", c, c); }
        if (col.width) take_next += strf("c%d[j] = nc%d[j]; ", c, c);
        if (tags) { q += strf("    int t%d[4], nt%d[4];\n", c, c); load_next += strf("ld_rows4_b8(p.tag[%d] + nb, nt%d); ", c, c); take_next += strf("t%d[j] = nt%d[j]; ", c, c); }
    }
    q += "    const i64 round_stride = (i64)gridDim.x * ROUND_TILES;\n";
    q += "    { const i64 nt_ = (i64)blockIdx.x * ROUND_TILES; if (nt_ < ntiles) { const i64 nb = nt_ * tile + threadIdx.x * 4; " + load_next + "} }\n";
    q += "    for (i64 t0 = (i64)blockIdx.x * ROUND_TILES; t0 < ntiles; t0 += round_stride) {\n";
    q += "        for (int i = threadIdx.x; i < NP; i += NQ_BLOCK) s_cnt[i] = 0;\n";
    q += "        if (threadIdx.x == 0) s_stop = *(volatile const int*)p.cancel;  // SendStop while the scan runs\n";
    q += "        __syncthreads();\n";
    q += "        if (s_stop) break;\n";
    q += "        for (int tt = 0; tt < ROUND_TILES && t0 + tt < ntiles; ++tt) {\n";
    q += "        const i64 base = (t0 + tt) * tile + threadIdx.x * 4;\n";
    q += "#pragma unroll\n";
    q += "        for (int j = 0; j < 4; ++j) { " + take_next + "}\n";
    q += "        {   // the tile after this one: the next of the round, or the first of this block's next round\n";
    q += "            const i64 nt_ = (tt + 1 < ROUND_TILES && t0 + tt + 1 < ntiles) ? t0 + tt + 1 : t0 + round_stride;\n";
    q += "            if (nt_ < ntiles) { const i64 nb = nt_ * tile + threadIdx.x * 4; " + load_next + "}\n";
    q += "        }\n";
    q += select_row(rc, decls, "base + j < nrows");
    q += "            if (pass) {\n";
    q += rc.key;
    q += rc.part_value;
    q += "                    const u32 rec = (u32)(klo & ((1ULL << GBITS) - 1)) | ((u32)hasv << GBITS) | ((u32)vlo << (GBITS + 1));\n";
    q += "                    const u32 part = (u32)(klo >> GBITS);\n";
    q += "                    const u32 pos = atomicAdd(&s_cnt[part], 1u);\n";
    q += "                    if (pos < BINCAP) s_bin[part * BINCAP + pos] = rec;\n";
    q += "                    else {  // the bin is full for this round: straight to the partition (rare unless the keys are skewed)\n";
    q += "                        const u32 at = atomicAdd(&g_cur[part], 1u);\n";
    q += "                        if (at < part_cap) g_recs[(u64)part * part_cap + at] = rec; else p.status[0] = 4;\n";
    q += "                    }\n";
    q += "            }\n";
    q += "        }\n";
    q += "        }\n";
    q += "        __syncthreads();\n";
    q += "        // flush: lane l of warp w reserves room for partition w * 32 + l (32 reservations in flight per warp), then the\n";
    q += "        // warp copies the 32 bins one after the other, a contiguous run of records each\n";
    q += "        for (int p0 = warp * 32; p0 < NP; p0 += NQ_BLOCK) {\n";
    q += "            const int mine = p0 + lane;\n";
    q += "            u32 n = mine < NP ? min(s_cnt[mine], (u32)BINCAP) : 0u, gb = 0;\n";
    q += "            if (n) gb = atomicAdd(&g_cur[mine], n);\n";
    q += "            for (int k = 0; k < 32; ++k) {\n";
    q += "                const u32 nk = __shfl_sync(0xffffffffu, n, k), bk = __shfl_sync(0xffffffffu, gb, k);\n";
    q += "                for (u32 i = lane; i < nk; i += 32) {\n";
    q += "                    if (bk + i < part_cap) g_recs[(u64)(p0 + k) * part_cap + bk + i] = s_bin[(p0 + k) * BINCAP + i]; else p.status[0] = 4;\n";
    q += "                }\n";
    q += "            }\n";
    q += "        }\n";
    q += "        __syncthreads();\n";
    q += "    }\n";
    q += "}\n";
    return q;
}

}  // namespace

KernelPlan generate_kernel(const Table& t, const Expr* where, const std::vector<ExprP>& keys,
                           const std::vector<ExprP>& aggs, const std::vector<std::string>& agg_texts,
                           double total_rows_bound) {
    KernelPlan kp = plan_layout(t, keys, aggs, agg_texts, total_rows_bound);
    Gen g(t);
    const RowCode rc = emit_row_code(g, kp, where, keys, aggs);
    for (auto& kv : g.colvar) kp.used_cols.push_back(kv.first);
    for (int c : kp.used_cols) kp.scan_bytes_per_row += t.scan_bytes(c);
    kp.source = scan_prologue(kp) + scan_state(kp) + scan_rows(kp, t, rc, g.decls) + (kp.cache_slots > 0 ? cache_flush(kp) : "") + scan_epilogue(kp);
    if (kp.part) kp.part_source = emit_partition(kp, t, rc, g.decls);
    kp.consts = g.consts;
    kp.in_sets = std::move(g.in_sets);
    return kp;
}

}  // namespace n1
