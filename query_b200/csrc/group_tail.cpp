// group_tail.cpp — see group_tail.hpp.  Numbers, logic and the MISSING / NULL folds are the value model of
// n1ql_value.cuh, the one the scan kernel runs, applied to the (class, payload) of host values.  Only strings differ:
// here they are compared and tested for truth as bytes, where the kernel compares dictionary ranks.
#include "group_tail.hpp"

#include <algorithm>
#include <cmath>
#include <functional>
#include <map>
#include <thread>

namespace n1 {
namespace execution {

namespace {

HValue missing() { return HValue::missing(); }
HValue null() { return HValue::null(); }

// A host value as n1ql_value.cuh sees it.  A string's payload says only whether it is non-empty, which is all that
// v_truth (with empty2 = 0) reads of it: comparisons of two strings are made on the bytes (str_cmp below).
Val val(const HValue& v) { return mkv(v.cls, v.cls == C_STRING ? (i64)!v.s.empty() : v.bits); }
bool both_strings(const HValue& a, const HValue& b) { return a.cls == C_STRING && b.cls == C_STRING; }
int str_cmp(const HValue& a, const HValue& b) { const int c = a.s.compare(b.s); return c < 0 ? -1 : (c > 0 ? 1 : 0); }

int compare(const HValue& a, const HValue& b) {  // Value.Compare
    return both_strings(a, b) ? str_cmp(a, b) : v_compare(val(a), val(b));
}
HValue eq(const HValue& a, const HValue& b) {  // Value.Equals (comp_eq.go:76-78)
    return both_strings(a, b) ? HValue::boolean(a.s == b.s) : HValue(v_eq(val(a), val(b)));
}
bool truth(const HValue& v) { return v_truth(val(v), 0); }  // Value.Truth

// What an expression node of the tail resolves to, decided once at add() time.
enum { R_EVAL = 0, R_KEY = 1, R_AGG = 2, R_LET = 3, R_ALIAS = 4 };

struct Scope {
    const std::vector<std::string>* key_texts = nullptr;
    const std::vector<std::string>* agg_texts = nullptr;
    std::vector<std::string> let_vars;  // LETTING variables visible to the expression
    std::vector<std::string> aliases;   // explicit projection aliases (ORDER BY only)
};

int index_of(const std::vector<std::string>& v, const std::string& s) {
    for (size_t i = 0; i < v.size(); ++i) if (v[i] == s) return (int)i;
    return -1;
}

// Binds a node: col = R_* << 16 | index.  Throws INELIGIBLE when a leaf is neither a group key, an aggregate of the
// group operators, a LETTING variable nor (ORDER BY) a projection alias.
void bind(Expr& e, const Scope& sc) {
    e.col = R_EVAL << 16;
    if (e.kind == EK::AGG) {
        const int a = sc.agg_texts ? index_of(*sc.agg_texts, e.str()) : -1;
        if (a < 0) N1_THROW(N1GPU_E_INELIGIBLE, "aggregate %s is not computed by the group operators", e.str().c_str());
        e.col = R_AGG << 16 | a;
        return;
    }
    if (e.kind != EK::CONST && sc.key_texts) {
        const int k = index_of(*sc.key_texts, e.str());
        if (k >= 0) { e.col = R_KEY << 16 | k; return; }
    }
    if (e.kind == EK::IDENT) {
        int i = index_of(sc.aliases, e.name);
        if (i >= 0) { e.col = R_ALIAS << 16 | i; return; }
        i = index_of(sc.let_vars, e.name);
        if (i >= 0) { e.col = R_LET << 16 | i; return; }
        N1_THROW(N1GPU_E_INELIGIBLE, "identifier `%s` is neither a group key, a LETTING variable nor a projection alias", e.name.c_str());
    }
    if (e.kind == EK::FIELD) N1_THROW(N1GPU_E_INELIGIBLE, "%s is not a group key", e.str().c_str());
    if (e.kind == EK::ARRAY) N1_THROW(N1GPU_E_INELIGIBLE, "an array construct is only evaluated as the right side of IN");
    if (e.kind == EK::IN) {
        if (e.ops[1]->kind != EK::ARRAY) N1_THROW(N1GPU_E_INELIGIBLE, "IN over something other than an array construct");
        bind(*e.ops[0], sc);
        e.ops[1]->col = R_EVAL << 16;
        for (auto& el : e.ops[1]->ops) bind(*el, sc);
        return;
    }
    for (auto& o : e.ops) bind(*o, sc);
}

struct Env {
    const Result* r = nullptr;
    i64 g = 0;
    const std::vector<HValue>* lets = nullptr;
    const std::vector<HValue>* aliases = nullptr;
};

HValue eval(const Expr& e, const Env& env) {
    const int how = e.col >> 16, idx = e.col & 0xffff;
    switch (how) {
        case R_KEY: return env.r->key(env.g, idx);
        case R_AGG: return env.r->agg(env.g, idx);
        case R_LET: return (*env.lets)[(size_t)idx];
        case R_ALIAS: return (*env.aliases)[(size_t)idx];
        default: break;
    }
    switch (e.kind) {
        case EK::CONST: return e.cval;
        case EK::ADD: case EK::MULT: {  // arith_add.go:51-70, arith_mult.go:51-70
            Val acc = mkint(e.kind == EK::ADD ? 0 : 1);
            bool m = false, n = false;
            for (auto& o : e.ops) {
                const Val a = val(eval(*o, env));
                if (e.kind == EK::ADD) add_arg(a, acc, m, n); else mult_arg(a, acc, m, n);
            }
            return arith_fin(acc, m, n);
        }
        case EK::SUB: return v_sub(val(eval(*e.ops[0], env)), val(eval(*e.ops[1], env)));
        case EK::DIV: return v_div(val(eval(*e.ops[0], env)), val(eval(*e.ops[1], env)));
        case EK::MOD: return v_mod(val(eval(*e.ops[0], env)), val(eval(*e.ops[1], env)));
        case EK::NEG: return v_neg(val(eval(*e.ops[0], env)));
        case EK::EQ: return eq(eval(*e.ops[0], env), eval(*e.ops[1], env));
        case EK::LT: { const int c = compare(eval(*e.ops[0], env), eval(*e.ops[1], env)); return cmp_result(c, c < 0); }
        case EK::LE: { const int c = compare(eval(*e.ops[0], env), eval(*e.ops[1], env)); return cmp_result(c, c <= 0); }
        case EK::BETWEEN: {  // comp_between.go:58-78
            const HValue x = eval(*e.ops[0], env);
            const int lc = compare(x, eval(*e.ops[1], env));
            if (lc == CMP_MISSING) return missing();
            const int hc = compare(x, eval(*e.ops[2], env));
            if (hc == CMP_MISSING) return missing();
            if (lc == CMP_NULL || hc == CMP_NULL) return null();
            return HValue::boolean(lc >= 0 && hc <= 0);
        }
        case EK::IN: {  // coll_in.go:61-91 over an array construct
            const HValue x = eval(*e.ops[0], env);
            if (e.ops[1]->kind != EK::ARRAY) N1_THROW(N1GPU_E_INELIGIBLE, "IN over a non-constructed array");
            bool hit = false, m = false, n = false;
            for (auto& el : e.ops[1]->ops) {
                const HValue ev = eval(*el, env);
                if (both_strings(x, ev)) hit = hit || x.s == ev.s; else in_arg(val(x), val(ev), hit, m, n);
            }
            return in_fin(val(x), hit, m, n);
        }
        case EK::AND: {  // logic_and.go:64-88
            bool f = false, m = false, n = false;
            for (auto& o : e.ops) and_arg(val(eval(*o, env)), 0, f, m, n);
            return and_fin(f, m, n);
        }
        case EK::OR: {  // logic_or.go:98-122
            bool t = false, m = false, n = false;
            for (auto& o : e.ops) or_arg(val(eval(*o, env)), 0, t, m, n);
            return or_fin(t, m, n);
        }
        case EK::NOT: return v_not(val(eval(*e.ops[0], env)), 0);  // logic_not.go:57-68
        case EK::ROUND: {  // expression/func_num.go:1304-1336 (Round.Apply) + :1715-1736 (roundFloat: half to even)
            const HValue a = eval(*e.ops[0], env);
            if (a.cls == C_MISSING) return a;
            if (!is_num(a.cls)) return null();
            i64 prec = 0;
            if (e.ops.size() > 1) {
                const HValue p = eval(*e.ops[1], env);
                if (p.cls == C_MISSING) return p;
                if (!is_num(p.cls) || p.num() != std::trunc(p.num())) return null();
                prec = go_i64(p.num());  // Go: p = int(pf)
            }
            double x = a.num();
            if (x != x || std::isinf(x)) return new_num(x);
            double sign = 1.0;
            if (x < 0) { sign = -1.0; x = -x; }
            const double pw = std::pow(10.0, (double)prec), inter = x * pw + 0.5;
            double r = std::floor(inter);
            if (r == inter && std::fmod(r, 2.0) != 0) r -= 1;
            return new_num(sign * r / pw);
        }
        case EK::IS_NULL: return v_is_null(val(eval(*e.ops[0], env)));
        case EK::IS_NOT_NULL: return v_is_not_null(val(eval(*e.ops[0], env)));
        case EK::IS_MISSING: return v_is_missing(val(eval(*e.ops[0], env)));
        case EK::IS_NOT_MISSING: return v_is_not_missing(val(eval(*e.ops[0], env)));
        case EK::IS_VALUED: return v_is_valued(val(eval(*e.ops[0], env)));
        case EK::IS_NOT_VALUED: return v_is_not_valued(val(eval(*e.ops[0], env)));
        default: break;
    }
    N1_THROW(N1GPU_E_INELIGIBLE, "expression %s cannot be evaluated over a group", e.str().c_str());
}

// expression Alias(): a field path is known by its last name, an identifier by its own (nav_field.go:55-57,260-262,
// identifier.go:66-68); everything else has none (base.go:163-165)
std::string expr_alias(const Expr& e) {
    if (e.kind == EK::FIELD || e.kind == EK::IDENT) return e.name;
    return std::string();
}

bool integral_operand(const Expr& e, i64* out) {  // offset.go:53-72, limit.go:53-72: a number whose Trunc equals itself
    const HValue v = eval_constant(e);
    if (!is_num(v.cls)) return false;
    const double d = v.num();
    if (std::trunc(d) != d) return false;
    *out = v.cls == C_INT ? v.bits : go_i64(d);
    return true;
}

}  // namespace

int collate_values(const HValue& a, const HValue& b) {
    return both_strings(a, b) ? str_cmp(a, b) : collate(val(a), val(b));
}

HValue eval_constant(const Expr& e) {
    ExprP copy = parse_expr(e.str());
    Scope sc;
    bind(*copy, sc);
    Env env;
    return eval(*copy, env);
}

std::string value_to_json(const HValue& v) {
    switch (v.cls) {
        case C_FALSE: return "false";
        case C_TRUE: return "true";
        case C_INT: return std::to_string(v.bits);
        case C_FLOAT: return json::format_float(v.f());
        case C_STRING: { std::string s; json::quote(v.s, s); return s; }
        default: return "null";
    }
}

bool GroupTail::add(const json::Node& op, const std::vector<std::string>& key_texts, const std::vector<std::string>& agg_texts) {
    const std::string name = op.str_or("#operator", "");
    try {
        Scope sc;
        sc.key_texts = &key_texts;
        sc.agg_texts = &agg_texts;
        for (auto& b : letting) sc.let_vars.push_back(b.var);
        if (name == "Let") {
            if (has_project || !having.empty() || !letting.empty()) return false;
            const json::Node* bs = op.get("bindings");
            if (!bs || bs->kind != json::Node::ARR) return false;
            std::vector<TailBinding> fresh;
            Scope none = sc;
            none.let_vars.clear();  // every binding is evaluated on the incoming item (let.go:53-60)
            for (auto& b : bs->arr) {
                TailBinding tb;
                tb.var = b.str_or("var", "");  // expression/binding.go:66-78
                tb.expr = b.str_or("expr", "");
                if (tb.var.empty() || tb.expr.empty() || b.get("desc") || b.get("name_var")) return false;
                tb.e = parse_expr(tb.expr);
                bind(*tb.e, none);
                fresh.push_back(std::move(tb));
            }
            letting = std::move(fresh);
        } else if (name == "Filter") {
            if (has_project || !having.empty()) return false;
            ExprP e = parse_expr(op.str_or("condition", ""));
            bind(*e, sc);
            having = op.str_or("condition", "");
            having_e = std::move(e);
        } else if (name == "InitialProject") {
            if (has_project) return false;
            const json::Node* d = op.get("distinct");
            const json::Node* raw = op.get("raw");
            if ((d && d->kind == json::Node::BOOL && d->b && !distinct_by_keys) || (raw && raw->kind == json::Node::BOOL && raw->b)) return false;
            const json::Node* ts = op.get("result_terms");
            if (!ts || ts->kind != json::Node::ARR || ts->arr.empty()) return false;
            std::vector<TailTerm> fresh;
            int next = 1;
            for (auto& t : ts->arr) {
                const json::Node* star = t.get("star");
                if (star && star->kind == json::Node::BOOL && star->b) return false;
                TailTerm tt;
                tt.expr = t.str_or("expr", "");
                tt.as = t.str_or("as", "");
                if (tt.expr.empty()) return false;
                tt.e = parse_expr(tt.expr);
                tt.alias = !tt.as.empty() ? tt.as : expr_alias(*tt.e);  // algebra/result.go:358-374
                // An explicit alias is also set on the scope ORDER BY sees, and setting a MISSING value there UNSETS it,
                // so a field of the item with the same name would show through (value/scope.go:31-45): keep such
                // plans - an alias named like the keyspace alias or a LETTING variable - with the caller.
                if (!tt.as.empty() && (tt.as == keyspace_alias || index_of(sc.let_vars, tt.as) >= 0)) return false;
                if (tt.alias.empty()) tt.alias = "$" + std::to_string(next++);
                bind(*tt.e, sc);
                // DISTINCT rows are the groups only while no two terms share an output name (a later one overrides)
                if (distinct_by_keys) for (auto& o : fresh) if (o.alias == tt.alias) return false;
                fresh.push_back(std::move(tt));
            }
            terms = std::move(fresh);
            has_project = true;
        } else if (name == "Distinct") {
            if (!distinct_by_keys || !has_project || !order.empty() || has_offset || has_limit) return false;  // already distinct: nothing to do
        } else if (name == "FinalProject") {
            if (!has_project || final_project) return false;
            final_project = true;
        } else if (name == "Order") {
            if (!has_project || final_project || !order.empty() || has_offset || has_limit) return false;
            const json::Node* ts = op.get("sort_terms");
            if (!ts || ts->kind != json::Node::ARR || ts->arr.empty()) return false;
            for (auto& t : terms) if (!t.as.empty()) sc.aliases.push_back(t.as);
            std::vector<TailSort> fresh;
            for (auto& t : ts->arr) {
                TailSort s;
                s.expr = t.str_or("expr", "");
                const json::Node* d = t.get("desc");
                s.desc = d && d->kind == json::Node::BOOL && d->b;
                if (s.expr.empty()) return false;
                s.e = parse_expr(s.expr);
                bind(*s.e, sc);
                fresh.push_back(std::move(s));
            }
            // Order may carry the statement's OFFSET / LIMIT as a hint (plan/order.go:68-73); the Offset and Limit
            // operators that follow still apply them, so the hint is not needed here
            order = std::move(fresh);
        } else if (name == "Offset") {
            if (!has_project || has_offset || has_limit) return false;
            ExprP e = parse_expr(op.str_or("expr", ""));
            if (!integral_operand(*e, &offset)) return false;
            has_offset = true;
        } else if (name == "Limit") {
            if (!has_project || has_limit) return false;
            ExprP e = parse_expr(op.str_or("expr", ""));
            if (!integral_operand(*e, &limit)) return false;
            has_limit = true;
        } else return false;
    } catch (const Error& err) {
        if (err.code == N1GPU_E_INELIGIBLE || err.code == N1GPU_E_PARSE) return false;
        throw;
    }
    operators.push_back(name);
    return true;
}

std::string GroupTail::Run(const Result& r, i64* rows_out) const {
    // Three phases, so that a million groups cost what HAVING, the sort keys and the surviving rows cost - not a
    // projected object per group: (A) per group: LETTING, HAVING, the explicitly aliased terms ORDER BY may name and the
    // sort keys (all host cores for large results); (B) ORDER BY / OFFSET / LIMIT over group indices (a partial sort when
    // LIMIT bounds the output); (C) the projection of the rows that are left, as JSON.
    std::vector<std::string> alias_names;
    std::vector<int> alias_term;  // the LAST term carrying each explicit alias: later terms override (project_initial.go:104-111)
    for (size_t t = 0; t < terms.size(); ++t) {
        if (terms[t].as.empty()) continue;
        const int i = index_of(alias_names, terms[t].as);
        if (i < 0) { alias_names.push_back(terms[t].as); alias_term.push_back((int)t); } else alias_term[(size_t)i] = (int)t;
    }
    const size_t nsort = order.size();
    struct Part { std::vector<i64> g; std::vector<HValue> keys; };  // surviving groups and their nsort sort keys each
    auto eval_lets = [&](Env& env, std::vector<HValue>& lets) {
        lets.clear();
        for (auto& b : letting) lets.push_back(eval(*b.e, env));
        env.lets = &lets;
    };
    auto phase_a = [&](i64 g0, i64 g1, Part& out) {
        std::vector<HValue> lets, aliases(alias_names.size());
        for (i64 g = g0; g < g1; ++g) {
            Env env;
            env.r = &r;
            env.g = g;
            eval_lets(env, lets);
            if (having_e && !truth(eval(*having_e, env))) continue;  // filter.go:49-61
            out.g.push_back(g);
            if (nsort) {
                for (size_t i = 0; i < alias_term.size(); ++i) aliases[i] = eval(*terms[(size_t)alias_term[i]].e, env);
                env.aliases = &aliases;
                for (auto& s : order) out.keys.push_back(eval(*s.e, env));
            }
        }
    };
    auto in_threads = [&](i64 n, const std::function<void(int, i64, i64)>& fn) -> int {
        const int nthr = n < 65536 ? 1 : (int)std::min<i64>(std::max(1u, std::thread::hardware_concurrency()), 32);
        if (nthr <= 1) { fn(0, 0, n); return 1; }
        std::vector<std::string> errs((size_t)nthr);
        std::vector<std::thread> pool;
        for (int t = 0; t < nthr; ++t)
            pool.emplace_back([&, t] { try { fn(t, n * t / nthr, n * (t + 1) / nthr); } catch (const std::exception& e) { errs[(size_t)t] = e.what(); } });
        for (auto& th : pool) th.join();
        for (auto& e : errs) if (!e.empty()) N1_THROW(N1GPU_E_INVALID, "%s", e.c_str());
        return nthr;
    };
    const bool trace = getenv("N1GPU_TRACE") != nullptr;
    double tp = now_sec();
    auto phase = [&](const char* name) { if (trace) { const double t = now_sec(); fprintf(stderr, "[n1gpu tail] %-28s %8.3f ms\n", name, (t - tp) * 1e3); tp = t; } };
    // survivors stay in the per-thread parts (no merge copy): a survivor is (part << 40 | index in part), which is also
    // its position in group order
    std::vector<Part> parts(32);
    const int nparts = in_threads(r.ngroups, [&](int t, i64 g0, i64 g1) {
        const size_t room = std::min<size_t>((size_t)(g1 - g0), having_e ? (size_t)1 << 16 : (size_t)1 << 22);  // HAVING usually drops most
        parts[(size_t)t].g.reserve(room);
        parts[(size_t)t].keys.reserve(room * nsort);
        phase_a(g0, g1, parts[(size_t)t]);
    });
    phase("LETTING / HAVING / sort keys");
    size_t nsurv = 0;
    for (int t = 0; t < nparts; ++t) nsurv += parts[(size_t)t].g.size();
    size_t first = 0, last = nsurv;
    if (has_offset && offset > 0) first = (size_t)std::min<i64>(offset, (i64)nsurv);  // offset.go:75-83
    if (has_limit) last = std::min(last, first + (size_t)std::max<i64>(limit, 0));   // limit.go:74-81
    std::vector<u64> idx;
    idx.reserve(nsurv);
    for (int t = 0; t < nparts; ++t)
        for (size_t j = 0; j < parts[(size_t)t].g.size(); ++j) idx.push_back(((u64)t << 40) | (u64)j);
    const u64 JMASK = ((u64)1 << 40) - 1;
    if (nsort) {
        // order.go:119-166: Collate per term, descending flips it.  The reference's sort.Sort leaves ties in no particular
        // order; here they keep group order (the survivor id is the last sort key), which also makes a partial sort exact.
        const HValue* kbase[32];
        for (int t = 0; t < 32; ++t) kbase[t] = parts[(size_t)t].keys.data();
        auto less = [&](u64 a, u64 b) {
            const HValue* ka = kbase[a >> 40] + (size_t)(a & JMASK) * nsort;
            const HValue* kb = kbase[b >> 40] + (size_t)(b & JMASK) * nsort;
            for (size_t i = 0; i < nsort; ++i) {
                const int c = collate_values(ka[i], kb[i]);
                if (c == 0) continue;
                return order[i].desc ? c > 0 : c < 0;
            }
            return a < b;
        };
        if (last < nsurv) std::partial_sort(idx.begin(), idx.begin() + (std::ptrdiff_t)last, idx.end(), less);
        else std::sort(idx.begin(), idx.end(), less);
    }
    phase("ORDER BY / OFFSET / LIMIT");
    auto render = [&](i64 i0, i64 i1, std::string& s) {
        std::vector<HValue> lets;
        std::vector<std::pair<const std::string*, HValue>> fields;  // the "projection" attachment of one row
        for (i64 i = i0; i < i1; ++i) {
            Env env;
            env.r = &r;
            const u64 id = idx[first + (size_t)i];
            env.g = parts[(size_t)(id >> 40)].g[(size_t)(id & JMASK)];
            eval_lets(env, lets);
            fields.clear();
            for (auto& t : terms) {  // project_initial.go:98-117; a MISSING value unsets the field (value/object.go:246-255)
                HValue v = eval(*t.e, env);
                size_t at = 0;
                while (at < fields.size() && *fields[at].first != t.alias) ++at;
                if (v.cls == C_MISSING) { if (at < fields.size()) fields.erase(fields.begin() + (std::ptrdiff_t)at); continue; }
                if (at < fields.size()) fields[at].second = std::move(v); else fields.emplace_back(&t.alias, std::move(v));
            }
            std::sort(fields.begin(), fields.end(), [](const auto& a, const auto& b) { return *a.first < *b.first; });  // Go marshals maps by sorted name
            s += i == 0 ? "{" : ",{";
            for (size_t f = 0; f < fields.size(); ++f) {
                if (f) s += ",";
                json::quote(*fields[f].first, s);
                s += ":";
                s += value_to_json(fields[f].second);
            }
            s += "}";
        }
    };
    std::string s = "[";
    {
        std::vector<std::string> chunks(32);
        const int used = in_threads((i64)(last - first), [&](int t, i64 i0, i64 i1) { render(i0, i1, chunks[(size_t)t]); });
        for (int t = 0; t < used; ++t) s += chunks[(size_t)t];
    }
    phase("projection + JSON");
    if (rows_out) *rows_out = (i64)(last - first);
    return s + "]";
}

}  // namespace execution
}  // namespace n1
