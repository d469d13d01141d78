// expr.cpp — Stringer-text parser, binder and static type analysis for the eligible expression subset.
#include "expr.hpp"

#include <cmath>

#include <algorithm>
#include <charconv>
#include <cstring>

#include "json.hpp"
#include "table.hpp"

namespace n1 {

// ---- Stringer ----------------------------------------------------------------------------------------
static std::string const_text(const HValue& v) {
    switch (v.cls) {
        case C_MISSING: return "missing";
        case C_NULL: return "null";
        case C_FALSE: return "false";
        case C_TRUE: return "true";
        case C_INT: return std::to_string(v.bits);
        case C_FLOAT: return json::format_float(v.f());
        default: { std::string s; json::quote(v.s, s); return s; }
    }
}

static std::string nary(const Expr& e, const char* sym) {
    std::string s = "(";
    for (size_t i = 0; i < e.ops.size(); ++i) { if (i) { s += " "; s += sym; s += " "; } s += e.ops[i]->str(); }
    return s + ")";
}

std::string Expr::str() const {
    switch (kind) {
        case EK::CONST: return param.empty() ? const_text(cval) : "$" + param;
        case EK::PARAM: return "$" + name;
        case EK::IDENT: return "`" + name + "`";
        case EK::FIELD: return "(" + ops[0]->str() + ".`" + name + "`)";
        case EK::ADD: return nary(*this, "+");
        case EK::MULT: return nary(*this, "*");
        case EK::SUB: return nary(*this, "-");
        case EK::DIV: return nary(*this, "/");
        case EK::MOD: return nary(*this, "%");
        case EK::NEG: return "(-" + ops[0]->str() + ")";
        case EK::EQ: return nary(*this, "=");
        case EK::LT: return nary(*this, "<");
        case EK::LE: return nary(*this, "<=");
        case EK::BETWEEN: return "(" + ops[0]->str() + " between " + ops[1]->str() + " and " + ops[2]->str() + ")";
        case EK::IN: return nary(*this, "in");
        case EK::AND: return nary(*this, "and");
        case EK::OR: return nary(*this, "or");
        case EK::NOT: return "(not " + ops[0]->str() + ")";
        case EK::IS_NULL: return "(" + ops[0]->str() + " is null)";
        case EK::IS_NOT_NULL: return "(" + ops[0]->str() + " is not null)";
        case EK::IS_MISSING: return "(" + ops[0]->str() + " is missing)";
        case EK::IS_NOT_MISSING: return "(" + ops[0]->str() + " is not missing)";
        case EK::IS_VALUED: return "(" + ops[0]->str() + " is valued)";
        case EK::IS_NOT_VALUED: return "(" + ops[0]->str() + " is not valued)";
        case EK::ARRAY: {
            if (!param.empty()) return "$" + param;
            std::string s = "[";
            for (size_t i = 0; i < ops.size(); ++i) { if (i) s += ", "; s += ops[i]->str(); }
            return s + "]";
        }
        case EK::AGG: {
            static const char* names[] = {"count", "countn", "sum", "avg", "min", "max"};
            std::string s = names[(int)agg];
            s += "(";
            if (distinct) s += "distinct ";
            s += star ? "*" : ops[0]->str();
            return s + ")";
        }
        case EK::ROUND: return "round(" + ops[0]->str() + (ops.size() > 1 ? ", " + ops[1]->str() : std::string()) + ")";  // stringer.go:581-604
    }
    return "?";
}

// ---- parser --------------------------------------------------------------------------------------------
namespace {
struct P {
    const std::string& s;
    size_t i = 0;
    explicit P(const std::string& t) : s(t) {}

    [[noreturn]] void bad(const char* what) { N1_THROW(N1GPU_E_PARSE, "%s at offset %zu in expression: %s", what, i, s.c_str()); }
    [[noreturn]] void inel(const std::string& what) { N1_THROW(N1GPU_E_INELIGIBLE, "%s (in %s)", what.c_str(), s.c_str()); }
    void ws() { while (i < s.size() && (s[i] == ' ' || s[i] == '\t' || s[i] == '\n')) ++i; }
    char peek() { ws(); return i < s.size() ? s[i] : '\0'; }
    bool eat(const char* tok) {
        ws();
        size_t n = strlen(tok);
        if (s.compare(i, n, tok) == 0) { i += n; return true; }
        return false;
    }
    void expect(const char* tok) { if (!eat(tok)) bad((std::string("expected '") + tok + "'").c_str()); }
    std::string word() {
        ws();
        size_t j = i;
        while (j < s.size() && (isalnum((unsigned char)s[j]) || s[j] == '_')) ++j;
        std::string w = s.substr(i, j - i);
        for (auto& c : w) c = (char)tolower((unsigned char)c);
        return w;
    }
    bool eat_word(const char* w) {
        if (word() == w) { i += strlen(w); return true; }
        return false;
    }
    std::string backtick() {
        expect("`");
        size_t j = s.find('`', i);
        if (j == std::string::npos) bad("unterminated identifier");
        std::string name = s.substr(i, j - i);
        i = j + 1;
        if (i < s.size() && s[i] == 'i' && !(i + 1 < s.size() && (isalnum((unsigned char)s[i + 1]) || s[i + 1] == '_' || s[i + 1] == '`')))
            inel("case-insensitive identifier");
        return name;
    }

    ExprP mk(EK k) { return ExprP(new Expr(k)); }

    ExprP expr() {
        char c = peek();
        if (c == '(') {
            ++i;
            ExprP e = inner();
            expect(")");
            return e;
        }
        if (c == '`') { ExprP e = mk(EK::IDENT); e->name = backtick(); return e; }
        if (c == '[') {
            ++i;
            ExprP a = mk(EK::ARRAY);
            if (!eat("]")) {
                for (;;) {
                    a->ops.push_back(expr());
                    if (eat("]")) break;
                    expect(",");
                }
            }
            return a;
        }
        if (c == '"') {
            json::Scanner sc(s.data() + i, s.data() + s.size());
            const char *rb, *re; bool esc;
            if (!sc.string_raw(rb, re, esc)) bad("bad string literal");
            ExprP e = mk(EK::CONST);
            e->cval.cls = C_STRING;
            if (esc) json::Scanner::unescape(rb, re, e->cval.s); else e->cval.s.assign(rb, re);
            i = (size_t)(sc.p - s.data());
            return e;
        }
        if (isdigit((unsigned char)c) || (c == '-' && i + 1 < s.size() && isdigit((unsigned char)s[i + 1]))) {
            json::Scanner sc(s.data() + i, s.data() + s.size());
            bool ii; i64 iv; double dv;
            if (!sc.number(ii, iv, dv)) bad("bad number literal");
            i = (size_t)(sc.p - s.data());
            ExprP e = mk(EK::CONST);
            e->cval = ii ? HValue::integer(iv) : new_num(dv);  // value.NewValue canonicalisation
            return e;
        }
        if (c == '{') inel("object construction");
        if (c == '$') {  // named / positional parameter: bound to a constant before analysis (bind_params)
            ++i;
            size_t j = i;
            while (j < s.size() && (isalnum((unsigned char)s[j]) || s[j] == '_')) ++j;
            if (j == i) bad("parameter name expected after '$'");
            ExprP e = mk(EK::PARAM);
            e->name = s.substr(i, j - i);
            i = j;
            return e;
        }
        std::string w = word();
        if (w.empty()) bad("unexpected character");
        i += w.size();
        if (w == "true") { ExprP e = mk(EK::CONST); e->cval = HValue::boolean(true); return e; }
        if (w == "false") { ExprP e = mk(EK::CONST); e->cval = HValue::boolean(false); return e; }
        if (w == "null") { ExprP e = mk(EK::CONST); e->cval = HValue::null(); return e; }
        if (w == "missing") { ExprP e = mk(EK::CONST); e->cval = HValue::missing(); return e; }
        if (eat("(")) {
            static const char* names[] = {"count", "countn", "sum", "avg", "min", "max"};
            int which = -1;
            for (int k = 0; k < 6; ++k) if (w == names[k]) which = k;
            if (w == "round") {  // the one scalar function the reference's aggregate goldens use (ROUND(AVG(x), 5))
                ExprP r = mk(EK::ROUND);
                r->ops.push_back(expr());
                if (eat(",")) r->ops.push_back(expr());
                expect(")");
                return r;
            }
            if (which < 0) inel("function " + w + "() is not on the GPU path");
            ExprP a = mk(EK::AGG);
            a->agg = (AggKind)which;
            if (eat_word("distinct")) a->distinct = true;
            if (eat("*")) {
                if (a->agg != AggKind::COUNT || a->distinct) inel(w + "(*)");
                a->star = true;
            } else a->ops.push_back(expr());
            if (peek() == ',') inel("multi-argument aggregate");
            expect(")");
            if (a->distinct && (a->agg == AggKind::MIN || a->agg == AggKind::MAX)) inel("MIN/MAX DISTINCT (n1ql.y:2756-2764)");
            return a;
        }
        inel("construct '" + w + "' is not on the GPU path");
    }

    ExprP unary(EK k, ExprP a) { ExprP e = mk(k); e->ops.push_back(std::move(a)); return e; }
    ExprP binary(EK k, ExprP a, ExprP b) { ExprP e = mk(k); e->ops.push_back(std::move(a)); e->ops.push_back(std::move(b)); return e; }

    ExprP inner() {
        ws();
        if (peek() == '-' && !(i + 1 < s.size() && isdigit((unsigned char)s[i + 1]))) { ++i; return unary(EK::NEG, expr()); }
        if (word() == "not") { i += 3; return unary(EK::NOT, expr()); }
        {
            std::string w = word();
            if (w == "case" || w == "any" || w == "every" || w == "array" || w == "first" || w == "object" || w == "exists" ||
                w == "distinct" || w == "all" || w == "select" || w == "correlated")
                inel("construct '" + w + "' is not on the GPU path");
        }
        ExprP first = expr();
        if (peek() == ')') return first;
        if (peek() == '.') {
            ++i;
            if (peek() == '[') inel("computed field name");
            ExprP f = mk(EK::FIELD);
            f->name = backtick();
            f->ops.push_back(std::move(first));
            return f;
        }
        if (peek() == '[') inel("array element / slice navigation");
        std::vector<ExprP> ops;
        ops.push_back(std::move(first));
        std::string sym;
        while (peek() != ')') {
            if (i >= s.size()) bad("unterminated expression");
            std::string t;
            static const char* syms[] = {"<=", ">=", "!=", "<>", "==", "=", "<", ">", "+", "-", "*", "/", "%", "||"};
            for (const char* c : syms) if (eat(c)) { t = c; break; }
            if (t.empty()) {
                std::string w = word();
                if (w == "and" || w == "or" || w == "in" || w == "between" || w == "is") { i += w.size(); t = w; }
                else if (w == "not") {
                    i += 3;
                    if (eat_word("between")) t = "not between";
                    else if (eat_word("in")) t = "not in";
                    else if (eat_word("like")) inel("LIKE");
                    else if (eat_word("within")) inel("WITHIN");
                    else bad("unexpected NOT");
                } else if (w == "like" || w == "within") inel(w);
                else bad("operator expected");
            }
            if (t == "||") inel("string concatenation");
            if (t == "is") {
                bool neg = eat_word("not");
                std::string what = word();
                i += what.size();
                EK k;
                if (what == "null") k = neg ? EK::IS_NOT_NULL : EK::IS_NULL;
                else if (what == "missing") k = neg ? EK::IS_NOT_MISSING : EK::IS_MISSING;
                else if (what == "valued") k = neg ? EK::IS_NOT_VALUED : EK::IS_VALUED;
                else bad("IS what?");
                if (ops.size() != 1) bad("IS after operator");
                return unary(k, std::move(ops[0]));
            }
            if (t == "between" || t == "not between") {
                if (ops.size() != 1) bad("BETWEEN after operator");
                ExprP b = mk(EK::BETWEEN);
                b->ops.push_back(std::move(ops[0]));
                b->ops.push_back(expr());
                if (!eat_word("and")) bad("BETWEEN without AND");
                b->ops.push_back(expr());
                return t == "between" ? std::move(b) : unary(EK::NOT, std::move(b));
            }
            if (!sym.empty() && t != sym) bad("mixed operators in one parenthesis");
            sym = t;
            ops.push_back(expr());
        }
        auto make_nary = [&](EK k) { ExprP e = mk(k); e->ops = std::move(ops); return e; };
        if (sym == "+") return make_nary(EK::ADD);
        if (sym == "*") return make_nary(EK::MULT);
        if (sym == "and") return make_nary(EK::AND);
        if (sym == "or") return make_nary(EK::OR);
        if (ops.size() != 2) bad("binary operator with more than two operands");
        ExprP a = std::move(ops[0]), b = std::move(ops[1]);
        if (sym == "=" || sym == "==") return binary(EK::EQ, std::move(a), std::move(b));
        if (sym == "!=" || sym == "<>") return unary(EK::NOT, binary(EK::EQ, std::move(a), std::move(b)));
        if (sym == "<") return binary(EK::LT, std::move(a), std::move(b));
        if (sym == "<=") return binary(EK::LE, std::move(a), std::move(b));
        if (sym == ">") return binary(EK::LT, std::move(b), std::move(a));
        if (sym == ">=") return binary(EK::LE, std::move(b), std::move(a));
        if (sym == "-") return binary(EK::SUB, std::move(a), std::move(b));
        if (sym == "/") return binary(EK::DIV, std::move(a), std::move(b));
        if (sym == "%") return binary(EK::MOD, std::move(a), std::move(b));
        if (sym == "in") return binary(EK::IN, std::move(a), std::move(b));
        if (sym == "not in") return unary(EK::NOT, binary(EK::IN, std::move(a), std::move(b)));
        bad("unknown operator");
    }
};
}  // namespace

ExprP parse_expr(const std::string& text) {
    P p(text);
    ExprP e = p.expr();
    p.ws();
    if (p.i != text.size()) p.bad("trailing text");
    return e;
}

// ---- binding ---------------------------------------------------------------------------------------------
static bool field_chain(const Expr& e, const std::string& alias, std::vector<std::string>& path) {
    if (e.kind == EK::IDENT) return e.name == alias;
    if (e.kind != EK::FIELD) return false;
    if (!field_chain(*e.ops[0], alias, path)) return false;
    path.push_back(e.name);
    return true;
}

void collect_paths(const Expr& e, const std::string& alias, std::vector<std::string>& out) {
    if (e.kind == EK::FIELD) {
        std::vector<std::string> path;
        if (!field_chain(e, alias, path))
            N1_THROW(N1GPU_E_INELIGIBLE, "navigation %s is not a field path below `%s`", e.str().c_str(), alias.c_str());
        std::string joined = join_path(path, '\x1f');
        if (std::find(out.begin(), out.end(), joined) == out.end()) out.push_back(joined);
        return;
    }
    if (e.kind == EK::IDENT)
        N1_THROW(N1GPU_E_INELIGIBLE, "bare identifier %s (whole-document or foreign reference)", e.str().c_str());
    for (auto& o : e.ops) collect_paths(*o, alias, out);
}

static bool add_fits(__int128 v) { return v >= (__int128)INT64_MIN && v <= (__int128)INT64_MAX; }

static u32 nonnum_bits(u32 m) { return m & (bit(C_NULL) | M_BOOL | bit(C_STRING)); }

void bind_params(Expr& e, const std::vector<ParamValue>& params) {
    if (e.kind == EK::PARAM) {
        for (auto& pv : params) {
            if (pv.name != e.name) continue;
            e.param = e.name;
            if (!pv.is_array) { e.kind = EK::CONST; e.cval = pv.value; return; }
            e.kind = EK::ARRAY;
            for (auto& v : pv.elems) { ExprP c(new Expr(EK::CONST)); c->cval = v; e.ops.push_back(std::move(c)); }
            return;
        }
        N1_THROW(N1GPU_E_INVALID, "No value for %s parameter $%s.", isdigit((unsigned char)e.name[0]) ? "positional" : "named", e.name.c_str());
    }
    for (auto& o : e.ops) bind_params(*o, params);
}

static HValue scalar_param(json::Scanner& sc, const std::string& text) {
    HValue v;
    const char c = sc.p < sc.end ? *sc.p : '\0';
    if (c == '"') {
        const char *rb, *re; bool esc;
        if (!sc.string_raw(rb, re, esc)) N1_THROW(N1GPU_E_PARSE, "bad string parameter value");
        v.cls = C_STRING;
        if (esc) json::Scanner::unescape(rb, re, v.s); else v.s.assign(rb, re);
    } else if (c == '-' || isdigit((unsigned char)c)) {
        bool ii; i64 iv; double dv;
        if (!sc.number(ii, iv, dv)) N1_THROW(N1GPU_E_PARSE, "bad number parameter value");
        v = ii ? HValue::integer(iv) : new_num(dv);  // value.NewValue canonicalisation, as for literals
    } else {
        auto word = [&](const char* w, size_t n) { return (size_t)(sc.end - sc.p) >= n && memcmp(sc.p, w, n) == 0; };
        if (word("true", 4)) { v = HValue::boolean(true); sc.p += 4; }
        else if (word("false", 5)) { v = HValue::boolean(false); sc.p += 5; }
        else if (word("null", 4)) { v = HValue::null(); sc.p += 4; }
        else N1_THROW(N1GPU_E_INELIGIBLE, "parameter value %s is not a scalar or an array of scalars (nested arrays / objects stay on the Go operators)", text.c_str());
    }
    return v;
}

ParamValue parse_param_value(const std::string& text) {
    json::Scanner sc(text.data(), text.data() + text.size());
    sc.ws();
    if (sc.p >= sc.end) N1_THROW(N1GPU_E_INVALID, "empty parameter value");
    ParamValue pv;
    if (*sc.p == '[') {
        pv.is_array = true;
        ++sc.p;
        sc.ws();
        if (sc.p < sc.end && *sc.p == ']') ++sc.p;
        else for (;;) {
            sc.ws();
            pv.elems.push_back(scalar_param(sc, text));
            sc.ws();
            if (sc.p < sc.end && *sc.p == ',') { ++sc.p; continue; }
            if (sc.p < sc.end && *sc.p == ']') { ++sc.p; break; }
            N1_THROW(N1GPU_E_PARSE, "bad array parameter value %s", text.c_str());
        }
    } else pv.value = scalar_param(sc, text);
    sc.ws();
    if (sc.p != sc.end) N1_THROW(N1GPU_E_PARSE, "trailing characters in parameter value %s", text.c_str());
    return pv;
}

bool in_takes_set(const Expr& in) {
    const Expr& list = *in.ops[1];
    if (!list.param.empty()) return true;  // array parameter: an operand that is a string constant is refused in codegen
    if (list.ops.size() <= IN_CHAIN_MAX) return false;
    for (auto& el : list.ops) if (el->kind != EK::CONST) return false;
    const TypeInfo& x = in.ops[0]->ti;
    return !(x.mask & bit(C_STRING)) || x.plain_col;
}

void bind_and_analyze(Expr& e, const std::string& alias, const Table& t) {
    TypeInfo& ti = e.ti;
    if (e.kind == EK::FIELD) {
        std::vector<std::string> path;
        if (!field_chain(e, alias, path)) N1_THROW(N1GPU_E_INELIGIBLE, "navigation %s is not a field path", e.str().c_str());
        int c = t.find_column(join_path(path, '\x1f'));
        if (c < 0) N1_THROW(N1GPU_E_INVALID, "column %s was not shredded", join_path(path, '.').c_str());
        const ColumnStats& st = t.cols[c].stats;
        if (st.class_mask & bit(C_OTHER))
            N1_THROW(N1GPU_E_INELIGIBLE, "column %s holds arrays/objects: plan stays on the Go operators", join_path(path, '.').c_str());
        e.col = c;
        ti.mask = st.class_mask ? st.class_mask : bit(C_MISSING);
        ti.plain_col = true;
        if (st.has_int) { ti.ranged = true; ti.lo = st.int_min; ti.hi = st.int_max; }
        ti.imax = !(ti.mask & bit(C_INT)) ? 0.0 : (st.has_int ? std::max(std::fabs((double)st.int_min), std::fabs((double)st.int_max)) : 1e300);
        if (ti.mask & bit(C_STRING)) ti.dict_col = c;
        return;
    }
    if (e.kind == EK::IDENT) N1_THROW(N1GPU_E_INELIGIBLE, "bare identifier %s", e.str().c_str());
    if (e.kind == EK::PARAM) N1_THROW(N1GPU_E_INVALID, "No value for parameter $%s.", e.name.c_str());
    for (size_t i = 0; i < e.ops.size(); ++i) {
        if (e.ops[i]->kind == EK::ARRAY && !(e.kind == EK::IN && i == 1))
            N1_THROW(N1GPU_E_INELIGIBLE, "array value outside the right operand of IN: %s", e.ops[i]->str().c_str());
        bind_and_analyze(*e.ops[i], alias, t);
    }
    auto any_has = [&](u32 bits) { for (auto& o : e.ops) if (o->ti.mask & bits) return true; return false; };
    auto string_dict = [&]() {  // the one dictionary string operands of a comparison live in
        int d = -1;
        for (auto& o : e.ops) {
            const Expr* x = o.get();
            std::vector<const Expr*> flat;
            if (x->kind == EK::ARRAY) for (auto& el : x->ops) flat.push_back(el.get()); else flat.push_back(x);
            for (const Expr* y : flat) {
                if (!(y->ti.mask & bit(C_STRING))) continue;
                if (y->kind == EK::CONST) continue;
                if (!y->ti.plain_col) N1_THROW(N1GPU_E_INELIGIBLE, "computed string operand %s", y->str().c_str());
                if (d >= 0 && d != y->ti.dict_col)
                    N1_THROW(N1GPU_E_INELIGIBLE, "comparison across two string dictionaries: %s", e.str().c_str());
                d = y->ti.dict_col;
            }
        }
        return d;
    };
    switch (e.kind) {
        case EK::CONST:
            ti.mask = bit(e.cval.cls);
            if (e.cval.cls == C_INT) { ti.ranged = true; ti.lo = ti.hi = e.cval.bits; }
            ti.imax = e.cval.cls == C_INT ? std::fabs((double)e.cval.bits) : 0.0;
            break;
        case EK::ARRAY:
            ti.mask = 0;  // only meaningful as the right side of IN
            break;
        case EK::ADD: case EK::MULT: case EK::SUB: case EK::NEG: case EK::DIV: case EK::MOD: {
            bool all_num_possible = true, all_int_only = true, any_float_only = false, all_ranged = true;
            for (auto& o : e.ops) {
                u32 nm = o->ti.mask & M_NUM;
                if (!nm) all_num_possible = false;
                if (nm != bit(C_INT)) all_int_only = false;
                if (nm == bit(C_FLOAT)) any_float_only = true;
                if (!o->ti.ranged) all_ranged = false;
                if (o->ti.mask & bit(C_STRING) && o->kind != EK::CONST && !o->ti.plain_col)
                    N1_THROW(N1GPU_E_INELIGIBLE, "computed string operand");
            }
            u32 m = 0;
            if (any_has(bit(C_MISSING))) m |= bit(C_MISSING);
            bool may_null = false;
            for (auto& o : e.ops) if (nonnum_bits(o->ti.mask)) may_null = true;
            if (e.kind == EK::DIV || e.kind == EK::MOD) {
                const Expr& dv = *e.ops[1];
                bool nonzero_const = dv.kind == EK::CONST && ((dv.cval.cls == C_INT && dv.cval.bits != 0) || (dv.cval.cls == C_FLOAT && dv.cval.f() != 0.0));
                if (!nonzero_const) may_null = true;
            }
            if (may_null) m |= bit(C_NULL);
            if (all_num_possible) {
                if (e.kind == EK::DIV || e.kind == EK::MOD) m |= M_NUM;
                else if (any_float_only) m |= bit(C_FLOAT);
                else if (all_int_only && all_ranged) {
                    // interval arithmetic following intValue.Add/Mult/Neg/Sub (value/integer.go:266-348)
                    bool int_only = true;
                    __int128 lo = 0, hi = 0;
                    if (e.kind == EK::ADD) {
                        lo = hi = 0;
                        for (auto& o : e.ops) {
                            __int128 xl = o->ti.lo, xh = o->ti.hi;
                            bool nn = lo >= 0 && xl >= 0 && add_fits(hi + xh);
                            bool ng = hi < 0 && xh < 0 && add_fits(lo + xl);
                            if (!(nn || ng)) { int_only = false; break; }
                            lo += xl; hi += xh;
                        }
                    } else if (e.kind == EK::MULT) {
                        lo = hi = 1;
                        for (auto& o : e.ops) {
                            __int128 c[4] = {lo * o->ti.lo, lo * o->ti.hi, hi * o->ti.lo, hi * o->ti.hi};
                            __int128 nl = c[0], nh = c[0];
                            for (auto v : c) { nl = std::min(nl, v); nh = std::max(nh, v); }
                            if (!add_fits(nl) || !add_fits(nh)) { int_only = false; break; }
                            lo = nl; hi = nh;
                        }
                    } else if (e.kind == EK::NEG) {
                        if (e.ops[0]->ti.lo == INT64_MIN) int_only = false;
                        else { lo = -(__int128)e.ops[0]->ti.hi; hi = -(__int128)e.ops[0]->ti.lo; }
                    } else {  // SUB
                        __int128 al = e.ops[0]->ti.lo, ah = e.ops[0]->ti.hi, bl = e.ops[1]->ti.lo, bh = e.ops[1]->ti.hi;
                        bool nn = al >= 0 && bh <= 0 && add_fits(ah - bl) && bl > (__int128)INT64_MIN;
                        bool ng = ah < 0 && bl > 0 && add_fits(al - bh);
                        if (!(nn || ng)) int_only = false;
                        lo = al - bh; hi = ah - bl;
                    }
                    if (int_only) { m |= bit(C_INT); ti.ranged = true; ti.lo = (i64)lo; ti.hi = (i64)hi; }
                    else m |= M_NUM;
                } else m |= M_NUM;
            }
            ti.mask = m;
            // magnitude bound of INT results.  + - * neg yield an INT only from INT operands (a float operand makes a
            // floatValue, integral or not: value/float.go:331-381), so interval arithmetic over the operands' INT bounds
            // holds; / and % canonicalise integral quotients to INT (arith_div.go:46-64) - no bound there.
            if (!(m & bit(C_INT))) ti.imax = 0.0;
            else if (e.kind == EK::DIV || e.kind == EK::MOD) ti.imax = 1e300;
            else {
                double b = e.kind == EK::MULT ? 1.0 : 0.0;
                for (auto& o : e.ops) b = e.kind == EK::MULT ? b * o->ti.imax : b + o->ti.imax;
                ti.imax = std::min(b, 1e300);
            }
            break;
        }
        case EK::EQ: case EK::LT: case EK::LE: case EK::BETWEEN: {
            u32 m = M_BOOL;
            if (any_has(bit(C_MISSING))) m |= bit(C_MISSING);
            if (any_has(bit(C_NULL))) m |= bit(C_NULL);
            ti.mask = m;
            ti.dict_col = string_dict();
            break;
        }
        case EK::IN: {
            if (e.ops[1]->kind != EK::ARRAY) N1_THROW(N1GPU_E_INELIGIBLE, "IN over a non-array: %s", e.str().c_str());
            u32 m = M_BOOL;
            u32 all = e.ops[0]->ti.mask;
            // a set: NULL whatever the elements (a NULL row, or a NULL element), MISSING when a literal list may hold one
            if (in_takes_set(e)) all |= bit(C_NULL) | (e.ops[1]->param.empty() ? bit(C_MISSING) : 0);
            else for (auto& el : e.ops[1]->ops) all |= el->ti.mask;
            if (all & bit(C_MISSING)) m |= bit(C_MISSING);
            if (all & bit(C_NULL)) m |= bit(C_NULL);
            ti.mask = m;
            ti.dict_col = string_dict();
            break;
        }
        case EK::AND: case EK::OR: {
            u32 m = M_BOOL;
            if (any_has(bit(C_MISSING))) m |= bit(C_MISSING);
            if (any_has(bit(C_NULL))) m |= bit(C_NULL);
            ti.mask = m;
            break;
        }
        case EK::NOT:
            ti.mask = (e.ops[0]->ti.mask & (bit(C_MISSING) | bit(C_NULL))) | M_BOOL;
            break;
        case EK::IS_NULL: case EK::IS_NOT_NULL:
            ti.mask = M_BOOL | (e.ops[0]->ti.mask & bit(C_MISSING));
            break;
        case EK::IS_MISSING: case EK::IS_NOT_MISSING: case EK::IS_VALUED: case EK::IS_NOT_VALUED:
            ti.mask = M_BOOL;
            break;
        case EK::AGG:
            ti.mask = 0;
            break;
        case EK::ROUND: N1_THROW(N1GPU_E_INELIGIBLE, "round() is evaluated over groups only, not on the GPU path");
        default: break;
    }
}

}  // namespace n1
