// expr.hpp — host-side mirror of the reference's `expression` / `algebra` node types for the eligible
// subset (SURVEY.md 8a rows a4-a7, a12-a17), parsed from the Stringer text that plan JSON carries.
//
//   expression/stringer.go (text form)        expression/comp_gt.go:15-17 (a > b is LT(b, a))
//   expression/comp_eq.go:92-94 (a != b is NOT(a = b))     algebra/agg_registry.go:41-62
#pragma once
#include <memory>
#include <string>
#include <vector>

#include "common.hpp"

namespace n1 {

struct Table;

enum class EK {
    CONST, IDENT, FIELD,  // navigation
    PARAM,                // $name / $1 (algebra/param_named.go:63, param_positional.go; expression/stringer.go:611-620)
    ADD, MULT, SUB, DIV, MOD, NEG,
    EQ, LT, LE, BETWEEN, IN,
    AND, OR, NOT,
    IS_NULL, IS_NOT_NULL, IS_MISSING, IS_NOT_MISSING, IS_VALUED, IS_NOT_VALUED,
    ARRAY,  // array construct (only as the right side of IN)
    AGG,    // aggregate call
    ROUND   // round(x [, digits]) - host only: the operators behind FinalGroup (group_tail.cpp); never reaches a kernel
};

struct TypeInfo {
    u32 mask = 0;          // classes the value may take
    bool ranged = false;   // INT values proven within [lo, hi]
    i64 lo = 0, hi = 0;
    double imax = 1e300;   // every INT value satisfies |x| <= imax (1e300: unknown); 0 when the value is never an INT
    int dict_col = -1;     // STRING values are ranks in this column's dictionary (-1: none / constant)
    bool plain_col = false;
};

struct Expr {
    EK kind;
    std::vector<std::unique_ptr<Expr>> ops;
    HValue cval;             // CONST
    std::string name;        // IDENT / FIELD name; PARAM: the name or position after '$'
    std::string param;       // CONST / ARRAY that stands for a bound parameter: its name (the Stringer text stays "$name")
    AggKind agg = AggKind::COUNT;
    bool distinct = false;
    bool star = false;       // count(*)
    // binding / analysis
    int col = -1;            // FIELD chain bound to a table column
    TypeInfo ti;

    explicit Expr(EK k) : kind(k) {}
    std::string str() const;  // Stringer text (expression/stringer.go)
};
typedef std::unique_ptr<Expr> ExprP;

// Parses Stringer text; throws Error(N1GPU_E_PARSE) on malformed text and Error(N1GPU_E_INELIGIBLE)
// on well-formed N1QL outside the subset (functions, CASE, ANY/EVERY, parameters, ...).
ExprP parse_expr(const std::string& text);

// Collects the field paths (joined with '\x1f') referenced below `alias`; throws INELIGIBLE for a bare
// alias reference (whole document), foreign identifiers or navigation on non-identifiers.
void collect_paths(const Expr& e, const std::string& alias, std::vector<std::string>& out);

// Replaces every PARAM by the constant bound to it (execution.Context.NamedArg / PositionalArg); a parameter without a
// value throws N1GPU_E_INVALID ("No value for named parameter $x", algebra/param_named.go:70-72).
// An array value binds to an ARRAY of constants, which is legal only as the right operand of IN (bind_and_analyze).
struct ParamValue {
    std::string name;
    HValue value;
    bool is_array = false;
    std::vector<HValue> elems;  // is_array: the elements
};
void bind_params(Expr& e, const std::vector<ParamValue>& params);
// a JSON scalar (number, string, true, false, null) as a constant, or a JSON array of such scalars; nested arrays and
// objects are outside the subset.  The name is left empty.
ParamValue parse_param_value(const std::string& json_text);

// `x IN list` is probed as a device-resident set, not unrolled into one in_arg per element, when the list is bound to an
// array parameter (whatever its length) or is a literal list of more than IN_CHAIN_MAX constants (DESIGN.md section 3.1);
// a string-capable operand must then be a dictionary column.  Needs the operand analysed.  For such an IN the analysis
// keeps the result's classes independent of the elements, so that the kernel text does not depend on them either.
constexpr size_t IN_CHAIN_MAX = 16;
bool in_takes_set(const Expr& in);

// Binds FIELD chains to columns of `t` and computes TypeInfo bottom-up.
void bind_and_analyze(Expr& e, const std::string& alias, const Table& t);

}  // namespace n1
