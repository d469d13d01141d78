"""Differential test of the host evaluator behind the operator's tail (query_b200/csrc/group_tail.cpp) against the
oracle (which is pinned to the reference's goldens): seeded random expression trees over group keys, aggregates and
constants - arithmetic with int64 overflow -> float64 promotion, collation across types, 4-valued logic, BETWEEN, IN,
IS [NOT] NULL / MISSING / VALUED, ROUND - evaluated over random groups whose values range over MISSING, NULL, booleans,
small and near-overflow ints, floats and strings.  Numbers and logic are the code of n1ql_value.cuh, which the scan
kernel runs too; the kernel itself is checked on the device by tests/test_gpu_parity.py."""
import json
import math
import random

import pytest

import query_b200 as q
from golden_plans import normalise
from oracle import n1ql_oracle as O
from plans_n1 import explain_plan
from util_n1 import write_keyspace

KEYS = ["(`d`.`k0`)", "(`d`.`k1`)"]
AGGS = sorted(["count(*)", "sum((`d`.`x`))", "min((`d`.`s`))", "max((`d`.`x`))"])
LEAVES = KEYS + AGGS

I63 = 2 ** 62


def rand_value(rng):
    r = rng.random()
    if r < 0.08:
        return O.MISSING
    if r < 0.16:
        return None
    if r < 0.22:
        return rng.random() < 0.5
    if r < 0.50:
        return rng.choice([0, 1, -1, 2, 3, 7, -5, 10, 100, rng.randint(-50, 50), rng.randint(-I63, I63), I63, -I63, 2 ** 53 + 1])
    if r < 0.75:
        return rng.choice([0.5, -0.5, 1.5, 2.5, 0.1, 3.25, -7.75, 1e6 + 0.5, rng.uniform(-100, 100), 1e15 + 0.5, 2.0 ** 63])
    return rng.choice(["", "a", "b", "abc", "Z", "é", "10", "a b"])


def const_text(rng):
    r = rng.random()
    if r < 0.35:
        return str(rng.choice([0, 1, 2, 3, -1, 5, 10, 2 ** 62, -(2 ** 62)]))
    if r < 0.55:
        return repr(rng.choice([0.5, 1.5, 2.5, -0.25, 100.125]))
    if r < 0.75:
        return json.dumps(rng.choice(["", "a", "abc", "b"]))
    return rng.choice(["true", "false", "null", "missing"])


def rand_expr(rng, depth):
    if depth <= 0 or rng.random() < 0.25:
        return rng.choice(LEAVES) if rng.random() < 0.7 else const_text(rng)
    sub = lambda: rand_expr(rng, depth - 1)
    kind = rng.choice(["+", "*", "-", "/", "%", "neg", "=", "<", "<=", "between", "in", "and", "or", "not", "is", "round"])
    if kind in ("+", "*", "and", "or"):
        return "(" + (" %s " % kind).join(sub() for _ in range(rng.choice([2, 2, 3]))) + ")"
    if kind in ("-", "/", "%", "=", "<", "<="):
        return "(%s %s %s)" % (sub(), kind, sub())
    if kind == "neg":
        return "(-%s)" % sub()
    if kind == "not":
        return "(not %s)" % sub()
    if kind == "between":
        return "(%s between %s and %s)" % (sub(), sub(), sub())
    if kind == "in":
        return "(%s in [%s])" % (sub(), ", ".join(sub() for _ in range(rng.choice([1, 2, 3]))))
    if kind == "is":
        return "(%s is %s%s)" % (sub(), rng.choice(["", "not "]), rng.choice(["null", "missing", "valued"]))
    return "round(%s%s)" % (sub(), rng.choice(["", ", 0", ", 1", ", 2", ", -1", ", %s" % sub()]))


def finite(rows):
    def ok(v):
        return not (isinstance(v, float) and (math.isnan(v) or math.isinf(v)))
    return all(ok(v) for r in rows for v in r.values())


@pytest.mark.parametrize("seed", range(40))
def test_random_expressions_over_random_groups(seed, tmp_path):
    rng = random.Random(1000 + seed)
    write_keyspace(str(tmp_path), "default", "d", [("k0", '{"k0": 1, "k1": "a", "x": 1, "s": "q"}')])
    groups = []
    for _ in range(40):
        ks = [rand_value(rng), rand_value(rng)]
        ag = {a: rand_value(rng) for a in AGGS}
        for a in AGGS:  # an aggregate is never MISSING (ComputeFinal yields NULL for "nothing")
            if ag[a] is O.MISSING:
                ag[a] = None
        doc = {n: v for n, v in zip(("k0", "k1"), ks) if v is not O.MISSING}
        groups.append(O.GroupRow(ks, ag, {"d": doc}))
    conv = lambda v: q.MISSING if v is O.MISSING else v
    rows = [([conv(k) for k in g.keys], [conv(g.aggregates[a]) for a in AGGS]) for g in groups]
    exprs, tries = [], 0
    while len(exprs) < 25 and tries < 400:
        tries += 1
        text = rand_expr(rng, rng.choice([1, 2, 2, 3]))
        try:
            canon = str(O.parse(text))
        except O.ParseError:
            continue
        exprs.append(canon)
    terms = [(e, "c%d" % i) for i, e in enumerate(exprs)]
    having = exprs[0]
    tail = dict(having=having, terms=terms)
    op = q.Operator(explain_plan("default", "d", "d", None, KEYS, AGGS, tail=tail), str(tmp_path), tail=True)
    assert op.tail_operators == ["Filter", "InitialProject", "FinalProject"], (op.tail_operators, exprs)
    got = op.run_tail(op.import_result(rows))
    want = O.run_tail(groups, having=having, terms=terms)
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        if not finite([w]):
            continue  # +-Inf / NaN have no JSON number form: rendered as strings, compared nowhere
        assert normalise(g) == normalise(w), "group %d\n%s" % (i, "\n".join(
            "%s: %r != %r   %s" % (k, g.get(k, "<missing>"), w.get(k, "<missing>"), dict(terms)[k] if False else exprs[int(k[1:])])
            for k in sorted(set(g) | set(w)) if normalise(g.get(k, "<missing>")) != normalise(w.get(k, "<missing>"))))
