"""Computed group keys, aggregate operands, DISTINCT operands and WHERE comparisons at the int64 limits and on both
sides of every range proof the expression analysis feeds.

For a computed `+ - * neg` the planner's range proof comes from the interval arithmetic of `bind_and_analyze`
(query_b200/csrc/expr.cpp), which restates intValue.Add / Mult / Neg / Sub: `+` folds from int 0 (0 counts as
non-negative, so a negative first addend already gives a float), `a - b` is `a + (-b)` unless b is MinInt64, `*` folds
from 1 with Go's `rv / this == n` check (so `-1 * MinInt64` is the int MinInt64 and `MinInt64 * -1` the float 2^63),
and `/` and `%` go through float64 and NewValue.  Every narrow layout - biased / offset-packed / mixed-radix keys,
dense / direct / hashed tables, one `isum` word, the float-carried sum, one-cell cached sums, 32-bit MIN / MAX cells,
the sign mix read off MIN / MAX, the partitioned DISTINCT aggregation - trusts that interval.  A value outside it packs
into another group's slot or wraps a narrow cell without any error, so the operand columns here hold rows at both
endpoints of their ranges (every corner of the computed interval is reached in every group), and the thresholds are
crossed by the computed interval, not by a column's statistics.

The reference takes each row's value from the oracle's expression tree (`O.parse(text).evaluate`, as `O.run_chain`
evaluates it) and reduces the groups with `exact_aggregates` of test_int_edges: COUNT / COUNTN / SUM / AVG over the
values as computed (an integral computed float stays a float in SUM), MIN / MAX, DISTINCT and group keys over the
canonical number (canon_num: an integral float is the equal int, as the reference's group text and value.Set key it).
value.Set keeps the member it was given, so for a set whose member is an integral computed float (`100 - x`) the
reference's SUM(DISTINCT) adds that float and gives a float of the same value; the device, and this reference, add the
set's key, the int.  The rendered number is the same.

The CPU tests pin which side of every threshold each fixture lands on, and check the analysis against the oracle on
seeded random expression trees over int64 endpoint values.
"""
import functools
import itertools
import json
import random
import re

import numpy as np
import pytest

import query_b200 as q
from oracle import n1ql_oracle as O
from test_int_edges import (FCARRY_ROWS, I64_MAX, I64_MIN, ISUM34_ROWS, KEY_COLUMNS, LAYOUTS, MM32_SPAN, T_FLOAT, T_INT,
                            T_MISSING, T_NULL, _agg_kind, _tight, assert_exact, exact_aggregates)
from util_n1 import gpu_rows

F = lambda c: "(`d`.`%s`)" % c
X, Y, Z = F("x"), F("y"), F("z")


# ---- fixtures: operand columns at both endpoints of their ranges, six groups ------------------------------------------
def _col(vals):
    """python values (int, non-integral float, None, MISSING) -> (tags, payload) of a pre-shredded column"""
    tags = np.array([T_MISSING if v is O.MISSING else T_NULL if v is None else T_FLOAT if isinstance(v, float) else T_INT
                     for v in vals], dtype=np.uint8)
    pay = np.array([0 if v is None or v is O.MISSING else v for v in vals], dtype=object)
    out = np.zeros(len(vals), dtype=np.int64)
    for i, (t, p) in enumerate(zip(tags.tolist(), pay.tolist())):
        out[i] = np.array([p], dtype=np.float64).view(np.int64)[0] if t == T_FLOAT else p
    return tags, out


class Case:
    def __init__(self, name, cols, exprs, n=3000, seed=0, global_rows=None, absent=True, floats=None, roles="abcd",
                 layouts=None, key_land=None, marks=None, gk=False):
        """cols: {column: (lo, hi)}; exprs: shape texts over X / Y / Z.  Every group gets every corner of the columns'
        ranges, `n` random rows, and (with `absent`) rows where one operand is MISSING or NULL.  floats: {column:
        non-integral floats sprinkled in}.  key_land: (mode, kernel text present, absent) of role (a) with the
        first expression as the key alone; marks: [(layout, present, absent)] of role (b); gk: an 8192-key column for the partitioned
        DISTINCT aggregation."""
        self.name, self.cols, self.exprs, self.global_rows = name, cols, exprs, global_rows
        self.roles, self.key_land, self.marks = roles, key_land, marks or []
        self.layouts = list(LAYOUTS) if layouts is None else layouts
        rng = np.random.default_rng(seed)
        names = sorted(cols)
        rows, gid = [], []
        corners = list(itertools.product(*[cols[c] for c in names]))
        for g in range(6):
            for _rep in range(3):
                rows += corners
            gid += [g] * 3 * len(corners)
            if absent:
                for c in range(len(names)):
                    for a in (O.MISSING, None):
                        r = list(corners[g % len(corners)])
                        r[c] = a
                        rows.append(tuple(r))
                        gid.append(g)
        rnd = [rng.integers(cols[c][0], cols[c][1], size=n, endpoint=True, dtype=np.int64).tolist() for c in names]
        rows += list(zip(*rnd))
        gid += rng.integers(0, 6, n).tolist()
        for c, fl in (floats or {}).items():
            for i, f in enumerate(fl):
                r = list(corners[i % len(corners)])
                r[names.index(c)] = float(f)
                rows.append(tuple(r))
                gid.append(i % 6)
        perm = np.random.default_rng(seed + 1).permutation(len(rows))
        self.rows = [rows[i] for i in perm]
        self.gid = np.asarray(gid, dtype=np.int64)[perm]
        self.names = names
        self.keys = dict(KEY_COLUMNS, g=_tight(-2))
        if gk:  # 8192 keys, both ends present
            k = rng.integers(0, 8192, len(self.rows))
            k[:2] = [0, 8191]
            self.keys = {"gk": [(T_INT, int(v)) for v in range(8192)]}
            self.gid = k.astype(np.int64)

    def __repr__(self):
        return self.name

    @functools.cached_property
    def table(self):
        t = q.Table(self.names + sorted(self.keys))
        for i, c in enumerate(self.names):
            tags, pay = _col([r[i] for r in self.rows])
            t.set_column(c, pay, tags=tags)
        for c, spec in self.keys.items():
            t.set_column(c, np.array([s[1] for s in spec], dtype=np.int64)[self.gid],
                         tags=np.array([s[0] for s in spec], dtype=np.uint8)[self.gid])
        if self.global_rows is not None:
            t.set_global_rows(self.global_rows)
        t.seal()
        return t

    @functools.cached_property
    def docs(self):
        """each row as the oracle's item: {alias: document}, MISSING fields left out"""
        return [{"d": {c: v for c, v in zip(self.names, r) if v is not O.MISSING}} for r in self.rows]

    @functools.lru_cache(maxsize=None)
    def values(self, text):
        e = O.parse(text)
        return [e.evaluate(item) for item in self.docs]

    def key_text(self, c, g):
        kt, kv = self.keys[c][g]
        return "MISSING" if kt == T_MISSING else "null" if kt == T_NULL else json.dumps(kv)

    def expected(self, keys, aggs, where=None):
        """keys: key column names or computed key texts; aggs: aggregate texts over one operand (or count(*))"""
        keep = [O.truth(v) for v in self.values(where)] if where else [True] * len(self.rows)
        ops = {a.split("(", 1)[1][:-1].replace("distinct ", "") for a in aggs if a != "count(*)"}
        assert len(ops) <= 1, aggs
        vals = self.values(ops.pop()) if ops else [0] * len(self.rows)
        kvals = [self.values(k) if k not in self.keys else None for k in keys]
        by = {}
        for i, g in enumerate(self.gid.tolist()):
            if keep[i]:
                k = tuple(self.key_text(c, g) if kv is None else _ktext(kv[i]) for c, kv in zip(keys, kvals))
                by.setdefault(k, []).append(vals[i])
        if not keys and not by:
            by[()] = []
        out = {}
        for k, vs in by.items():
            raw, approx = exact_aggregates(vs)
            can, _ = exact_aggregates([_canon(v) for v in vs])
            dst, dapprox = exact_aggregates([_canon(v) for v in vs], distinct=True)
            r = {}
            for a in aggs:
                kind = _agg_kind(a)
                r[a] = (dst if "distinct" in a else can if kind in ("min", "max") else raw)[kind]
            out[k] = (r, dapprox if any("distinct" in a for a in aggs) else approx)
        return out


def _canon(v):
    """canon_num: an integral float is the equal int (value.NewValue)"""
    return O.new_value(v) if isinstance(v, float) else v


def _ktext(v):
    """a group key as gpu_rows renders it"""
    return "MISSING" if v is O.MISSING else json.dumps(O.to_python(_canon(v)))


def _cases():
    m31, m62 = 1 << 31, 1 << 62
    a = 7 * 73 * 127 * 337                      # a * b == 2^63 - 1
    b = I64_MAX // a
    assert a * b == I64_MAX
    big = 80000                                  # rows where cells must carry
    c = []
    # shapes
    c.append(Case("sub_nn", {"x": (0, 100), "y": (-100, 0)}, ["(%s - %s)" % (X, Y), "(7 - %s)" % Y, "(100 - %s)" % X],
                  seed=1, key_land=("dense-shared-memory", [], ["canon_num("])))
    c.append(Case("sub_nn_across", {"x": (-1, 100), "y": (-100, 0)}, ["(%s - %s)" % (X, Y)], seed=2, roles="abd"))
    c.append(Case("sub_ng", {"x": (-100, -1), "y": (1, 100)}, ["(%s - %s)" % (X, Y)], seed=3,
                  key_land=("dense-shared-memory", [], ["canon_num("])))
    c.append(Case("sub_ng_across", {"x": (-100, 0), "y": (1, 100)}, ["(%s - %s)" % (X, Y)], seed=4,
                  key_land=(None, ["canon_num("], [])))
    c.append(Case("sub_nn_max", {"x": (0, m62), "y": (-(m62 - 1), 0)}, ["(%s - %s)" % (X, Y)], seed=5,
                  key_land=("hbm-hash-128", [], ["canon_num("])))
    c.append(Case("sub_nn_max_across", {"x": (0, m62), "y": (-m62, 0)}, ["(%s - %s)" % (X, Y)], seed=6,
                  key_land=("hbm-hash-128", ["canon_num("], [])))
    c.append(Case("sub_ng_min", {"x": (-m62, -1), "y": (1, m62)}, ["(%s - %s)" % (X, Y)], seed=7,
                  key_land=("hbm-hash-128", [], ["canon_num("])))
    c.append(Case("sub_ng_min_across", {"x": (-m62, -1), "y": (1, m62 + 1)}, ["(%s - %s)" % (X, Y)], seed=8,
                  key_land=("hbm-hash-128", ["canon_num("], [])))
    c.append(Case("neg_min1", {"x": (I64_MIN + 1, I64_MAX)}, ["(-%s)" % X], seed=9,
                  key_land=("hbm-hash-128", [], ["canon_num(", "C_FLOAT ?"])))
    c.append(Case("neg_min", {"x": (I64_MIN, I64_MAX)}, ["(-%s)" % X, "(-1 * %s)" % X, "(%s * -1)" % X], seed=10,
                  key_land=("hbm-hash-128", ["canon_num(", "C_FLOAT ?"], [])))
    c.append(Case("mul_const", {"x": (0, 1 << 20)}, ["(%s * 4096)" % X], seed=11, key_land=("hbm-hash-64", [], ["canon_num("])))
    c.append(Case("mul_max", {"x": (-a, a), "y": (-b, b)}, ["(%s * %s)" % (X, Y)], seed=12,
                  key_land=("hbm-hash-128", [], ["canon_num("])))
    c.append(Case("mul_max_across", {"x": (-a, a), "y": (-b, b + 1)}, ["(%s * %s)" % (X, Y)], seed=13,
                  key_land=("hbm-hash-128", ["canon_num("], [])))
    c.append(Case("add_max", {"x": (0, m62), "y": (0, m62 - 1)}, ["(%s + %s)" % (X, Y)], seed=14,
                  key_land=("hbm-hash-128", [], ["canon_num("])))
    c.append(Case("add_max_across", {"x": (0, m62), "y": (0, m62)}, ["(%s + %s)" % (X, Y)], seed=15,
                  key_land=("hbm-hash-128", ["canon_num("], [])))
    c.append(Case("add_neg_first", {"x": (-100, -1), "y": (-100, -1)}, ["(%s + %s)" % (X, Y)], seed=16,
                  key_land=("hbm-hash-128", ["canon_num("], [])))
    c.append(Case("add_mixed", {"x": (-100, 100), "y": (0, 50)}, ["(%s + %s)" % (X, Y)], seed=17, roles="abd"))
    c.append(Case("add_partial_overflow", {"x": (m62, I64_MAX), "y": (0, m62), "z": (-m62, -1)}, ["(%s + %s + %s)" % (X, Y, Z)],
                  seed=18, key_land=("hbm-hash-128", ["canon_num("], [])))
    c.append(Case("div_mod", {"x": ((1 << 53) + 1, (1 << 53) + 4097), "y": (-2, 2)},
                  ["(%s / 1)" % X, "(%s / 2)" % X, "(%s %% 7)" % X, "(%s / 0)" % X, "(%s %% %s)" % (X, Y)], seed=19))
    # thresholds: key width and bias (role a), MISSING and NULL offset-packed into the computed key
    c.append(Case("keybits12", {"x": (0, 2046), "y": (0, 2047)}, ["(%s + %s)" % (X, Y)], seed=20, roles="a",
                  key_land=("dense-shared-memory", [], [])))
    c.append(Case("keybits13", {"x": (0, 2046), "y": (0, 2048)}, ["(%s + %s)" % (X, Y)], seed=21, roles="a",
                  key_land=("hbm-direct", [], [])))
    c.append(Case("keybits22", {"x": (0, (1 << 21) - 1), "y": (0, (1 << 21) - 2)}, ["(%s + %s)" % (X, Y)], seed=22, roles="a",
                  global_rows=1 << 19, key_land=("hbm-direct", [], [])))
    c.append(Case("keybits23", {"x": (0, (1 << 21) - 1), "y": (0, (1 << 21) - 1)}, ["(%s + %s)" % (X, Y)], seed=23, roles="a",
                  global_rows=1 << 19, key_land=("hbm-hash-64", [], [])))
    c.append(Case("keybias62", {"x": (0, m62 - 1)}, ["(-%s)" % X], seed=24, roles="a", absent=False, key_land=("hbm-hash-64", [], [])))
    c.append(Case("keybias62_across", {"x": (0, m62)}, ["(-%s)" % X], seed=25, roles="a", absent=False,
                  key_land=("hbm-hash-128", [], [])))
    c.append(Case("tight", {"x": (2, 4), "y": (-1, 0)}, ["(%s - %s)" % (X, Y)], seed=26, roles="a",
                  key_land=("dense-shared-memory", ["s_priv"], [])))
    # thresholds of the accumulators (role b)
    grid = ["ungrouped", "dense-shared", "direct-cache256", "direct-nocache", "direct-nopair", "direct-nosign", "hash64", "hash128"]
    c.append(Case("isum_in", {"x": (0, 1 << 33), "y": (0, 1 << 33)}, ["(%s + %s)" % (X, Y)], n=big, seed=27, roles="b",
                  layouts=grid, global_rows=ISUM34_ROWS, marks=[("direct-cache256", [], [".b >> 32)"])]))
    c.append(Case("isum_out", {"x": (0, 1 << 33), "y": (0, 1 << 33)}, ["(%s + %s)" % (X, Y)], n=big, seed=27, roles="b",
                  layouts=grid, global_rows=ISUM34_ROWS + 1, marks=[("direct-cache256", [".b >> 32)"], [])]))
    fl = np.arange(200) + 0.25
    c.append(Case("fcarry_in", {"x": (0, 1 << 35), "y": (0, 1 << 35)}, ["(%s + %s)" % (X, Y)], n=big, seed=28, roles="b",
                  layouts=grid, floats={"y": fl}, global_rows=FCARRY_ROWS, marks=[("direct-cache256", ["num_f("], [])]))
    c.append(Case("fcarry_out", {"x": (0, 1 << 35), "y": (0, 1 << 35)}, ["(%s + %s)" % (X, Y)], n=big, seed=28, roles="b",
                  layouts=grid, floats={"y": fl}, global_rows=FCARRY_ROWS + 1, marks=[("direct-cache256", [], ["num_f("])]))
    wl = ["direct-cache256", "direct-cache1024", "direct-nosign", "hash64"]
    for nm, ylo, w in (("wide1", -(m31 - 1 - (1 << 30)), True), ("wide", -(m31 - (1 << 30)), False)):
        mk = [(l, ["cache_add_carry("] if w else ["cache_add_wide("], ["cache_add_wide("] if w else ["cache_add_carry("]) for l in wl[:2]]
        c.append(Case(nm, {"x": (0, 1 << 30), "y": (ylo, 0)}, ["(%s - %s)" % (X, Y), "(-(%s - %s))" % (X, Y)], n=big, seed=29,
                      roles="b", layouts=wl, marks=mk))
    for nm, s in (("mm32", MM32_SPAN), ("mm32_across", MM32_SPAN + 1)):
        mk = [(l, ["cache_mm32"], []) if s == MM32_SPAN else (l, [], ["cache_mm32"]) for l in ("direct-cache1024", "direct-nopair")]
        c.append(Case(nm, {"x": (0, m31), "y": (-(s - m31), 0)}, ["(%s - %s)" % (X, Y)], n=20000, seed=30, roles="b",
                      layouts=["ungrouped", "direct-cache1024", "direct-nopair", "hash64"], marks=mk))
    c.append(Case("sign_straddle", {"x": (-1000, 1000)}, ["(%s * 3)" % X], n=big, seed=31, roles="b", layouts=wl,
                  marks=[("direct-cache1024", [], [".b < 0)"]), ("direct-nosign", [".b < 0)"], [])]))
    c.append(Case("sign_one_side", {"x": (0, 1000)}, ["(%s * 3)" % X], n=big, seed=32, roles="b", layouts=wl,
                  marks=[("direct-cache1024", [], [".b < 0)"]), ("direct-nosign", [], [".b < 0)"])]))
    # the partitioned DISTINCT aggregation: a 12-bit computed value (4096 values) and one more
    for nm, hi in (("part4096", 4094), ("part4097", 4095)):
        c.append(Case(nm, {"x": (0, hi), "y": (-1, 0)}, ["(%s - %s)" % (X, Y)], n=40000, seed=33, roles="c", absent=False,
                      global_rows=1 << 20, gk=True))
    return {x.name: x for x in c}


@functools.lru_cache(maxsize=None)
def cases():
    return _cases()


# ---- roles -------------------------------------------------------------------------------------------------------------
def _aggs(e):
    return ["count(*)", "count(%s)" % e, "countn(%s)" % e, "sum(%s)" % e, "avg(%s)" % e, "min(%s)" % e, "max(%s)" % e]


def _daggs(e):
    return ["count(*)", "count(distinct %s)" % e, "sum(distinct %s)" % e, "avg(distinct %s)" % e]


def _params():
    """(case, expression index, role, variant) of every GPU run"""
    out = []
    for c in cases().values():
        for i, _e in enumerate(c.exprs):
            if "a" in c.roles:
                out += [(c.name, i, "key", v) for v in ("alone", "with-g")]
            if "b" in c.roles:
                out += [(c.name, i, "operand", l) for l in c.layouts]
            if "c" in c.roles:
                out += [(c.name, i, "distinct", v) for v in (["gk"] if c.name.startswith("part") else ["ungrouped", "gd"])]
            if "d" in c.roles:
                out += [(c.name, i, "where", v) for v in ("le-lo", "eq-hi", "between")]
    return out


PARAMS = _params()


def _where(c, e, variant):
    nums = [_canon(v) for v in c.values(e) if isinstance(v, (int, float))] or [0]  # / 0: nothing is selected
    lo, hi = O.marshal(min(nums)), O.marshal(max(nums))
    return {"le-lo": "(%s <= %s)" % (e, lo), "eq-hi": "(%s = %s)" % (e, hi), "between": "(%s between %s and %s)" % (e, lo, hi)}[variant]


def _make(c, keys, aggs, env, where, monkeypatch):
    """keys: key column names or computed key texts"""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    qq = q.Query(c.table, "d", where, [F(k) if k in c.keys else k for k in keys], aggs)
    for k in env:
        monkeypatch.delenv(k)
    return qq


def plan(name, i, role, variant, monkeypatch):
    """Builds the query of one run and checks that it lands where the run means it to; returns (case, query, keys, aggs,
    where)."""
    c = cases()[name]
    e = c.exprs[i]
    where, env, mode, must, mustnot = None, {}, None, [], []
    if role == "key":
        keys = [e] if variant == "alone" else ["g", e]
        aggs = ["count(*)"] if variant == "alone" else ["count(*)", "sum(%s)" % e]
        if variant == "alone" and c.key_land and i == 0:
            mode, must, mustnot = c.key_land
    elif role == "operand":
        lk, env, mode, must, mustnot = LAYOUTS[variant]
        keys = list(lk)
        aggs = _aggs(e)
        if variant == "dense-priv" and "canon_num(" in _make(c, [], aggs, {}, None, monkeypatch).kernel_source:
            aggs = ["count(*)", "sum(%s)" % e, "avg(%s)" % e]  # FLOAT class words of MIN / MAX overflow the 48 private words
        for l, mu, mn in c.marks:
            if l == variant:
                must, mustnot = must + mu, mustnot + mn
    elif role == "distinct":
        keys = [] if variant == "ungrouped" else [variant]
        aggs = _daggs(e)
    else:
        keys = ["gd"]
        aggs = ["count(*)", "count(%s)" % e, "min(%s)" % e, "max(%s)" % e]
        where = _where(c, e, variant)
    qq = _make(c, keys, aggs, env, where, monkeypatch)
    src = qq.kernel_source
    what = (name, e, role, variant)
    if mode is not None:
        assert qq.info["mode"] == mode, (what, qq.info)
    assert all(m in src for m in must) and not any(m in src for m in mustnot), (what, must, mustnot)
    if role == "operand" and variant == "dense-priv":
        assert qq.info["slots"] == 6
    if name == "tight" and variant == "alone":
        assert qq.info["slots"] == 6  # MISSING, NULL and four ints: a six-slot mixed-radix table
    if name.startswith("part"):
        assert bool(qq.part_source) == (name == "part4096"), what
    return c, qq, keys, aggs, where


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def _device():
    q.init(0)


@pytest.mark.gpu
@pytest.mark.parametrize("name,i,role,variant", PARAMS, ids=["%s-%d-%s-%s" % p for p in PARAMS])
def test_computed_values_match_the_exact_reference(name, i, role, variant, _device, monkeypatch):
    c, qq, keys, aggs, where = plan(name, i, role, variant, monkeypatch)
    got = gpu_rows(qq.execute(), aggs)
    assert_exact(c.expected(keys, aggs, where), got, "%s %s as %s (%s)" % (name, c.exprs[i], role, variant))


# ---- CPU: landing ----------------------------------------------------------------------------------------------------
def test_gpu_runs_land_on_their_layouts(monkeypatch):
    """Every GPU run reaches the mode and kernel text it relies on, so a planner change cannot move a fixture to the
    other side of its threshold unnoticed."""
    for name, i, role, variant in PARAMS:
        c = cases()[name]
        if role == "operand" or (variant == "alone" and c.key_land and i == 0) or role == "distinct" and variant == "gk":
            plan(name, i, role, variant, monkeypatch)


def test_fixtures_reach_the_corners_the_shapes_are_about():
    """The values the shapes exist for occur in the fixtures (the reference itself, checked against hand-made facts)."""
    vals = lambda name, k: {(type(v), v) for v in cases()[name].values(cases()[name].exprs[k])}
    assert (int, I64_MAX) in vals("sub_nn_max", 0) and (float, 2.0 ** 63) in vals("sub_nn_max_across", 0)
    assert (int, I64_MIN) in vals("sub_ng_min", 0) and (float, -(2.0 ** 63)) in vals("sub_ng_min_across", 0)
    assert (float, 2.0 ** 63) in vals("neg_min", 0) and (float, 2.0 ** 63) not in vals("neg_min1", 0)
    assert (int, I64_MIN) in vals("neg_min", 1) and (float, 2.0 ** 63) in vals("neg_min", 2)  # -1 * MinInt64, MinInt64 * -1
    assert (int, I64_MAX) in vals("mul_max", 0) and (int, -I64_MAX) in vals("mul_max", 0)
    assert any(t is float for t, _v in vals("mul_max_across", 0))
    assert (int, I64_MAX) in vals("add_max", 0) and (float, 2.0 ** 63) in vals("add_max_across", 0)
    assert (float, -200.0) in vals("add_neg_first", 0) and not any(t is int for t, _v in vals("add_neg_first", 0))
    # MaxInt64 + 1 overflows to a float before -1 brings the total back into int64
    assert (float, 2.0 ** 63) in vals("add_partial_overflow", 0)
    dm = cases()["div_mod"]
    assert (int, 1 << 53) in {(type(v), v) for v in dm.values(dm.exprs[0])}   # (2^53 + 1) / 1
    assert {v for v in dm.values(dm.exprs[3])} >= {None, O.MISSING}          # / 0
    assert O.parse("((-5) + (-3))").evaluate({}) == -8.0 and isinstance(O.parse("((-5) + (-3))").evaluate({}), float)


# ---- CPU: the reference against the oracle ---------------------------------------------------------------------------
def test_exact_reference_matches_the_oracle_on_same_sign_fixtures():
    """Where every computed int has one sign no evaluation order can overflow differently, so the oracle's own chain must
    give the exact reference's results, class included."""
    for name in ("sub_nn", "sub_ng", "keybits12", "tight"):
        c = cases()[name]
        e = c.exprs[0]
        for keys in ([], [e]):
            aggs = _aggs(e)
            want = {}
            for r in O.run_chain([d["d"] for d in c.docs], "d", None, [F(k) if k in c.keys else k for k in keys], aggs):
                want[tuple(_ktext(v) for v in r.keys)] = dict(r.aggregates)
            exp = c.expected(keys, aggs)
            assert set(want) == set(exp), (name, keys)
            for k, (ag, _approx) in exp.items():
                for a, v in ag.items():
                    assert type(want[k][a]) is type(v) and want[k][a] == v, (name, keys, k, a, want[k][a], v)


# ---- CPU: soundness of the analysis on random trees --------------------------------------------------------------------
ENDPOINTS = [I64_MIN, I64_MIN + 1, -(1 << 62), -(1 << 31), -1, 0, 1, 2, 7, 1 << 31, 1 << 62, I64_MAX - 1, I64_MAX]
_INT_PAY = re.compile(r"pack_bits\(klo, khi, kpos, \((\w+)\.c == C_INT \? (?:\(\(u64\)\1\.b - \(u64\)\(\(i64\)(0x[0-9a-f]+)ULL\)\)|\(u64\)\1\.b) : (.*), (\d+)\);$")


def _tree(rng, d):
    if d == 0 or rng.random() < 0.25:
        return rng.choice([X, Y]) if rng.random() < 0.7 else str(rng.choice(ENDPOINTS) if rng.random() < 0.6 else rng.randint(-9, 9))
    k = rng.choice("+-*n")
    if k == "n":
        return "(-%s)" % _tree(rng, d - 1)
    return "(%s %s %s)" % (_tree(rng, d - 1), k, _tree(rng, d - 1))


def test_key_packing_holds_every_value_of_random_trees(monkeypatch):
    """Random `+ - * neg` trees over x and y whose ranges end at int64 endpoints, compiled as a group key (with MIN, MAX
    and SUM over it): for every combination of endpoint values the oracle's INT result must fit the bias and width the
    kernel packs, and a FLOAT result needs a FLOAT class or an unbiased 64-bit INT payload (after canon_num)."""
    rng = random.Random(7)
    checked = 0
    while checked < 120:
        xs, ys = sorted(rng.sample(ENDPOINTS, 2)), sorted(rng.sample(ENDPOINTS, 2))
        e = _tree(rng, 3)
        if X not in e and Y not in e:
            continue
        e = str(O.parse(e))
        t = q.Table(["x", "y"])
        t.set_column("x", np.array(xs + [xs[0]], dtype=np.int64))
        t.set_column("y", np.array(ys + [ys[1]], dtype=np.int64))
        t.seal()
        monkeypatch.setenv("N1GPU_NO_TIGHT", "1")  # the bit-packed key form (a mixed-radix slot hides the payload's width)
        qq = q.Query(t, "d", None, [e], ["count(*)", "min(%s)" % e, "max(%s)" % e, "sum(%s)" % e])
        monkeypatch.delenv("N1GPU_NO_TIGHT")
        src = qq.kernel_source
        packs = {m.group(2, 3, 4) for m in (_INT_PAY.match(l.strip()) for l in src.splitlines()) if m}
        assert len(packs) == 1, e  # the same key packing in every row loop of the kernel
        b, other, bits = packs.pop()
        bias = None if b is None else int(b, 16) - (1 << 64 if int(b, 16) >= 1 << 63 else 0)
        bits, has_float = int(bits), "C_FLOAT" in other
        tree = O.parse(e)
        for a, b in itertools.product(xs, ys):
            v = tree.evaluate({"d": {"x": a, "y": b}})
            cv = _canon(v)
            if isinstance(v, float):
                assert has_float or (bias is None and bits == 64), (e, xs, ys, a, b, v)
            if isinstance(cv, int):
                assert bias is None and bits == 64 or 0 <= cv - bias < (1 << bits), (e, xs, ys, a, b, v, bias, bits)
        checked += 1
