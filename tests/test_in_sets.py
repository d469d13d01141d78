"""IN over array parameters and long literal lists: `x IN $p` binds a JSON array, and the list is probed as a device-resident
set (NqInSet in n1ql_value.cuh) whose contents are kernel arguments, so every binding of a statement runs one cubin.
Literal lists of at most IN_CHAIN_MAX elements keep the unrolled in_arg chain."""
import functools
import json
import os

import numpy as np
import pytest

import query_b200 as q
from gen_n1 import F, config4_docs, config5_docs, make_docs
from util_n1 import assert_same, gpu_rows, make_table, oracle_rows

IN_CHAIN_MAX = 16  # codegen.hpp: literal lists longer than this are probed as a set (DESIGN.md section 3.1)
MAX_IN_SETS = 8
I64_MIN, I64_MAX = -(1 << 63), (1 << 63) - 1
MISSING = object()  # a `missing` element: only a literal list can hold one (JSON has no MISSING)


def lit(v):
    """an element as N1QL literal text"""
    if v is MISSING:
        return "missing"
    if isinstance(v, float):
        return repr(v)
    return json.dumps(v, ensure_ascii=False)


def lit_list(vals):
    return "[" + ", ".join(lit(v) for v in vals) + "]"


def _table(docs, where, keys, aggs):
    t = make_table(docs, where, keys, aggs)
    t.seal()
    return t


# ---- CPU: binding, eligibility, one kernel per shape ------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _cpu_docs():
    return make_docs(600, seed=31)


def test_one_kernel_per_statement_shape():
    docs = _cpu_docs()
    where = "(%s in $p)" % F("n")
    keys, aggs = [F("g")], ["count(*)", "sum(%s)" % F("i")]
    t = _table(docs, where.replace("$p", "[1]"), keys, aggs)
    c0, _ = q.jit_stats()
    bindings = [[1], list(range(50000)), [1, 2.5, None, True, False, "a", -0.0, 2.0 ** 63, -1]]
    qs = [q.Query(t, "d", where, keys, aggs, params={"p": b}) for b in bindings]
    c1, _ = q.jit_stats()
    assert len({x.kernel_source for x in qs}) == 1 and c1 - c0 <= 1
    assert "in_set(" in qs[0].kernel_source and "in_arg(" not in qs[0].kernel_source
    # two different literal lists longer than the chain limit: one kernel as well
    long1 = "(%s in %s)" % (F("n"), lit_list(list(range(IN_CHAIN_MAX + 1))))
    long2 = "(%s in %s)" % (F("n"), lit_list([2.5, "x", None] + list(range(-500, 500, 7))))
    a, b = q.Query(t, "d", long1, keys, aggs), q.Query(t, "d", long2, keys, aggs)
    c2, _ = q.jit_stats()
    assert a.kernel_source == b.kernel_source and "in_set(" in a.kernel_source and c2 - c1 <= 1
    # a literal list of IN_CHAIN_MAX elements is still today's chain, one in_arg per element
    chain = q.Query(t, "d", "(%s in %s)" % (F("n"), lit_list(list(range(IN_CHAIN_MAX)))), keys, aggs).kernel_source
    assert chain.count("in_arg(") == IN_CHAIN_MAX and "in_set(" not in chain


def test_element_classes_never_reach_the_kernel_text():
    """The result classes of an IN that takes the set do not depend on the elements: binding [1] or [1, null] - or a long
    literal list with or without a null / missing - to an IN in a group key or an aggregate operand over a column that
    holds no NULL gives one kernel text and one compile."""
    import numpy as np
    t = q.Table(["v", "g"])
    t.set_column("v", np.arange(1000, dtype=np.int64))
    t.set_column("g", np.arange(1000, dtype=np.int64) % 7)
    t.seal()
    v, g = F("v"), F("g")
    shapes = [(None, ["(%s in $p)" % v], ["count(*)"]), (None, [g], ["count((%s in $p))" % v, "sum((%s in $p))" % v]),
              ("(not (%s in $p))" % v, [g], ["count(*)"])]
    for where, keys, aggs in shapes:
        c0, _ = q.jit_stats()
        srcs = {q.Query(t, "d", where, keys, aggs, params={"p": b}).kernel_source for b in ([1], [1, None], [], [None, "a", True, 2.5])}
        c1, _ = q.jit_stats()
        assert len(srcs) == 1 and c1 - c0 <= 1, (where, keys, aggs)
        if any("$p" in a for a in aggs):
            continue  # an aggregate's text is a comment in the kernel: each literal list there is a text of its own
        base = list(range(IN_CHAIN_MAX + 4))
        sub = lambda vals, x: x.replace("$p", lit_list(vals)) if x else x
        lits = {q.Query(t, "d", sub(vals, where), [sub(vals, k) for k in keys], [sub(vals, a) for a in aggs]).kernel_source
                for vals in (base, base + [None], base + [MISSING], base + [MISSING, None, "x"])}
        assert len(lits) == 1 and "in_set(" in lits.pop(), (where, keys, aggs)


def test_string_and_boolean_operands_take_the_set():
    docs = _cpu_docs()
    for x, vals in ((F("s"), ["ab", "", "absent"]), (F("b"), [True]), (F("m"), [1, "a", 2.5, False, None])):
        t = _table(docs, "(%s in [1])" % x, [], ["count(*)"])
        src = q.Query(t, "d", "(not (%s in $p))" % x, [], ["count(*)"], params={"p": vals}).kernel_source
        assert "in_set(" in src, x


@pytest.mark.parametrize("where,keys,aggs", [
    ("(%s between $p and 5)" % F("i"), [], ["count(*)"]),
    ("(%s = $p)" % F("i"), [], ["count(*)"]),
    ("((%s + $p) < 3)" % F("i"), [], ["count(*)"]),
    (None, ["$p"], ["count(*)"]),
    (None, ["(%s + $p)" % F("i")], ["count(*)"]),
    (None, [], ["sum($p)"]),
    (None, [], ["count($p)"]),
    ("($p in [1, 2])", [], ["count(*)"]),
    ("(%s in [$p, 2])" % F("i"), [], ["count(*)"]),
], ids=["between", "eq", "arith", "group_key", "group_key_arith", "sum_operand", "count_operand", "left_of_in", "inside_a_list"])
def test_array_parameter_outside_in_is_ineligible(where, keys, aggs):
    docs = _cpu_docs()
    t = _table(docs, "(%s < 1)" % F("i"), [F("i")], ["count(*)"])
    with pytest.raises(q.Ineligible):
        q.Query(t, "d", where, keys, aggs, params={"p": [1, 2]})


@pytest.mark.parametrize("value", [[[1]], [1, [2]], [{"a": 1}], 3, "x", None], ids=["nested", "nested_late", "object", "int", "string", "null"])
def test_non_array_or_nested_values_are_ineligible_in_in(value):
    docs = _cpu_docs()
    t = _table(docs, "(%s < 1)" % F("i"), [], ["count(*)"])
    with pytest.raises(q.Ineligible):
        q.Query(t, "d", "(%s in $p)" % F("i"), [], ["count(*)"], params={"p": value})


def test_malformed_array_values_are_parse_errors():
    t = _table(_cpu_docs(), "(%s < 1)" % F("i"), [], ["count(*)"])
    h = q.lib()
    import ctypes as C
    for text in (b"[1, 2", b"[1 2]", b"[1] x", b"[\"a\" 3]"):
        out = C.c_void_p()
        where = ("(%s in $p)" % F("i")).encode()
        aggs = (C.c_char_p * 1)(b"count(*)")
        rc = h.n1gpu_query_compile_params(t._h, b"d", where, (C.c_char_p * 1)(), 0, aggs, 1, (C.c_char_p * 1)(b"p"), (C.c_char_p * 1)(text), 1, C.byref(out))
        assert rc == q._lib.E_PARSE, (text, rc)


def test_set_limit_per_chain():
    docs = _cpu_docs()
    cols = ["i", "p", "n", "f", "m", "s", "b", "g", "h"]
    t = _table(docs, "(" + " and ".join("(%s < 1)" % F(c) for c in cols) + ")", [], ["count(*)"])
    conds = ["(%s in $p%d)" % (F(c), k) for k, c in enumerate(cols)]
    params = {"p%d" % k: [1, "a", True] for k in range(len(cols))}
    ok = q.Query(t, "d", "(" + " or ".join(conds[:MAX_IN_SETS]) + ")", [], ["count(*)"], params=params)
    assert ok.kernel_source.count("in_set(") == MAX_IN_SETS
    with pytest.raises(q.Ineligible):
        q.Query(t, "d", "(" + " or ".join(conds[:MAX_IN_SETS + 1]) + ")", [], ["count(*)"], params=params)


def test_parameter_text_and_empty_array():
    t = _table(_cpu_docs(), "(%s < 1)" % F("i"), [], ["count(*)"])
    qq = q.Query(t, "d", "(not (%s in $ids))" % F("i"), [], ["count(*)"], params={"$ids": []})
    assert "in_set(" in qq.kernel_source


# ---- GPU: oracle parity --------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def _device():
    q.init(0)


@functools.lru_cache(maxsize=None)
def _docs():
    return make_docs(2000, seed=77)


def _big_ns():
    """a few `n` values of the documents beyond 2^53, and their neighbours"""
    ns = sorted({json.loads(d)["n"] for d in _docs() if isinstance(json.loads(d).get("n"), int) and abs(json.loads(d)["n"]) > 2 ** 53})
    pick = ns[:: max(1, len(ns) // 6)][:6]
    return pick + [v + 1 for v in pick] + [2 ** 53, 2 ** 53 + 1, 2 ** 53 + 2, 2 ** 53 + 8, -(2 ** 53) - 2]


def _pad(vals):
    """a literal list longer than the chain limit (elements that match nothing in the documents)"""
    return vals + [0.123 + k for k in range(IN_CHAIN_MAX + 1 - len(vals))]


LISTS = {
    "empty": lambda: [],
    "duplicates": lambda: [1, 1, 2, 2, -1, -1, "a", "a", True, True, 2.5, 2.5],
    "null": lambda: [None, 3, 4, "ab"],
    "missing": lambda: _pad([MISSING, 5, "b"]),
    "missing_null": lambda: _pad([MISSING, None, 7]),
    "only_missing": lambda: [MISSING] * (IN_CHAIN_MAX + 1),
    "strings": lambda: ["", "ab", "nope", "zeta", "日本", "q\"uote", "tab\there", "x y"],
    "limits": lambda: [I64_MIN, I64_MAX, -1, 0],
    "big_floats": lambda: [2.0 ** 63, 9.3e18, -9.3e18, 1e300, -1e300, -(2.0 ** 63)],
    "beyond_2p53": _big_ns,
    "neg_zero": lambda: [-0.0, 0.5, 2.0, -3],
    "mixed": lambda: [1, 2.5, None, True, False, "a", "é", -0.0, 3.0],
    "long_ints": lambda: list(range(-50, 51, 3)),
}
OPERANDS = {"i": F("i"), "n": F("n"), "f": F("f"), "m": F("m"), "s": F("s"), "b": F("b"),
            "i_x1.5": "(%s * 1.5)" % F("i"), "n_plus_half": "(%s + 0.5)" % F("n")}


def _bind(text, name, vals):
    """(statement text for libn1gpu, params, statement text for the oracle)"""
    if any(v is MISSING for v in vals):
        t = text.replace("$" + name, lit_list(vals))
        return t, None, t
    return text, {name: vals}, text.replace("$" + name, lit_list(vals))


@pytest.mark.gpu
@pytest.mark.parametrize("lname", list(LISTS))
@pytest.mark.parametrize("oname", list(OPERANDS))
def test_in_and_not_in_against_the_oracle(oname, lname, _device):
    docs = _docs()
    x, vals = OPERANDS[oname], LISTS[lname]()
    # the IN result as the group key: TRUE / FALSE / NULL / MISSING rows counted in one run; NOT IN as the filter
    for where, keys, aggs in ((None, ["(%s in $p)" % x], ["count(*)", "sum(%s)" % F("i")]),
                              ("(not (%s in $p))" % x, [], ["count(*)", "sum(%s)" % F("p"), "min(%s)" % F("m")])):
        w, params, wo = _bind(where, "p", vals) if where else (None, None, None)
        k, kp, ko = _bind(keys[0], "p", vals) if keys else (None, None, None)
        params = params or kp
        gk, ok = ([k], [ko]) if keys else ([], [])
        t = _table(docs, wo, ok, aggs)
        qq = q.Query(t, "d", w, gk, aggs, params=params)
        assert "in_set(" in qq.kernel_source
        exp = oracle_rows(docs, "d", wo, ok, aggs)
        assert_same(exp, gpu_rows(qq.execute(), aggs), "%s in %s" % (oname, lname))


def _limit_docs():
    """documents whose `z` sits at the int64 limits, at 2^63 as a float, and on both sides of the values that round to it"""
    vals = ["9223372036854775807", "9223372036854775707", "9223372036854774807", "9223372036854775295",
            "-9223372036854775808", "-9223372036854775708", "9223372036854775808", "9.3e18", "-9.3e18", "-0.0", "0", "-1", "null"]
    return ['{"z": %s}' % v for v in vals] + ['{"y": 1}']


LIMIT_LISTS = {
    "limits": [I64_MIN, I64_MAX, -1],
    "p63": [2.0 ** 63],
    "p63_and_ints": [2.0 ** 63, I64_MIN, 0],
    "near_limits": [I64_MAX - 100, -(1 << 63) + 100, 9.3e18],
    "neg_floats": [-9.3e18, -(2.0 ** 63), 0.5],
}


@pytest.mark.gpu
@pytest.mark.parametrize("lname", list(LIMIT_LISTS))
@pytest.mark.parametrize("x", ["(`d`.`z`)", "((`d`.`z`) + 0.5)", "((`d`.`z`) - 0.5)"], ids=["z", "z_plus_half", "z_minus_half"])
def test_rows_at_the_int64_limits(x, lname, _device):
    """INT rows at INT64_MAX and within 512 below it equal the FLOAT element 2^63 (float64 rounding); FLOAT rows of 2^63
    equal the INT elements that round to it; INT64_MIN is the float -2^63."""
    docs = _limit_docs()
    vals = LIMIT_LISTS[lname]
    keys, aggs = ["(%s in $p)" % x, "(`d`.`z`)"], ["count(*)"]
    okeys = [k.replace("$p", lit_list(vals)) for k in keys]
    t = _table(docs, None, okeys, aggs)
    qq = q.Query(t, "d", None, keys, aggs, params={"p": vals})
    assert "in_set(" in qq.kernel_source
    assert_same(oracle_rows(docs, "d", None, okeys, aggs), gpu_rows(qq.execute(), aggs), "%s in %s" % (x, lname))


# (group keys, environment, mode, text the kernel must contain)
LAYOUTS = {
    "ungrouped": ([], {}, "ungrouped", "nq_scan"),
    "dense-priv": ([], {}, "dense-shared-memory", "s_priv"),  # the IN key alone: four groups
    "dense-shared": ([F("g")], {"N1GPU_NO_PRIV": "1"}, "dense-shared-memory", "s_tab"),
    "hbm-direct": ([F("p"), F("g")], {}, "hbm-direct", "cache_claim"),
    "hash64": ([F("h")], {"N1GPU_NO_DIRECT": "1"}, "hbm-hash-64", "table_insert64"),
    "hash128": ([F("h"), F("n")], {}, "hbm-hash-128", "table_insert128"),
}
LAYOUT_LISTS = {
    "a": ([1, 2, 3, -1, 50, 2.5, None], [5, 7, 11, 13, I64_MIN], ["ab", "", "zeta", "nope"], [0.5, -0.0, 3.0, None]),
    "b": ([], list(range(0, 1001, 2)), ["a"], [2.0 ** 63, 1.0, 2.0]),
}


def _layout_query(layout, lists, monkeypatch):
    keys, env, mode, must = LAYOUTS[layout]
    a, b, c, d = lists
    # two sets in the filter, one in a group key, one in a count(...) operand and one in a sum(...) operand
    where = "((%s in $a) or (not (%s in $b)))" % (F("i"), F("p"))
    keys = keys + (["(%s in $c)" % F("s")] if layout != "ungrouped" else [])  # TRUE / FALSE / NULL / MISSING
    aggs = ["count(*)", "count((%s in $d))" % F("f"), "sum((%s in $c))" % F("m"), "sum(%s)" % F("i")]
    if layout == "dense-priv":
        aggs = aggs[:2]
    params = {"a": a, "b": b, "c": c, "d": d}
    lit = lambda s: s.replace("$a", lit_list(a)).replace("$b", lit_list(b)).replace("$c", lit_list(c)).replace("$d", lit_list(d))
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    t = _table(_docs(), lit(where), [lit(k) for k in keys], [lit(x) for x in aggs])
    qq = q.Query(t, "d", where, keys, aggs, params=params)
    for k in env:
        monkeypatch.delenv(k)
    assert qq.info["mode"] == mode and must in qq.kernel_source, (layout, qq.info)
    return qq, lit(where), [lit(k) for k in keys], aggs, [lit(x) for x in aggs]


@pytest.mark.gpu
@pytest.mark.parametrize("lists", list(LAYOUT_LISTS))
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_sets_through_every_layout(layout, lists, _device, monkeypatch):
    from oracle import n1ql_oracle as O
    qq, where, keys, aggs, oaggs = _layout_query(layout, LAYOUT_LISTS[lists], monkeypatch)
    names = [str(O.parse(x)) for x in oaggs]  # the oracle keys aggregates by its own Stringer text
    got = {k: {names[i]: v for i, v in enumerate(d.values())} for k, d in gpu_rows(qq.execute(), aggs).items()}
    assert_same(oracle_rows(_docs(), "d", where, keys, oaggs), got, layout)


def test_gpu_layout_queries_land_on_their_layouts(monkeypatch):
    for layout in LAYOUTS:
        for lists in LAYOUT_LISTS.values():
            _layout_query(layout, lists, monkeypatch)


DISTINCT_SHAPES = {
    "partitioned": ({"N1GPU_PART": "1"}, lambda qq: "in_set(" in qq.part_source),
    "sliced-bitmap": ({"N1GPU_NO_PART": "1", "N1GPU_SET_PASSES": "2"}, lambda qq: not qq.part_source and "p.set_pass" in qq.kernel_source),
}


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(DISTINCT_SHAPES))
def test_distinct_shapes_filter_through_the_set(shape, _device, monkeypatch):
    docs = config4_docs(30000, 20000, 5)
    keys, aggs = ["(`d`.`g`)"], ["count(distinct (`d`.`x`))", "sum(distinct (`d`.`x`))", "count(*)"]
    vals = list(range(0, 1000, 3)) + [-1, 2.5]
    where = "((`d`.`x`) in $p)"
    wo = where.replace("$p", lit_list(vals))
    env, check = DISTINCT_SHAPES[shape]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    t = make_table(docs, wo, keys, aggs)
    t.set_global_rows(1 << 31)  # a bitmap beyond what the L2 keeps: the multi-pass scan
    t.seal()
    qq = q.Query(t, "d", where, keys, aggs, params={"p": vals})
    assert qq.info["mode"] == "hbm-direct" and check(qq), (shape, qq.info)
    got = gpu_rows(qq.execute(), aggs)
    assert_same(oracle_rows(docs, "d", wo, keys, aggs), got, shape)


# ---- GPU: scale --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_large_sets_on_ten_million_rows(_device):
    import torch
    rng = np.random.default_rng(8)
    n = 10_000_000
    v = rng.integers(-(1 << 40), 1 << 40, n)
    v[::3] = rng.integers(0, 3_000_000, (n + 2) // 3)
    words = sorted("w%06d" % i for i in range(100_000))
    codes = rng.integers(0, len(words), n).astype(np.uint32)
    t = q.Table(["v", "k"])
    t.set_column("v", v)
    t.set_column("k", codes, dictionary=words)
    t.seal()
    aggs = ["count(*)", "sum((`d`.`v`))"]
    for size in (100_000, 1_000_000):
        lst = rng.choice(3_000_000, size, replace=False)
        lst[:10] = v[1:30:3][:10]  # a few of the large values too
        qq = q.Query(t, "d", "((`d`.`v`) in $p)", [], aggs, params={"p": lst.tolist()})
        (_, (cnt, sm)), = qq.execute().rows()
        sel = np.isin(v, lst)
        exp_sum = int(torch.tensor(v[sel]).sum()) if sel.any() else None
        assert cnt == int(sel.sum()) and sm == exp_sum, size
    pick = sorted(rng.choice(len(words), 5000, replace=False).tolist())
    qq = q.Query(t, "d", "((`d`.`k`) in $p)", [], aggs, params={"p": [words[i] for i in pick] + ["absent"]})
    (_, (cnt, sm)), = qq.execute().rows()
    sel = np.isin(codes, np.array(pick, dtype=np.uint32))
    assert cnt == int(sel.sum()) and sm == int(v[sel].sum())


# ---- GPU: ranks through the peer arena ---------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("nranks", [2, 3])
def test_long_literal_in_on_the_config5_key_across_ranks(nranks, _device):
    from query_b200 import dist as qd
    docs = config5_docs(24000, 3000, 17)
    vals = ["w%05d" % k for k in range(0, 3000, 7)] + ["absent", ""]
    where = "(((`d`.`v`) is not missing) and ((`d`.`k`) in %s))" % lit_list(vals)
    keys, aggs = ["(`d`.`k`)"], ["count(*)", "count((`d`.`v`))", "sum((`d`.`v`))", "min((`d`.`v`))", "max((`d`.`v`))"]
    parts = [docs[len(docs) * r // nranks: len(docs) * (r + 1) // nranks] for r in range(nranks)]
    tables = [make_table(p, where, keys, aggs) for p in parts]
    qd.agree_local(tables)
    mbs = [q.Mailbox(nranks, r, 1024, arena_bytes=16 << 20) for r in range(nranks)]
    for r in range(nranks):
        for o in range(nranks):
            mbs[r].set_peer(o, mbs[o].base)
    qs = []
    for r in range(nranks):
        tables[r].seal()
        qq = q.Query(tables[r], "d", where, keys, aggs)
        assert qq.info["mode"] == "hbm-direct" and "in_set(" in qq.kernel_source
        qq.set_mailbox(mbs[r])
        assert qq.peer_mode == 1
        qs.append(qq)
    exp = oracle_rows(docs, "d", where, keys, aggs)
    for step in range(2):
        for qq in qs:
            qq.launch()
        got = {}
        for qq in qs:
            part = gpu_rows(qq.collect(), aggs)
            assert not (set(part) & set(got)), "a group was finalised by two ranks"
            got.update(part)
        assert_same(exp, got, "%d ranks, step %d" % (nranks, step))
