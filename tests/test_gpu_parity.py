"""GPU parity tests (run with -m gpu on the B200 box): the CUDA path, driven through the C ABI, against
(a) the reference's golden vectors, (b) the oracle on seeded synthetic documents, bit-exact for
COUNT / MIN / MAX / integer SUM / group keys / DISTINCT sets and <= 1e-12 relative for float SUM/AVG."""
import json

import numpy as np
import pytest

import query_b200 as q
from gen_n1 import QUERIES, F, config5_docs, make_docs
from golden_plans import CASES, WHERE_CASES, _MISSING, keyspaces, normalise
from plans_n1 import distinct_plan, explain_plan
from util_n1 import assert_same, gpu_rows, make_table, oracle_rows, run_both, write_keyspace

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _device():
    q.init(0)


def _groups_for_projection(result, aggs):
    out = []
    for ks, ag in result.rows():
        keys = [_MISSING if k is q.MISSING else k for k in ks]
        out.append((keys, {a: normalise(v) for a, v in zip(aggs, ag)}))
    return out


@pytest.mark.parametrize("case", CASES, ids=lambda c: c.id)
def test_golden_through_query_abi(case):
    docs = [t for _k, t in case.docs()]
    aggs = sorted(set(case.aggs))
    qq, res = run_both(docs, case.alias, case.where, case.keys, aggs, case.id)
    got = case.project(_groups_for_projection(res, aggs))
    assert normalise(got) == normalise(case.golden["results"]), case.golden["statements"]


@pytest.mark.parametrize("case", WHERE_CASES, ids=lambda c: c.id)
def test_golden_filters_through_query_abi(case):
    docs = [t for _k, t in case.docs()]
    qq, res = run_both(docs, case.alias, case.where, case.keys, case.aggs, case.id)
    assert res.rows() == [([], [len(case.golden["results"])])]


def _with_row_id(text, i):
    """the document with a unique field `__row` (the statements of case_where project whole documents: row identity)"""
    t = text.strip()
    if not t.startswith("{"):
        return text
    rest = t[1:].lstrip()
    return '{"__row": %d%s%s' % (i, "" if rest.startswith("}") else ", ", rest)


@pytest.mark.parametrize("case", WHERE_CASES, ids=lambda c: c.id)
def test_golden_filters_select_the_same_documents(case):
    """Row identity, not only the row count: every document gets a unique `__row`; GROUP BY it under the golden statement's
    WHERE yields one group per selected document - the same documents as the oracle selects, as many as the golden holds."""
    docs = [_with_row_id(t, i) for i, (_k, t) in enumerate(case.docs())]
    key = "(`%s`.`__row`)" % case.alias
    qq, res = run_both(docs, case.alias, case.where, [key], ["count(*)"], case.id + " rows")
    rows = res.rows()
    assert len(rows) == len(case.golden["results"]) and all(a == [1] for _k, a in rows), case.golden["statements"]


@pytest.mark.parametrize("ks,alias,sql,where,keys,aggs,tail", [
    ("sampledb/dimestore/product", "product",
     "SELECT color, COUNT(*), SUM(unitPrice), AVG(unitPrice), MIN(unitPrice), MAX(unitPrice) FROM product WHERE unitPrice > 10 GROUP BY color",
     "(10 < (`product`.`unitPrice`))", ["(`product`.`color`)"],
     ["count(*)", "sum((`product`.`unitPrice`))", "avg((`product`.`unitPrice`))", "min((`product`.`unitPrice`))", "max((`product`.`unitPrice`))"],
     dict(terms=[("(`product`.`color`)", None), ("count(*)", None), ("sum((`product`.`unitPrice`))", None), ("avg((`product`.`unitPrice`))", None),
                 ("min((`product`.`unitPrice`))", None), ("max((`product`.`unitPrice`))", None)], order=[("(`product`.`color`)", False)])),
    ("sampledb/dimestore/review", "review", "SELECT rating, COUNT(*) FROM review WHERE rating > 1 GROUP BY rating",
     "(1 < (`review`.`rating`))", ["(`review`.`rating`)"], ["count(*)"],
     dict(terms=[("(`review`.`rating`)", None), ("count(*)", None)], order=[("(`review`.`rating`)", False)])),
], ids=["product", "review"])
def test_baseline_config1_statements_through_the_operator(ks, alias, sql, where, keys, aggs, tail, tmp_path):
    """BASELINE.json configs[0] (SURVEY.md 8d.1): the two statements on data/sampledb/dimestore - 900 products (float
    unitPrice, 31 colours) and 10 000 reviews (int rating) - from the reference's plan JSON through the operator and its tail,
    against the oracle's chain + tail over the same documents (the oracle is pinned to the reference's golden rows over these
    very products: test/multistore/test_cases/aggregate_functions/case_group_by_having.json)."""
    from oracle import n1ql_oracle as O
    docs = keyspaces()[ks]
    name = ks.split("/")[-1]
    write_keyspace(str(tmp_path), "dimestore", name, docs)
    aggs_sorted = sorted(set(aggs))
    op = q.Operator(explain_plan("dimestore", name, alias, where, keys, aggs_sorted, tail=tail), str(tmp_path), tail=True)
    got = op.run_tail(op.run_once())
    groups = O.run_chain([O.parse_document(t) for _k, t in docs], alias, where, keys, aggs_sorted)
    want = O.run_tail(groups, terms=tail["terms"], order=tail["order"])
    assert len(got) == len(want) > 3
    for g, w in zip(got, want):
        assert g.keys() == w.keys()
        for k in g:
            a, b = normalise(g[k]), normalise(w[k])
            if isinstance(a, float) or isinstance(b, float):
                assert abs(a - b) <= 1e-12 * max(abs(a), abs(b)), (sql, k, a, b)
            else:
                assert a == b, (sql, k, a, b)


@pytest.mark.parametrize("case", CASES[:6] + CASES[10:14], ids=lambda c: c.id)
def test_golden_through_plan_operator(case, tmp_path):
    """The reference-facing entry: plan JSON in EXPLAIN shape + a file-datastore directory."""
    ns, ks = "default", case.keyspace.split("/")[-1]
    write_keyspace(str(tmp_path), ns, ks, case.docs())
    aggs = sorted(set(case.aggs))
    plan = explain_plan(ns, ks, case.alias, case.where, case.keys, aggs)
    op = q.Operator(plan, str(tmp_path))
    assert op.rest_index == 5  # the caller still runs the projection Parallel
    res = op.run_once()
    got = case.project(_groups_for_projection(res, aggs))
    assert normalise(got) == normalise(case.golden["results"])
    m = op.marshal_json()
    assert m["#operator"] == "GpuGroupAggregate" and m["#stats"]["#itemsIn"] == len(case.docs())
    # EXPLAIN in the reference's group-aggregate pushdown shape (plan/scan_index_groupagg.go:188-222)
    ga = m["group_aggs"]
    assert ga["name"] == "GpuGroupAggregate" and [g["expr"] for g in ga.get("group", [])] == list(case.keys)
    assert [g["id"] for g in ga.get("group", [])] == list(range(len(case.keys)))
    assert len(ga["aggregates"]) == len(aggs) and all(a["aggregate"] in ("COUNT", "COUNTN", "SUM", "AVG", "MIN", "MAX") for a in ga["aggregates"])
    assert [a["id"] for a in ga["aggregates"]] == list(range(len(case.keys), len(case.keys) + len(aggs)))
    assert all(bool(a.get("distinct")) == ("distinct" in t) for a, t in zip(ga["aggregates"], aggs))
    rows = res.to_json()
    assert len(rows) == res.num_groups
    for r in rows:
        assert set(r["aggregates"].keys()) == set(aggs)
    with pytest.raises(q.N1GpuError):
        op.run_once()  # util.Once


@pytest.mark.parametrize("case", [c for c in CASES if c.tail is not None], ids=lambda c: c.id)
def test_golden_statement_end_to_end_with_tail(case, tmp_path):
    """SURVEY.md 8f rows 1-2: the whole statement - scan, filter, groups on the device, then HAVING / projection /
    ORDER BY / LIMIT in the operator's tail - from the reference's plan JSON to the reference's golden rows."""
    ns, ks = "default", case.keyspace.split("/")[-1]
    write_keyspace(str(tmp_path), ns, ks, case.docs())
    aggs = sorted(set(case.aggs))
    op = q.Operator(explain_plan(ns, ks, case.alias, case.where, case.keys, aggs, tail=case.tail), str(tmp_path), tail=True)
    assert op.tail_operators and op.rest_index == 6
    res = op.run_once()
    got = op.run_tail(res)
    assert normalise(got) == normalise(case.golden["results"]), case.golden["statements"]


@pytest.mark.parametrize("where,terms", [(None, [(F("t"), None)]), ("(%s < 500)" % F("p"), [(F("t"), "kind"), (F("h"), None)]),
                                         (None, [("(%s %% 5)" % F("p"), "m"), (F("s"), None)])], ids=["one", "two_where", "computed"])
def test_select_distinct_end_to_end(where, terms, tmp_path):
    """SURVEY.md 8f row 4: SELECT DISTINCT runs as GROUP BY <terms> with no aggregates on the device, its projection in
    the operator's tail; the rows equal the oracle's Filter -> InitialProject -> Distinct."""
    from oracle import n1ql_oracle as O
    docs = make_docs(3000, seed=61)
    write_keyspace(str(tmp_path), "default", "d", [("k%06d" % i, t) for i, t in enumerate(docs)])
    op = q.Operator(distinct_plan("default", "d", "d", where, terms), str(tmp_path), tail=True)
    got = op.run_tail(op.run_once())
    want = O.run_distinct([O.parse_document(d) for d in docs], "d", where, terms)
    canon = lambda rows: sorted(json.dumps(normalise(r), sort_keys=True) for r in rows)
    assert canon(got) == canon(want)


@pytest.mark.parametrize("name,where,keys,aggs", QUERIES, ids=[x[0] for x in QUERIES])
def test_matrix_against_oracle(name, where, keys, aggs):
    docs = make_docs(3000, seed=21)
    qq, res = run_both(docs, "d", where, keys, aggs, name)
    assert res.stats["rows"] == 3000


_GROUPED = [x for x in QUERIES if x[2]]


@pytest.mark.parametrize("knob", ["N1GPU_NO_DIRECT", "N1GPU_NO_BITMAP", "N1GPU_NO_OFFSET_PACK", "N1GPU_NO_CACHE", "N1GPU_NO_PACK",
                                  "N1GPU_NO_KEY32", "N1GPU_NO_COMPLEMENT", "N1GPU_CACHE_BLOCK=1024", "N1GPU_CACHE_BLOCK=256",
                                  "N1GPU_SET_PASSES=4", "N1GPU_NO_FCARRY", "N1GPU_NO_TIGHT", "N1GPU_PART",
                                  "N1GPU_NO_WIDE1", "N1GPU_NO_SIGN_FROM_MINMAX",
                                  "N1GPU_PRIV_BLOCK=640", "N1GPU_PRIV_BLOCK=96", "N1GPU_NO_MM_PAIR"])
@pytest.mark.parametrize("name,where,keys,aggs", _GROUPED, ids=[x[0] for x in _GROUPED])
def test_grouped_matrix_through_the_alternate_layouts(name, where, keys, aggs, knob, monkeypatch):
    """The planner picks direct-indexed tables, DISTINCT bitmaps, offset-packed keys, the shared-memory front cache
    (direct-mapped u32 keys, one large or five small blocks per SM), packed table counters and complemented COUNT(x)
    counters whenever statistics allow; the layouts they replace (open addressing, hash sets, class-bits packing,
    uncached updates, 64-bit cache keys, one counter per word) stay reachable for wider keys / larger keyspaces and are
    kept under test by switching each choice off (or, for the tuning knobs, on)."""
    k, _, v = knob.partition("=")
    monkeypatch.setenv(k, v or "1")
    docs = make_docs(3000, seed=22)
    run_both(docs, "d", where, keys, aggs, "%s %s" % (name, knob))


@pytest.mark.parametrize("block", ["256", "1024", "1024-wide"])
def test_skewed_string_keys_with_missing_and_null(block, monkeypatch):
    """BASELINE config 5 shape at oracle size: Zipf-skewed string keys, MISSING / NULL keys and values, more groups than
    the front cache holds (misses take the table path), both block shapes; bit-exact against the oracle."""
    block, _, variant = block.partition("-")
    for knob in {"wide": ["N1GPU_NO_WIDE1", "N1GPU_NO_SIGN_FROM_MINMAX"]}.get(variant, []):
        monkeypatch.setenv(knob, "1")
    monkeypatch.setenv("N1GPU_CACHE_BLOCK", block)
    monkeypatch.setenv("N1GPU_CACHE_KB", "2")  # a 2 KiB cache: most of the 3 000 keys miss
    docs = config5_docs(20000, 3000, 11)
    run_both(docs, "d", "((`d`.`v`) is not missing)", ["(`d`.`k`)"],
             ["count(*)", "count((`d`.`v`))", "sum((`d`.`v`))", "min((`d`.`v`))", "max((`d`.`v`))", "avg((`d`.`v`))"], "config5 shape block=" + block)


@pytest.mark.parametrize("groups,skew", [(40000, False), (3000, False), (40000, True)])
def test_partitioned_distinct_aggregation(groups, skew, monkeypatch):
    """BASELINE config 4 shape at oracle size through the partitioned DISTINCT aggregation (forced: the planner only picks it
    for keyspaces large enough to profit): records radix-partitioned by group range, one block per partition; with skewed
    group keys a partition overflows its share and the handle falls back to the general scan - same rows either way."""
    from gen_n1 import config4_docs
    monkeypatch.setenv("N1GPU_PART", "1")
    docs = config4_docs(30000, groups, 41)
    if skew:  # most rows in a handful of neighbouring groups: one partition receives far more than its share
        docs = docs[:2000] + ['{"g": %d, "x": %d}' % (7 + i % 3, i % 1000) for i in range(28000)]
    where, keys = None, ["(`d`.`g`)"]
    aggs = ["count(distinct (`d`.`x`))", "sum(distinct (`d`.`x`))", "count(*)", "avg(distinct (`d`.`x`))"]
    qq, res = run_both(docs, "d", where, keys, aggs, "partitioned distinct groups=%d skew=%s" % (groups, skew))
    assert "NP " in qq.part_source and qq.info["mode"] == "hbm-direct"
    # negative values: SUM(DISTINCT) counts them for the int / float class of the result (0 + negative -> float)
    docs2 = ['{"g": %d, "x": %d}' % (i % 5000, (i * 7) % 600 - 300) for i in range(30000)]
    run_both(docs2, "d", None, keys, aggs, "partitioned distinct, negative values")


@pytest.mark.parametrize("nranks", [2, 3])
def test_peer_arena_merge_owner_sharded(nranks):
    """The collective-free multi-GPU merge of direct-indexed tables, with all ranks driven by this one process on one
    device (n1gpu_mailbox_set_peer instead of CUDA IPC): every rank scans its row range into a table inside its arena,
    raises its flag, and rank r's finalisation folds slot range r of ALL tables - the union of the ranks' results must be
    the oracle's groups over the whole keyspace, each group finalised by exactly one rank.  Two steps: both table buffers."""
    from query_b200 import dist as qd
    docs = config5_docs(12000, 3000, 17)
    where, keys = "((`d`.`v`) is not missing)", ["(`d`.`k`)"]
    aggs = ["count(*)", "count((`d`.`v`))", "sum((`d`.`v`))", "min((`d`.`v`))", "max((`d`.`v`))", "avg((`d`.`v`))"]
    parts = [docs[len(docs) * r // nranks: len(docs) * (r + 1) // nranks] for r in range(nranks)]
    tables = [make_table(p, where, keys, aggs) for p in parts]
    qd.agree_local(tables)
    mbs = [q.Mailbox(nranks, r, 1024, arena_bytes=8 << 20) for r in range(nranks)]
    for r in range(nranks):
        for o in range(nranks):
            mbs[r].set_peer(o, mbs[o].base)
    qs = []
    for r in range(nranks):
        tables[r].seal()
        qq = q.Query(tables[r], "d", where, keys, aggs)
        assert qq.info["mode"] == "hbm-direct"
        qq.set_mailbox(mbs[r])
        qs.append(qq)
    assert len({x.kernel_source for x in qs}) == 1, "ranks must compile the same kernel"
    exp = oracle_rows(docs, "d", where, keys, aggs)
    for step in range(3):
        for qq in qs:
            qq.launch()      # every rank's scan + flag first: the finalisations below wait for all flags of the step
        got = {}
        for r, qq in enumerate(qs):
            part = gpu_rows(qq.collect(), aggs)
            assert not (set(part) & set(got)), "a group was finalised by two ranks"
            got.update(part)
        assert_same(exp, got, "peer merge, %d ranks, step %d" % (nranks, step))


def test_partial_import_grows_the_owners_table():
    """An owner whose own partition holds a handful of groups imports thousands from a peer: its hash table (sized for its
    own rows) and DISTINCT set grow and the merge is redone - CumulateIntermediate must not fail for lack of slots."""
    import torch
    from query_b200 import dist as qd
    docs = make_docs(6000, seed=91)
    where, keys = None, [F("h")]   # a high-cardinality key: hash table mode
    aggs = ["count(*)", "sum(%s)" % F("p"), "count(distinct %s)" % F("i")]
    small, big = make_table(docs[:8], where, keys, aggs), make_table(docs[8:], where, keys, aggs)
    qd.agree_local([small, big])
    small.seal()
    big.seal()
    qs, qb = q.Query(small, "d", where, keys, aggs), q.Query(big, "d", where, keys, aggs)
    assert qs.info["mode"].startswith("hbm-hash")
    parts = []
    for qq in (qs, qb):
        qq.scan_partial()
        ng, nd, rw = qq.partial_counts()
        recs = torch.empty(max(1, ng) * rw, dtype=torch.int64, device="cuda")
        dents = torch.empty(max(1, nd) * 2, dtype=torch.int64, device="cuda")
        counts, dcounts = qq.partial_export(1, recs.data_ptr(), ng, dents.data_ptr(), nd)
        parts.append((recs[: int(counts[0]) * rw], dents[: int(dcounts[0]) * 2], int(counts[0]), int(dcounts[0])))
    assert parts[1][2] > 2000
    allrec = torch.cat([p[0] for p in parts])
    alld = torch.cat([p[1] for p in parts])
    qs.partial_reset()
    qs.partial_import(allrec.data_ptr(), parts[0][2] + parts[1][2], alld.data_ptr(), parts[0][3] + parts[1][3])
    assert_same(oracle_rows(docs, "d", where, keys, aggs), gpu_rows(qs.finalize(), aggs), "import into a small owner")


def test_prepared_statement_parameters_against_the_oracle():
    """$name / $1 bound at build time (execution.Context.NamedArg / PositionalArg): the same rows as the statement with the
    values written out, for several bindings that all run the one compiled kernel."""
    docs = make_docs(4000, seed=61)
    keys = [F("t")]
    aggs = ["count(*)", "sum(%s)" % F("p"), "min(%s)" % F("s"), "avg((%s + $1))" % F("i")]
    where = "(((%s between $lo and $hi) or (%s in [$a, \"zz\", $b])) and (%s >= $f))" % (F("p"), F("s"), F("f"))
    t = make_table(docs, "(((%s < 1) or (%s = \"x\")) and (%s > 1))" % (F("p"), F("s"), F("f")), keys, ["sum(%s)" % F("i")] + aggs[:3])
    t.seal()
    sources = set()
    for lo, hi, a, b, f, one in [(100, 700, "s3", "s7", -2.5, 1), (-50, 20, "s1", "nope", 0.25, 1), (300, 300, "", "s2", -100, 1), (5, 9, "a", "b", 1, 40)]:
        qq = q.Query(t, "d", where, keys, aggs, params={"lo": lo, "hi": hi, "a": a, "b": b, "f": f, "1": one})
        sources.add(qq.kernel_source)
        lit_where = where.replace("$lo", str(lo)).replace("$hi", str(hi)).replace("$a", json.dumps(a)).replace("$b", json.dumps(b)).replace("$f", repr(f) if isinstance(f, float) else str(f))
        lit_aggs = [x.replace("$1", str(one)) for x in aggs]
        got = {k: {lit_aggs[i]: v for i, v in enumerate(d.values())} for k, d in gpu_rows(qq.execute(), aggs).items()}
        assert_same(oracle_rows(docs, "d", lit_where, keys, lit_aggs), got, "parameters %r" % ((lo, hi, a, b, f, one),))
    # bounds and string constants never change the kernel; the class of $f (int / float) and a constant that feeds the range
    # proof of a sum (avg(i + $1): the proof is part of the generated layout) may
    assert len(sources) <= 3


def test_peer_arena_partitioned_distinct(monkeypatch):
    """BASELINE config 4 across ranks, all driven by this process on one device: every rank partitions its rows' (group,
    value) records into its arena, rank r aggregates partition range r from every rank's records and finalises exactly
    those groups; three steps reuse the single record buffer behind the "consumed" flags."""
    from gen_n1 import config4_docs
    from query_b200 import dist as qd
    monkeypatch.setenv("N1GPU_PART", "1")
    nranks = 3
    docs = config4_docs(24000, 30000, 43)
    where, keys = None, ["(`d`.`g`)"]
    aggs = ["count(distinct (`d`.`x`))", "sum(distinct (`d`.`x`))", "count(*)"]
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
        qq.set_mailbox(mbs[r])
        assert qq.peer_mode == 2 and qq.part_source
        qs.append(qq)
    exp = oracle_rows(docs, "d", where, keys, aggs)
    for step in range(3):
        for qq in qs:
            qq.launch()
        got = {}
        for qq in qs:
            part = gpu_rows(qq.collect(), aggs)
            assert not (set(part) & set(got)), "a group was finalised by two ranks"
            got.update(part)
        assert_same(exp, got, "partitioned distinct over peers, step %d" % step)


@pytest.mark.parametrize("n", [0, 1, 3, 127, 128, 129, 1023, 1024, 1025, 4097])
def test_ragged_sizes(n):
    docs = make_docs(n, seed=100 + n)
    for name, where, keys, aggs in [QUERIES[0], QUERIES[6], QUERIES[33], QUERIES[41], QUERIES[50]]:
        run_both(docs, "d", where, keys, aggs, "%s n=%d" % (name, n))


def test_empty_table_defaults_row():
    """group_final.go:108-117: no keys and no input -> one row of Default() values; with keys -> nothing."""
    t = q.Table(["n"])
    t.append_json([])
    t.seal()
    r = q.Query(t, "d", None, [], ["count(*)", "sum((`d`.`n`))", "avg((`d`.`n`))", "min((`d`.`n`))", "count(distinct (`d`.`n`))"]).execute()
    assert r.rows() == [([], [0, None, None, None, 0])]
    assert q.Query(t, "d", None, ["(`d`.`n`)"], ["count(*)"]).execute().rows() == []


def test_int_sum_overflow_and_sign_semantics():
    """value/integer.go:266-277 through SUM: exact int64 near MaxInt64 (golden integers/case_select.json:33-40),
    overflow -> float64, mixed signs -> float64 (integral, renders as an integer)."""
    def s(xs):
        t = q.Table(["n"])
        t.append_json([json.dumps({"n": x}) for x in xs])
        t.seal()
        return q.Query(t, "d", None, [], ["sum((`d`.`n`))"]).execute().rows()[0][1][0]
    assert s([9223372036854775707, 99, 1]) == 9223372036854775807 and isinstance(s([9223372036854775707, 99, 1]), int)
    v = s([9223372036854775807, 1])
    assert isinstance(v, float) and v == 9.223372036854775808e18
    v = s([5, -3])
    assert isinstance(v, float) and v == 2.0
    assert s([-5, -6]) == -11 and isinstance(s([-5, -6]), int)
    v = s([-9223372036854775808, -1])
    assert isinstance(v, float) and v == -9.223372036854775808e18


def test_preshredded_columns_properties_10m():
    """BASELINE config 2 at full size through size-independent properties: counts add up, SUM is linear over a
    partition of the predicate, MIN/MAX bound the selection, exact against numpy int64 arithmetic."""
    n = 10_000_000
    rng = np.random.default_rng(1)
    nn = rng.integers(0, 1_000_000, n, dtype=np.int64)
    ff = rng.random(n)
    t = q.Table(["n", "f"])
    t.set_column("n", nn)
    t.set_column("f", ff, tags=np.full(n, 5, dtype=np.uint8))
    t.seal()
    aggs = ["count(*)", "count((`d`.`n`))", "sum((`d`.`n`))", "avg((`d`.`n`))", "min((`d`.`n`))", "max((`d`.`n`))", "sum((`d`.`f`))"]
    tot = None
    parts = []
    for lo, hi in [(0, 999_999), (0, 9_999), (10_000, 499_999), (500_000, 999_999)]:
        r = q.Query(t, "d", "((`d`.`n`) between %d and %d)" % (lo, hi), [], aggs).execute().rows()[0][1]
        m = (nn >= lo) & (nn <= hi)
        assert r[0] == int(m.sum()) and r[1] == r[0]
        assert r[2] == int(nn[m].sum())
        assert r[4] == int(nn[m].min()) and r[5] == int(nn[m].max())
        exp_avg = float(int(nn[m].sum())) / float(int(m.sum()))
        assert r[3] == (int(exp_avg) if exp_avg == int(exp_avg) else exp_avg)
        fs = float(np.sum(ff[m]))
        assert abs(r[6] - fs) <= 1e-12 * abs(fs)
        if tot is None:
            tot = r
        else:
            parts.append(r)
    assert sum(p[0] for p in parts) == tot[0]
    assert sum(p[2] for p in parts) == tot[2]
    assert abs(sum(p[6] for p in parts) - tot[6]) <= 1e-12 * tot[6]
    # run-to-run determinism of the float sum (fixed reduction order)
    qq = q.Query(t, "d", None, [], ["sum((`d`.`f`))"])
    a = qq.execute().rows()[0][1][0]
    b = qq.execute().rows()[0][1][0]
    assert a == b


@pytest.mark.parametrize("table_kind,set_kind", [("direct", "bitmap"), ("hash", "bitmap"), ("hash", "hash"), ("direct", "hash"),
                                                 ("direct", "bitmap-8-passes"), ("hash", "bitmap-2-passes")])
def test_preshredded_group_by_high_cardinality_2m(table_kind, set_kind, monkeypatch):
    """1M-group style GROUP BY (BASELINE config 4 shape) checked against numpy: exact counts / int sums / DISTINCT,
    through both group-table layouts (direct-indexed / open addressing) and both DISTINCT set layouts (bitmap / hash)."""
    if table_kind == "hash":
        monkeypatch.setenv("N1GPU_NO_DIRECT", "1")
    if set_kind == "hash":
        monkeypatch.setenv("N1GPU_NO_BITMAP", "1")
    if set_kind.endswith("passes"):  # the sliced bitmap a 200 M-row scan uses, forced at test size
        monkeypatch.setenv("N1GPU_SET_PASSES", set_kind.split("-")[1])
    n = 2_000_000
    rng = np.random.default_rng(3)
    g = rng.integers(0, 200_000, n, dtype=np.int64)
    x = rng.integers(0, 1000, n, dtype=np.int64)
    t = q.Table(["g", "x"])
    t.set_column("g", g)
    t.set_column("x", x)
    t.seal()
    aggs = ["count(*)", "sum((`d`.`x`))", "count(distinct (`d`.`x`))", "sum(distinct (`d`.`x`))", "max((`d`.`x`))"]
    qq = q.Query(t, "d", None, ["(`d`.`g`)"], aggs)
    assert qq.info["mode"] == ("hbm-direct" if table_kind == "direct" else "hbm-hash-64")
    res = qq.execute()
    rows = res.rows()
    order = np.argsort(g, kind="stable")
    gs, xs = g[order], x[order]
    uniq, start = np.unique(gs, return_index=True)
    assert len(rows) == len(uniq)
    cnt = np.diff(np.append(start, n))
    sums = np.add.reduceat(xs, start)
    maxs = np.maximum.reduceat(xs, start)
    pair = np.unique(gs * 1000 + xs)
    pg = pair // 1000
    pv = pair % 1000
    dcount = np.bincount(np.searchsorted(uniq, pg), minlength=len(uniq))
    dsum = np.bincount(np.searchsorted(uniq, pg), weights=pv.astype(np.float64), minlength=len(uniq)).astype(np.int64)
    idx = {int(k): i for i, k in enumerate(uniq)}
    for ks, ag in rows:
        i = idx[ks[0]]
        assert ag == [int(cnt[i]), int(sums[i]), int(dcount[i]), int(dsum[i]), int(maxs[i])]


def test_launch_collect_pipeline_and_rebind():
    n = 100_000
    rng = np.random.default_rng(5)
    tabs = []
    for k in range(2):
        t = q.Table(["n"])
        t.set_column("n", np.arange(n, dtype=np.int64) if k == 0 else np.arange(n, dtype=np.int64)[::-1].copy())
        t.seal()
        tabs.append(t)
    qq = q.Query(tabs[0], "d", "((`d`.`n`) < 1000)", [], ["count(*)", "sum((`d`.`n`))"])
    before = q.launch_count()
    qq.launch()
    r0 = qq.collect().rows()
    qq.rebind(tabs[1])
    r1 = qq.execute().rows()
    assert r0 == r1 == [([], [1000, 499500])]
    assert q.launch_count() - before >= 2  # an ungrouped step is exactly one kernel launch (nq_scan)
    assert qq.last_scan_ns > 0


def test_multi_rank_partial_merge_single_gpu():
    """The Intermediate->Final exchange (group_intermediate.go:56-104) emulated on one GPU: two 'ranks' scan
    half the rows each, export owner-bucketed records to device buffers, the owners import and finalise; the
    union of the owners' groups equals the single-scan result.  (NCCL only moves the buffers.)"""
    import torch
    docs = make_docs(6000, seed=77)
    for name, where, keys, aggs in [QUERIES[0], QUERIES[33], QUERIES[40], QUERIES[41], QUERIES[43], QUERIES[49], QUERIES[50], QUERIES[53]]:
        full = make_table(docs, where, keys, aggs)
        halves = [make_table(docs[:3000], where, keys, aggs), make_table(docs[3000:], where, keys, aggs)]
        # global dictionaries + statistics so every rank compiles the same kernel (n1gpu_table_dict_*/stats_*)
        for c in range(len(full.columns)):
            merged = sorted(set(halves[0].dictionary(c)) | set(halves[1].dictionary(c)))
            st = [h.stats(c) for h in halves]
            g = st[0].copy()
            g[0] = st[0][0] | st[1][0]
            has = [s[1] != 0 for s in st]
            g[1] = int(any(has))
            mins = [s[2] for s, h in zip(st, has) if h]
            maxs = [s[3] for s, h in zip(st, has) if h]
            g[2] = min(mins) if mins else 0
            g[3] = max(maxs) if maxs else 0
            g[4] = st[0][4] | st[1][4]
            g[5] = len(merged)
            for h in halves:
                h.import_dictionary(c, merged)
                h.set_stats(c, g)
        full.seal()
        exp = gpu_rows(q.Query(full, "d", where, keys, aggs).execute(), aggs)
        assert_same(oracle_rows(docs, "d", where, keys, aggs), exp, name)
        qs = []
        for h in halves:
            h.seal()
            qq = q.Query(h, "d", where, keys, aggs)
            qq.scan_partial()
            qs.append(qq)
        nranks = 2
        exported = []
        for qq in qs:
            ng, nd, rw = qq.partial_counts()
            recs = torch.zeros(max(1, ng) * rw, dtype=torch.int64, device="cuda")
            dents = torch.zeros(max(1, nd) * 2, dtype=torch.int64, device="cuda")
            counts, dcounts = qq.partial_export(nranks, recs.data_ptr(), ng, dents.data_ptr(), nd)
            assert counts.sum() == ng and dcounts.sum() == nd
            exported.append((recs, dents, counts, dcounts, rw))
        got = {}
        for owner in range(nranks):
            qq = qs[owner]
            qq.partial_reset()
            for recs, dents, counts, dcounts, rw in exported:
                o = int(counts[:owner].sum())
                do = int(dcounts[:owner].sum())
                r = recs[o * rw:(o + int(counts[owner])) * rw].contiguous()
                d = dents[do * 2:(do + int(dcounts[owner])) * 2].contiguous()
                qq.partial_import(r.data_ptr() if counts[owner] else 0, int(counts[owner]), d.data_ptr() if dcounts[owner] else 0, int(dcounts[owner]))
            part = gpu_rows(qq.finalize(), aggs)
            assert not (set(part) & set(got)), "a group was finalised by two owners"
            got.update(part)
        assert_same(exp, got, name + " (2-rank merge)")
