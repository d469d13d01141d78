"""GROUP BY keys wider than 127 bits: the `hbm-hash-wide` table (KW = ceil(key bits / 64) key words per group).

A numeric column that holds INT and FLOAT rows packs as a class bit plus 64 payload bits, so two such columns (TPC-H's
`l_discount, l_tax` as whole and fractional hundredths) or two unbounded int64 columns already need 128-132 bits.  The
CPU tests pin where each key width lands and that every kernel compiles; the GPU tests compare every group, bit-exact, with
the oracle: contention on one slot, a thousand groups, every row its own group, the owner-record exchange with growth of
an owner's table, and the plan-level operator.
"""
import json
import random
import re
import tempfile

import numpy as np
import pytest

import query_b200 as q
from oracle import n1ql_oracle as O
from gen_n1 import ALL_AGGS_ON, F
from plans_n1 import explain_plan
from util_n1 import assert_same, gpu_rows, make_table, oracle_rows, write_keyspace

I64_MIN, I64_MAX = -(1 << 63), (1 << 63) - 1
T_MISSING, T_NULL, T_INT, T_FLOAT = 0, 1, 4, 5
AGGS = ["count(*)"] + ALL_AGGS_ON(F("v"))[1:] + ["min(%s)" % F("k0"), "max(%s)" % F("k1")]


# ---- where a key width lands (no GPU) ----------------------------------------------------------------------------------
def _int_table(widths, rows=256, seed=3):
    """one INT column per width: 64 = unbounded int64 (both limits occur), w < 63 = the range [0, 2^w - 1] (biased key)"""
    rng = np.random.default_rng(seed)
    t = q.Table(["c%d" % i for i in range(len(widths))])
    for i, w in enumerate(widths):
        if w == 64:
            v = rng.integers(I64_MIN, I64_MAX, rows, dtype=np.int64)
            v[0], v[1] = I64_MIN, I64_MAX
        else:
            v = rng.integers(0, 1 << w, rows, dtype=np.int64)
            v[0], v[1] = 0, (1 << w) - 1
        t.set_column("c%d" % i, v)
    t.seal()
    return t


def _mixed_column(rng, rows, absent):
    """hundredths as TPC-H's discount and tax: whole ones are INT, the others FLOAT; optionally MISSING / NULL rows"""
    v = rng.integers(0, 11, rows)
    tags = np.where(v % 100 == 0, T_INT, T_FLOAT).astype(np.uint8)
    pay = np.where(v % 100 == 0, v // 100, (v / 100.0).view(np.int64))
    if absent:
        tags[rng.integers(0, 10, rows) == 0] = T_MISSING
        tags[rng.integers(0, 10, rows) == 1] = T_NULL
    return pay, tags


WIDTHS = {  # key bits -> the columns that pack into them
    127: [64, 62, 1],
    128: [64, 64],
    129: [64, 64, 1],
    191: [64, 64, 62, 1],
    192: [64, 64, 64],
    193: [64, 64, 64, 1],
}


@pytest.mark.parametrize("bits", list(WIDTHS))
def test_key_width_selects_the_table(bits):
    t = _int_table(WIDTHS[bits])
    qq = q.Query(t, "d", None, ["(`d`.`c%d`)" % i for i in range(len(WIDTHS[bits]))], ["count(*)", "sum((`d`.`c0`))"])
    src = qq.kernel_source
    if bits <= 127:
        assert qq.info["mode"] == "hbm-hash-128" and "table_insert128(" in src
    else:
        kw = (bits + 63) // 64
        assert qq.info["mode"] == "hbm-hash-wide"
        assert "u64 kwd[%d] = {};" % kw in src and "table_insert_wide<%d>(" % kw in src
        assert "s_ckey" not in src, "a wide key has no front cache"


def _widest_docs(rows=70):
    """16 columns, each holding MISSING, NULL, FALSE, TRUE, INT (both int64 limits), FLOAT and STRING: 3 class bits and
    64 payload bits per component, 1072 bits, 17 key words"""
    vals = [None, False, True, I64_MIN, I64_MAX, 2.5, "s"]
    docs = []
    for i in range(rows):
        d = {}
        for c in range(16):
            j = (i + c) % 8
            if j < 7:
                d["k%d" % c] = vals[j]
        docs.append(json.dumps(d))
    return docs


def test_sixteen_component_key_takes_17_words():
    docs = _widest_docs()
    keys = [F("k%d" % c) for c in range(16)]
    t = make_table(docs, None, keys, ["count(*)"])
    t.seal()
    qq = q.Query(t, "d", None, keys, ["count(*)", "max(%s)" % F("k3")])
    assert qq.info["mode"] == "hbm-hash-wide"
    assert "u64 kwd[17] = {};" in qq.kernel_source and "table_insert_wide<17>(" in qq.kernel_source


def test_wide_key_with_distinct_stays_ineligible():
    t = _int_table([64, 64])
    with pytest.raises(q.Ineligible, match=r"DISTINCT entry needs \d+ bits \(> 127\)"):
        q.Query(t, "d", None, ["(`d`.`c0`)", "(`d`.`c1`)"], ["count(*)", "count(distinct (`d`.`c0`))"])


@pytest.mark.parametrize("absent,bits", [(False, 130), (True, 132)])
def test_mixed_int_float_keys_are_eligible(absent, bits):
    rng = np.random.default_rng(5)
    t = q.Table(["l_discount", "l_tax"])
    for c in ("l_discount", "l_tax"):
        pay, tags = _mixed_column(rng, 4096, absent)
        t.set_column(c, pay, tags=tags)
    t.seal()
    qq = q.Query(t, "l", None, ["(`l`.`l_discount`)", "(`l`.`l_tax`)"], ["count(*)", "sum((`l`.`l_tax`))"])
    assert qq.info["mode"] == "hbm-hash-wide"
    assert "u64 kwd[3] = {};" in qq.kernel_source
    assert sum(map(int, re.findall(r"pack_bits\(kwd, kpos, .*, (\d+)\);", qq.kernel_source))) == bits


# ---- against the oracle (GPU) -------------------------------------------------------------------------------------------
_POOL = [I64_MIN, I64_MAX, 0, -0.0, 1, -1, 2.5, -1e300, "a", "zz", True, None]


def _key_value(rnd, distinct_id=None):
    if distinct_id is not None:  # an odd multiplier permutes the int64 range: distinct, and spread over all of it
        return (distinct_id * 0x9E3779B97F4A7C15) % (1 << 64) - (1 << 63)
    r = rnd.random()
    if r < 0.08:
        return O.MISSING
    if r < 0.5:
        return rnd.choice(_POOL)
    return rnd.choice([rnd.randint(I64_MIN, I64_MAX), rnd.uniform(-1e6, 1e6)])


_OUTLIERS = [[I64_MAX, 1.5, 2.5, None], ["s", I64_MAX, -1.0, I64_MIN]]


def wide_docs(n, nkeys, groups, seed):
    """groups: "one" (every row the same key, 0 and -0.0 alternating, but for two rows whose outlying values make the
    column statistics wide and whose f the filter drops), "thousand" (a pool of 1000 key tuples), "distinct" (every row
    its own group).  The value column v mixes INT, FLOAT, STRING, NULL and MISSING (the int64 limits are in the keys, and
    MIN / MAX over keys aggregate them: a float SUM over them would depend on the order of the additions); f filters."""
    rnd = random.Random(seed)
    pool = [[_key_value(rnd) for _ in range(nkeys)] for _ in range(1000)]
    docs = []
    for i in range(n):
        if groups == "one":
            ks = (_OUTLIERS[i] if i < 2 else [I64_MIN, -0.0 if i % 2 else 0, "x", I64_MAX])[:nkeys]
        elif groups == "thousand":
            ks = pool[rnd.randrange(1000)]
        else:
            ks = [_key_value(rnd, i)] + [_key_value(rnd) for _ in range(nkeys - 1)]
        d = {"k%d" % c: v for c, v in enumerate(ks) if v is not O.MISSING}
        r = rnd.random()
        if r < 0.05:
            pass
        elif r < 0.1:
            d["v"] = None
        elif r < 0.15:
            d["v"] = rnd.choice(["s", "t"])
        elif r < 0.6:
            d["v"] = rnd.randint(-10 ** 6, 10 ** 6)
        else:
            d["v"] = rnd.randint(-4000, 4000) / 4  # quarters: float sums are exact in any order
        d["f"] = 99 if groups == "one" and i < 2 else rnd.randint(0, 99)
        docs.append(json.dumps(d))
    return docs


def _keys(nkeys):
    return [F("k%d" % c) for c in range(nkeys)]


@pytest.fixture(scope="module")
def _device():
    q.init(0)


@pytest.mark.gpu
@pytest.mark.parametrize("where", [None, "(%s < 60)" % F("f")], ids=["all", "filter"])
@pytest.mark.parametrize("groups,n", [("one", 20000), ("thousand", 20000), ("distinct", 100000)])
@pytest.mark.parametrize("nkeys", [2, 3, 4])
def test_wide_groups_match_the_oracle(nkeys, groups, n, where, _device):
    docs = wide_docs(n, nkeys, groups, seed=nkeys * 10 + len(groups))
    keys = _keys(nkeys)
    aggs = AGGS
    t = make_table(docs, where, keys, aggs)
    t.seal()
    qq = q.Query(t, "d", where, keys, aggs)
    assert qq.info["mode"] == "hbm-hash-wide"
    got = gpu_rows(qq.execute(), aggs)
    exp = oracle_rows(docs, "d", where, keys, aggs)
    if groups == "one":
        assert len(exp) == (1 if where else 3)
    assert_same(exp, got, "%d wide keys, %s" % (nkeys, groups))
    t2 = make_table(docs, where, keys, aggs)  # a rebound query runs the same kernel over another copy of the table
    t2.seal()
    qq.rebind(t2)
    assert_same(exp, gpu_rows(qq.execute(), aggs), "rebound")


@pytest.mark.gpu
def test_million_distinct_int64_keys(_device):
    """every one of 10^6 rows its own group of three unbounded int64 keys: the table grows (x4 and rerun) past its
    first capacity, and every group's count, sum, min and max is the row's own value"""
    n = 1_000_000
    rng = np.random.default_rng(11)
    a = rng.permutation(n).astype(np.int64) * 9_223_372_036_001 + I64_MIN  # distinct, from INT64_MIN up
    b, c = rng.integers(I64_MIN, I64_MAX, n, dtype=np.int64), rng.integers(I64_MIN, I64_MAX, n, dtype=np.int64)
    t = q.Table(["a", "b", "c"])
    for name, v in (("a", a), ("b", b), ("c", c)):
        t.set_column(name, v)
    t.seal()
    K = ["(`d`.`a`)", "(`d`.`b`)", "(`d`.`c`)"]
    qq = q.Query(t, "d", None, K, ["count(*)", "sum((`d`.`b`))", "min((`d`.`c`))", "max((`d`.`a`))"])
    assert qq.info["mode"] == "hbm-hash-wide"
    kc, kv, ac, av, _ = qq.execute().arrays()
    assert kc.size == 3 * n and (kc == T_INT).all() and (ac == T_INT).all()
    kv, av = kv.reshape(n, 3), av.reshape(n, 4)
    got, want = kv[np.argsort(kv[:, 0])], np.argsort(a)
    av = av[np.argsort(kv[:, 0])]
    assert (got[:, 0] == a[want]).all() and (got[:, 1] == b[want]).all() and (got[:, 2] == c[want]).all()
    assert (av[:, 0] == 1).all() and (av[:, 1] == b[want]).all() and (av[:, 2] == c[want]).all() and (av[:, 3] == a[want]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("nranks", [2, 3])
def test_owner_records_of_wide_keys(nranks, _device):
    """partial_export to every owner, partial_import, finalize in one process: the owners' union is the oracle's result,
    each group comes from one owner, and the owner whose own rows are few grows its table for the imported groups"""
    import torch
    docs = wide_docs(9000, 3, "distinct", seed=nranks)
    keys, aggs = _keys(3), AGGS
    parts = [docs[:8]] + [docs[8 + (len(docs) - 8) * r // (nranks - 1): 8 + (len(docs) - 8) * (r + 1) // (nranks - 1)] for r in range(nranks - 1)]
    from query_b200 import dist as qd
    tables = [make_table(p, None, keys, aggs) for p in parts]
    qd.agree_local(tables)
    qs = []
    for t in tables:
        t.seal()
        qq = q.Query(t, "d", None, keys, aggs)
        assert qq.info["mode"] == "hbm-hash-wide"
        qs.append(qq)
    recs_to = [[] for _ in range(nranks)]
    rw = None
    for qq in qs:
        qq.scan_partial()
        ng, nd, rw = qq.partial_counts()
        kw = int(re.search(r"u64 kwd\[(\d+)\]", qq.kernel_source).group(1))
        assert rw == kw + len(qq.word_ops()) and nd == 0  # [k0 .. k(KW-1), words]
        recs = torch.empty(max(1, ng) * rw, dtype=torch.int64, device="cuda")
        dents = torch.empty(2, dtype=torch.int64, device="cuda")
        counts, _ = qq.partial_export(nranks, recs.data_ptr(), ng, dents.data_ptr(), 0)
        at = 0
        for r in range(nranks):
            recs_to[r].append(recs[at * rw: (at + int(counts[r])) * rw])
            at += int(counts[r])
    cap0 = qs[0].info["slots"]
    got = {}
    for r, qq in enumerate(qs):
        mine = torch.cat(recs_to[r])
        qq.partial_reset()
        qq.partial_import(mine.data_ptr(), mine.numel() // rw, 0, 0)
        part = gpu_rows(qq.finalize(), aggs)
        assert not (set(part) & set(got)), "a group was finalised by two owners"
        got.update(part)
    assert qs[0].info["slots"] > cap0, "the small owner's table did not grow"
    assert_same(oracle_rows(docs, "d", None, keys, aggs), got, "%d owners" % nranks)


@pytest.mark.gpu
def test_plan_operator_with_order_by_tail(_device):
    docs = wide_docs(3000, 2, "thousand", seed=4)
    keys, aggs = _keys(2), sorted({"count(*)", "sum(%s)" % F("v"), "max(%s)" % F("f")})
    tail = dict(terms=[(F("k0"), "a"), (F("k1"), "b"), ("count(*)", "n"), ("sum(%s)" % F("v"), "s")],
                order=[("`n`", True), ("`a`", False), ("`b`", False)], limit=50)
    with tempfile.TemporaryDirectory() as root:
        write_keyspace(root, "default", "d", [("k%05d" % i, t) for i, t in enumerate(docs)])
        op = q.Operator(explain_plan("default", "d", "d", None, keys, aggs, tail=tail), root, tail=True)
        assert op.marshal_json()["kernel"]["mode"] == "hbm-hash-wide"
        got = op.run_tail(op.run_once())
    groups = O.run_chain([O.parse_document(t) for t in docs], "d", None, keys, aggs)
    want = O.run_tail(groups, terms=tail["terms"], order=tail["order"], limit=tail["limit"])
    assert got == want  # (numbers compare by value: the operator renders an integral float SUM as Go does, without ".0")
