#!/usr/bin/env python
"""Digest of what the scan-kernel generator (query_b200/csrc/codegen.cpp) produces for the test statements under the
layout knobs: one line per case, `<case> <knob setting> <sha256 prefix>` over the kernel text, the partition kernel
text, the plan info and the word ops.  Needs no GPU (NVRTC still compiles the kernels).  A change that must leave the
generated kernels alone is checked by running it at both commits and diffing the outputs."""
import hashlib
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import query_b200 as q  # noqa: E402
import test_in_sets as ins  # noqa: E402
import test_int_edges as ie  # noqa: E402
from gen_n1 import QUERIES, config4_docs, make_docs  # noqa: E402
from util_n1 import make_table  # noqa: E402
from workloads import Config2, Config3, Config4, Config5  # noqa: E402

# the settings of test_grouped_matrix_through_the_alternate_layouts (tests/test_gpu_parity.py), N1GPU_NO_PRIV, and the
# remaining layout knobs of the generator
KNOBS = ["", "N1GPU_NO_DIRECT", "N1GPU_NO_BITMAP", "N1GPU_NO_OFFSET_PACK", "N1GPU_NO_CACHE", "N1GPU_NO_PACK",
         "N1GPU_NO_KEY32", "N1GPU_NO_COMPLEMENT", "N1GPU_CACHE_BLOCK=1024", "N1GPU_CACHE_BLOCK=256", "N1GPU_SET_PASSES=4",
         "N1GPU_NO_FCARRY", "N1GPU_NO_TIGHT", "N1GPU_PART", "N1GPU_NO_WIDE1", "N1GPU_NO_SIGN_FROM_MINMAX",
         "N1GPU_PRIV_BLOCK=640", "N1GPU_PRIV_BLOCK=96", "N1GPU_NO_MM_PAIR", "N1GPU_NO_PRIV",
         "N1GPU_MIN_BLOCKS=4", "N1GPU_CACHE_KB=2", "N1GPU_NO_PART"]
SEEN = set()
ENV = types.SimpleNamespace(setenv=os.environ.__setitem__, delenv=os.environ.pop)  # pytest's monkeypatch, for test helpers


def digest(case, setting, make):
    env = dict(kv.partition("=")[::2] for kv in setting.split(",") if kv)
    os.environ.update({k: v or "1" for k, v in env.items()})
    try:
        qq = make()
        h = hashlib.sha256("\0".join([qq.kernel_source, qq.part_source, repr(qq.info), repr(qq.word_ops())]).encode()).hexdigest()[:16]
    except Exception as e:  # noqa: BLE001 - an ineligible shape is part of the output
        h = "ERR %s: %s" % (type(e).__name__, (str(e).splitlines() or [""])[0])
    finally:
        for k in env:
            os.environ.pop(k)
    SEEN.add(h)
    print(case, setting or "-", h, flush=True)


def config_tables(rng, n=20000):
    """configs 2-5's columns at n rows, with their full-size row counts declared (layout decisions read them)"""
    absent = lambda present: np.where(rng.integers(0, 10, n) < 2, rng.integers(0, 2, n), present).astype(np.uint8)
    t2 = q.Table(["n", "f"])
    t2.set_column("n", rng.integers(0, 1_000_000, n))
    t2.set_column("f", (rng.integers(1, 1_000_000, n) / 1e6).view(np.int64), tags=np.full(n, 5, np.uint8))
    t3 = q.Table(["l_shipdate", "l_returnflag", "l_linestatus", "l_quantity", "l_extendedprice", "l_discount", "l_tax"])
    t3.set_column("l_shipdate", rng.integers(0, len(Config3.DATES), n).astype(np.uint32), dictionary=Config3.DATES)
    t3.set_column("l_returnflag", rng.integers(0, 3, n).astype(np.uint32), dictionary=["A", "N", "R"])
    t3.set_column("l_linestatus", rng.integers(0, 2, n).astype(np.uint32), dictionary=["F", "O"])
    t3.set_column("l_quantity", rng.integers(1, 51, n))
    for c, hi in (("l_extendedprice", 10500000), ("l_discount", 11), ("l_tax", 9)):  # hundredths; whole ones are INT
        v = rng.integers(0, hi, n)
        t3.set_column(c, np.where(v % 100 == 0, v // 100, (v / 100.0).view(np.int64)), tags=np.where(v % 100 == 0, 4, 5).astype(np.uint8))
    t4 = q.Table(["g", "x"])
    t4.set_column("g", rng.integers(0, 1_000_000, n))
    t4.set_column("x", rng.integers(0, 1000, n))
    t5 = q.Table(["k", "v"])
    t5.set_column("k", rng.integers(0, 100_000, n).astype(np.uint32), tags=absent(6), dictionary=["w%06d" % i for i in range(100_000)])
    t5.set_column("v", rng.integers(-1000, 1_000_000, n), tags=absent(4))
    for cfg, t in ((Config2, t2), (Config3, t3), (Config4, t4), (Config5, t5)):
        t.set_global_rows(cfg.rows)
        t.seal()
        yield cfg, t


def main():
    docs = make_docs(3000, seed=22)
    for name, where, keys, aggs in QUERIES:
        t = make_table(docs, where, keys, aggs)
        t.seal()
        for k in KNOBS:
            digest(name, k, lambda: q.Query(t, "d", where, keys, aggs))
    for cfg, t in config_tables(np.random.default_rng(1)):
        for k in KNOBS:
            digest(cfg.name, k, lambda: q.Query(t, cfg.alias, cfg.where, list(cfg.keys), list(cfg.aggs)))
    for name in ie.VALUE_FIXTURES + ie.MM_FIXTURES:
        for layout, (keys, env, *_) in ie.LAYOUTS.items():
            fx = ie.fixture(name)
            digest("int_edges:%s:%s" % (name, layout), ",".join(map("=".join, env.items())),
                   lambda: q.Query(fx.table, "d", None, [ie.K(c) for c in keys], ie._layout_aggs(fx, layout)))
    for near_min in (True, False):
        for layout, (env, _) in ie.DISTINCT_LAYOUTS.items():
            digest("int_edges:distinct_%d:%s" % (near_min, layout), ",".join(map("=".join, env.items())),
                   lambda: q.Query(ie.distinct_fixture(near_min).table, "d", None, ["(`d`.`gk`)"], ie.DAGGS))
    for layout in ins.LAYOUTS:  # $p arrays
        for lists in ins.LAYOUT_LISTS:
            digest("in_sets:%s:%s" % (layout, lists), "", lambda: ins._layout_query(layout, ins.LAYOUT_LISTS[lists], ENV)[0])
    for oname, x in ins.OPERANDS.items():  # $p arrays, and literal lists over IN_CHAIN_MAX where an element is MISSING
        for lname, vals in ins.LISTS.items():
            for where, key, aggs in ((None, "(%s in $p)" % x, ["count(*)", "sum(%s)" % ins.F("i")]),
                                     ("(not (%s in $p))" % x, None, ["count(*)", "sum(%s)" % ins.F("p"), "min(%s)" % ins.F("m")])):
                text, params, olit = ins._bind(where or key, "p", vals())
                t = ins._table(ins._docs(), olit if where else None, [] if where else [olit], aggs)
                digest("in_sets:%s:%s:%s" % (oname, lname, "where" if where else "key"), "",
                       lambda: q.Query(t, "d", text if where else None, [] if where else [text], aggs, params=params))
    vals = list(range(0, 1000, 3)) + [-1, 2.5]
    t = make_table(config4_docs(30000, 20000, 5), "((`d`.`x`) in %s)" % ins.lit_list(vals), ["(`d`.`g`)"], ["count(distinct (`d`.`x`))"])
    t.set_global_rows(1 << 31)
    t.seal()
    for k in KNOBS:
        digest("in_sets:distinct", k, lambda: q.Query(t, "d", "((`d`.`x`) in $p)", ["(`d`.`g`)"],
                                                      ["count(distinct (`d`.`x`))", "sum(distinct (`d`.`x`))", "count(*)"], params={"p": vals}))
    print("# %d distinct digests" % len(SEEN), file=sys.stderr)


if __name__ == "__main__":
    main()
