"""Refresh of a resident directory keyspace after document writes (execution.cpp refresh_table, Table::splice): only the
changed documents are read again and spliced into the HBM columns.  After every mutation the operator must give what the
oracle computes over the current documents, and what a load from scratch of a copy of the directory gives - with the same
dictionaries, statistics and widths, so the cold build compiles no kernel the refreshed one did not."""
import json
import os
import random
import shutil
import subprocess
import sys
import time

import pytest

import query_b200 as q
from gen_n1 import F, make_docs
from plans_n1 import explain_plan
from util_n1 import assert_same, gpu_rows, oracle_rows, write_keyspace

pytestmark = pytest.mark.gpu

RACY_SLEEP = 0.06  # past the 20 ms racily-clean margin of the operator
WHERE = None
KEYS = [F("t")]
AGGS = sorted({"count(*)", "sum(%s)" % F("p"), "min(%s)" % F("s"), "max(%s)" % F("s"), "count(distinct %s)" % F("h"),
               "avg(%s)" % F("f"), "sum(%s)" % F("i"), "max(%s)" % F("i")})


def current_docs(d):
    """The documents of a file-datastore keyspace directory as the primary scan + fetch see them: sorted entries, each
    reads <name minus its last extension>.json, a missing one is no document."""
    out = []
    for name in sorted(os.listdir(d)):
        if os.path.isdir(os.path.join(d, name)):
            continue
        base = name.rsplit(".", 1)[0] if "." in name else name
        try:
            with open(os.path.join(d, base + ".json"), "rb") as f:
                out.append(f.read().decode("utf-8", "surrogateescape"))
        except (FileNotFoundError, IsADirectoryError):
            pass
    return out


class Keyspace:
    def __init__(self, tmp_path, docs, where=WHERE, keys=KEYS, aggs=AGGS, sleep=True):
        self.tmp = tmp_path
        self.root = str(tmp_path / "ds")
        self.dir = write_keyspace(self.root, "default", "d", docs)
        self.where, self.keys, self.aggs = where, keys, aggs
        self.plan = explain_plan("default", "d", "d", where, keys, aggs)
        self.copies = 0
        if sleep:
            time.sleep(RACY_SLEEP)

    def path(self, key):
        return os.path.join(self.dir, key)

    def put(self, key, text):
        with open(self.path(key if "." in key else key + ".json"), "w", encoding="utf-8") as f:
            f.write(text)

    def delete(self, key):
        os.remove(self.path(key if "." in key else key + ".json"))

    def operator(self, root=None):
        return q.Operator(self.plan, root or self.root)

    def check(self, docs_read, sleep=True):
        """The refreshed operator against the oracle and against a cold load of a copy; returns its rows."""
        if sleep:
            time.sleep(RACY_SLEEP)
        op = self.operator()
        got = gpu_rows(op.run_once(), self.aggs)
        stats = op.marshal_json().get("#stats", {})
        assert stats.get("#docsRead") == (docs_read or None), stats
        docs = current_docs(self.dir)
        assert_same(oracle_rows(docs, "d", self.where, self.keys, self.aggs), got, "refreshed vs oracle")
        self.copies += 1
        cold_root = str(self.tmp / ("cold%d" % self.copies))
        shutil.copytree(self.root, cold_root)
        compiled = q.jit_stats()[0]
        cold = self.operator(cold_root)
        cold_rows = gpu_rows(cold.run_once(), self.aggs)
        assert q.jit_stats()[0] == compiled, "the cold load compiled another kernel: its statistics or dictionaries differ"
        assert cold.marshal_json()["kernel"] == op.marshal_json()["kernel"]
        assert_same(cold_rows, got, "refreshed vs cold")
        return got


def docs_of(n, seed):
    return [("k%05d" % i, t) for i, t in enumerate(make_docs(n, seed=seed))]


@pytest.fixture(autouse=True)
def _device():
    q.init(0)


def test_update_in_place_same_size(tmp_path):
    ks = Keyspace(tmp_path, docs_of(400, 1))
    ks.check(400)
    old = open(ks.path("k00010.json")).read()
    new = json.dumps({"t": "t1", "p": 7, "s": "abc", "i": 3})
    assert len(new) <= len(old)
    ks.put("k00010", new + " " * (len(old) - len(new)))  # trailing white space: the same size
    ks.check(1)


def test_inserts_first_middle_last(tmp_path):
    ks = Keyspace(tmp_path, docs_of(300, 2))
    ks.check(300)
    ks.put("a0000", '{"t": "first", "p": 1, "s": "zz"}')
    ks.put("k00150x", '{"t": "t3", "p": 2}')
    ks.put("z9999", '{"t": "last", "i": -4, "h": 12}')
    ks.check(3)


def test_deletes_then_empty_then_inserts(tmp_path):
    ks = Keyspace(tmp_path, docs_of(50, 3))
    ks.check(50)
    for k in ("k00000", "k00025", "k00049"):
        ks.delete(k)
    ks.check(0)
    for name in os.listdir(ks.dir):
        os.remove(ks.path(name))
    ks.check(0)
    ks.put("n1", '{"t": "x", "p": 3}')
    ks.put("n2", '{"t": "y", "s": "b"}')
    ks.check(2)


def test_new_string_sorts_before_every_rank(tmp_path):
    ks = Keyspace(tmp_path, docs_of(200, 4))
    ks.check(200)
    ks.put("k00100", '{"t": "\\u0001 first of all", "s": "", "p": 9}')
    ks.put("k00101", '{"t": "!", "s": " "}')
    ks.check(2)


def test_dictionary_shrinks_across_a_power_of_two(tmp_path):
    # 17 distinct keys -> 16: the key takes one bit less
    docs = [("k%03d" % i, '{"t": "g%02d", "p": %d}' % (i % 17, i)) for i in range(170)]
    ks = Keyspace(tmp_path, docs)
    ks.check(170)
    for i in range(170):
        if i % 17 == 16:
            ks.delete("k%03d" % i)
    ks.check(0)
    ks.put("k016", '{"t": "g16", "p": 1}')
    ks.check(1)


def test_strings_column_gains_and_loses_a_number(tmp_path):
    docs = [("k%03d" % i, '{"t": "t%d", "s": "v%d", "p": %d}' % (i % 5, i % 7, i)) for i in range(100)]
    ks = Keyspace(tmp_path, docs)
    ks.check(100)
    ks.put("k050", '{"t": 5, "s": 2.5, "p": 1}')  # width 4 -> 8
    ks.check(1)
    ks.put("k050", '{"t": "t0", "s": "v0", "p": 1}')  # and back to 4
    ks.check(1)


def test_column_becomes_all_missing(tmp_path):
    docs = [("k%03d" % i, '{"t": "t%d", "i": %d}' % (i % 3, i) if i % 10 else '{"t": "t1"}') for i in range(60)]
    ks = Keyspace(tmp_path, docs)
    ks.check(60)
    for i in range(0, 60):
        if i % 10:
            ks.put("k%03d" % i, '{"t": "t%d"}' % (i % 3))
    ks.check(54)


def test_int_range_growth(tmp_path):
    docs = [("k%03d" % i, '{"t": "t%d", "p": %d, "i": %d}' % (i % 4, i, i - 50)) for i in range(100)]
    ks = Keyspace(tmp_path, docs)
    ks.check(100)
    ks.put("k001", '{"t": "t1", "p": %d, "i": %d}' % (2 ** 62, -(2 ** 62)))
    ks.check(1)
    ks.put("k001", '{"t": "t1", "p": 1, "i": 0}')
    ks.check(1)


def test_invalid_json_and_host_fixups(tmp_path):
    ks = Keyspace(tmp_path, docs_of(200, 5))
    ks.check(200)
    ks.put("k00003", '{"t": "t1", "p": 4,')  # invalid: every field MISSING
    ks.put("k00004", '{"t": "esc\\"aped\\u00e9", "p": 123456789012345678901234, "s": "tab\\there"}')  # host fix-up
    ks.put("k00005", '{"t\\u0031": "t1", "t": "t2", "i": 5}')  # an escaped field name: host fix-up
    ks.check(3)


def test_array_value_is_ineligible_both_ways(tmp_path):
    ks = Keyspace(tmp_path, docs_of(100, 6))
    ks.check(100)
    ks.put("k00007", '{"t": ["a", "b"], "p": 1}')
    time.sleep(RACY_SLEEP)
    with pytest.raises(q.N1GpuError) as e1:
        ks.operator()
    shutil.copytree(ks.root, str(tmp_path / "cold"))
    with pytest.raises(q.N1GpuError) as e2:
        ks.operator(str(tmp_path / "cold"))
    assert e1.value.code == e2.value.code == -3
    ks.put("k00007", '{"t": "a", "p": 1}')
    ks.check(1)


def test_txt_next_to_json_then_json_deleted(tmp_path):
    ks = Keyspace(tmp_path, docs_of(20, 7) + [("a", '{"t": "a-doc", "p": 5}')], sleep=False)
    ks.put("a.txt", "not a document")  # a second row of a.json
    ks.check(22)
    ks.delete("a")  # a.txt now stands for no document: read again, nothing found
    ks.check(0)


def test_directory_touch_and_identical_rewrite(tmp_path):
    ks = Keyspace(tmp_path, docs_of(150, 8))
    ks.check(150)
    os.utime(ks.dir, None)
    ks.check(0)
    text = open(ks.path("k00011.json")).read()
    ks.put("k00011", text)
    ks.check(1)


def test_racy_write_is_read_again(tmp_path):
    ks = Keyspace(tmp_path, [("k%03d" % i, '{"t": "t%d", "p": %d}' % (i % 7, i % 10)) for i in range(100)])
    ks.check(100)
    ks.put("k020", '{"t": "t9", "p": 5}')  # same size as before
    op = ks.operator()  # no sleep: the rewrite is racily clean
    assert op.marshal_json()["#stats"].get("#docsRead") == 1
    ks.put("k020", '{"t": "t8", "p": 4}')  # within the same timestamp tick its stat need not change
    ks.check(1)


def test_two_column_sets_and_an_operator_built_before(tmp_path):
    ks = Keyspace(tmp_path, docs_of(300, 10))
    other = explain_plan("default", "d", "d", "(%s < 500)" % F("p"), [F("g")], ["count(*)", "sum(%s)" % F("i")])
    ks.check(300)
    q.Operator(other, ks.root)
    before_docs = current_docs(ks.dir)
    before = ks.operator()
    ks.put("k00001", '{"t": "fresh", "g": 3, "p": 2, "i": 9}')
    ks.delete("k00002")
    ks.check(1)
    time.sleep(RACY_SLEEP)
    op = q.Operator(other, ks.root)
    assert op.marshal_json()["#stats"].get("#docsRead") == 1
    assert_same(oracle_rows(current_docs(ks.dir), "d", "(%s < 500)" % F("p"), [F("g")], ["count(*)", "sum(%s)" % F("i")]),
                gpu_rows(op.run_once(), ["count(*)", "sum(%s)" % F("i")]), "second column set")
    assert_same(oracle_rows(before_docs, "d", WHERE, KEYS, AGGS), gpu_rows(before.run_once(), AGGS), "operator built before")


def test_random_mutation_fuzz(tmp_path):
    rnd = random.Random(20)
    pool = make_docs(400, seed=21)
    ks = Keyspace(tmp_path, docs_of(200, 22))
    ks.check(200)
    live = set("k%05d" % i for i in range(200))
    for _ in range(20):
        changed = set()
        for _ in range(rnd.choice([1, 2, 5, 20])):
            r = rnd.random()
            k = rnd.choice(sorted(live)) if live and r < 0.4 or r >= 0.7 else "k%05d" % rnd.randint(0, 400)
            if r >= 0.7 and live:
                live.discard(k)
                changed.discard(k)
                ks.delete(k)
            elif r < 0.7:
                live.add(k)
                changed.add(k)
                ks.put(k, rnd.choice(pool))
        time.sleep(RACY_SLEEP)
        op = ks.operator()
        assert op.marshal_json().get("#stats", {}).get("#docsRead", 0) == len(changed)
        got = gpu_rows(op.run_once(), AGGS)
        assert_same(oracle_rows(current_docs(ks.dir), "d", WHERE, KEYS, AGGS), got, "fuzz")
    ks.check(0)


def test_segment_written_from_the_refreshed_table(tmp_path):
    segs = str(tmp_path / "segments")
    os.makedirs(segs)
    q.set_segment_dir(segs)
    try:
        ks = Keyspace(tmp_path, docs_of(500, 23))
        ks.check(500)
        ks.put("k00100", '{"t": "new", "p": 77, "s": "q"}')
        ks.delete("k00200")
        got = ks.check(1)
        script = (
            "import json, sys\n"
            "sys.path[:0] = [%r, %r]\n"
            "import query_b200 as q\n"
            "from util_n1 import gpu_rows\n"
            "q.init(0)\n"
            "q.set_segment_dir(%r)\n"
            "op = q.Operator(json.loads(%r), %r)\n"
            "rows = gpu_rows(op.run_once(), json.loads(%r))\n"
            "print(json.dumps({'stats': op.marshal_json().get('#stats', {}), 'rows': [[list(k), v] for k, v in sorted(rows.items())]}))\n"
        ) % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.dirname(os.path.abspath(__file__)), segs,
             json.dumps(ks.plan), ks.root, json.dumps(AGGS))
        out = subprocess.run([sys.executable, "-c", script], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-3000:]
        res = json.loads(out.stdout.strip().splitlines()[-1])
        assert "#docsRead" not in res["stats"]  # loaded from the segment: no document read
        fresh = {tuple(k): v for k, v in res["rows"]}
        assert_same(got, fresh, "fresh process from the segment")
    finally:
        q.set_segment_dir("")
