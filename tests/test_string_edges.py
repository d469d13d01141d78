"""String, boolean and mixed-class values at every dictionary-size threshold, in every table layout and across partitions.

Most layout decisions for a string column come from its dictionary size (query_b200/csrc/codegen.cpp): an offset-packed
string key takes bits_for(nfree + ndict) bits (nfree: the payload-free classes MISSING / NULL / FALSE / TRUE that occur),
and that bit count picks the table (thread-private, shared-memory, direct-indexed or hashed HBM), the mixed-radix slot
count, the 32-bit front-cache keys and the 64 / 128-bit hash.  MIN / MAX of a string keep a rank word; the winner across
classes comes from a `seen:` OR word, or from a counter when only one class occurs.  String constants in WHERE become
2 * rank, or 2 * lower_bound - 1 when absent.  The fixtures here sit on both sides of those thresholds; every result is
compared bit-exact, class included, with a reference that reduces Python values under `O.collate`.

The CPU tests (no `gpu` mark) pin which side of each threshold every fixture lands on, from the generated kernel text.
"""
import functools
import json

import numpy as np
import pytest

import query_b200 as q
from oracle import n1ql_oracle as O
from test_int_edges import assert_exact, exact_aggregates
from util_n1 import gpu_rows

T_MISSING, T_NULL, T_FALSE, T_TRUE, T_INT, T_STRING = 0, 1, 2, 3, 4, 6
M = O.MISSING

X = "(`d`.`x`)"
K = lambda c: "(`d`.`%s`)" % c
AGGS = ["count(*)", "count(%s)" % X, "countn(%s)" % X, "min(%s)" % X, "max(%s)" % X]
NAGGS = AGGS + ["sum(%s)" % X, "avg(%s)" % X]  # operands whose numbers are ints
DAGGS = ["count(*)", "count(distinct %s)" % X]


def utf8_sorted(strings):
    """Bytewise (UTF-8) order: the collation of N1QL strings and the order of every dictionary."""
    return sorted(set(strings), key=lambda s: s.encode("utf-8"))


# Multi-byte UTF-8 (U+FFFF sorts before U+1F600 bytewise, after it in UTF-16), case pairs, prefixes of each other,
# strings sharing their first 8 bytes and differing at byte 8 or 9, and an 8-byte string next to its 9-byte extension.
EDGE_STRINGS = ["A", "Zeta", "zeta", "a", "ab", "abc", "abcdefgh", "abcdefgh\x01", "abcdefgha", "abcdefghb", "abcdefghaa",
                "abcdefghab", "abcdefgi", "café", "cafe", "€", "￿", "\U0001F600", "\U0001F600x", "~"]
DICT = utf8_sorted([""] + EDGE_STRINGS)   # "" is rank 0
DICT_NE = utf8_sorted(EDGE_STRINGS)       # no ""


# ---- exact reference -------------------------------------------------------------------------------------------------
def _vkey(v):
    """Distinct-value identity: True and 1 are different N1QL values."""
    return (type(v).__name__, v)


def string_aggregates(values):
    """{aggregate kind: value} of one group whose operand values are str / bool / int / None / MISSING."""
    present = [v for v in values if v is not None and v is not M]
    ints = [v for v in present if isinstance(v, int) and not isinstance(v, bool)]
    out, _approx = exact_aggregates(ints + [None] * (len(values) - len(ints)))
    out["count"] = len(present)
    cmp = functools.cmp_to_key(O.collate)
    out["min"] = min(present, key=cmp) if present else None
    out["max"] = max(present, key=cmp) if present else None
    out["dcount"] = len({_vkey(v) for v in present})
    return out


def _agg_kind(text):
    if text == "count(*)":
        return "count*"
    if "distinct" in text:
        return "dcount"
    return text.split("(", 1)[0]


def key_text(v):
    return "MISSING" if v is M else json.dumps(v)


# ---- pre-shredded columns --------------------------------------------------------------------------------------------
def encode(values, dictionary):
    """(payload, tags) of Python values: uint32 ranks when no number occurs, else int64 (a string's rank as it is)."""
    rank = {s: i for i, s in enumerate(dictionary)}
    tags = np.zeros(len(values), dtype=np.uint8)
    pay = np.zeros(len(values), dtype=np.int64)
    for i, v in enumerate(values):
        if v is M:
            tags[i] = T_MISSING
        elif v is None:
            tags[i] = T_NULL
        elif isinstance(v, bool):
            tags[i] = T_TRUE if v else T_FALSE
        elif isinstance(v, int):
            tags[i], pay[i] = T_INT, v
        else:
            tags[i], pay[i] = T_STRING, rank[v]
    return (pay if (tags == T_INT).any() else pay.astype(np.uint32)), tags


class Fixture:
    def __init__(self, name, rows, xdict, keys, global_rows=None, import_dict=None):
        """rows: [(group id, x value)]; keys: {column: (values per group id, dictionary or None)}."""
        self.name, self.xdict, self.keys, self.global_rows, self.import_dict = name, xdict, keys, global_rows, import_dict
        self.gid = [g for g, _v in rows]
        self.x = [v for _g, v in rows]

    def columns(self):
        cols = {"x": (self.x, self.xdict)}
        for c, (per_group, d) in self.keys.items():
            cols[c] = ([per_group[g] for g in self.gid], d)
        return cols

    @functools.cached_property
    def table(self):
        t = q.Table(sorted(self.columns()))
        for c, (vals, d) in self.columns().items():
            pay, tags = encode(vals, d or [])
            t.set_column(c, pay, tags=tags, dictionary=d)
        if self.import_dict is not None:
            t.import_dictionary("x", self.import_dict)
        if self.global_rows is not None:
            t.set_global_rows(self.global_rows)
        t.seal()
        return t

    def expected(self, keys, aggs):
        by = {}
        for g, v in zip(self.gid, self.x):
            by.setdefault(g if keys else 0, []).append(v)
        out = {}
        for g, vs in by.items():
            k = tuple(key_text(self.keys[c][0][g]) for c in keys)
            r = string_aggregates(vs)
            out[k] = ({a: r[_agg_kind(a)] for a in aggs}, False)
        return out


def shuffled(groups, seed):
    """groups: {group id: [x values]} -> rows in a random order (every group spans many blocks)."""
    rows = [(g, v) for g, vs in groups.items() for v in vs]
    perm = np.random.default_rng(seed).permutation(len(rows))
    return [rows[i] for i in perm]


DIRECT_DICT = ["k%05d" % i for i in range((1 << 14) - 2)]  # with MISSING and NULL: exactly 14 bits


def key_columns(ngroups):
    """Six or more groups (ids 0..n-1) under keys that select each layout.  Group 0 has a MISSING key, group 1 a NULL
    key; the others strings.  g: offset-packed, n slots (mixed radix); gd: 14 bits, direct-indexed; gw: all 64 bits
    of an int (with gd: 78 bits, hash-128)."""
    tight = utf8_sorted(["t%dé" % i for i in range(ngroups - 2)])
    return {
        "g": ([M, None] + tight, tight),
        "gd": ([M, None] + [DIRECT_DICT[0], DIRECT_DICT[-1]] + DIRECT_DICT[1:ngroups - 3], DIRECT_DICT),
        "gw": ([(-(1 << 63)) if i % 2 else (1 << 63) - 1 - i for i in range(ngroups)], None),
    }


def _string_groups(rng, dictionary, n=6):
    """Every group: the first and the last string, MISSING and NULL rows, and a random share of the dictionary."""
    out = {}
    for g in range(n):
        body = rng.choice(len(dictionary), size=3000 + 700 * g).tolist()
        out[g] = [dictionary[0], dictionary[-1], M, None, M, None] + [dictionary[i] for i in body]
    return out


def _mixed_groups(rng, dictionary, n=6):
    """Every group: FALSE, TRUE, ints, the first and last strings, MISSING and NULL."""
    out = {}
    for g in range(n):
        vals = [False, True, dictionary[0], dictionary[-1], M, None, -7 - g, 1000 + g]
        for i in rng.integers(0, 5, 4000).tolist():
            vals.append([False, True, M, None][i % 4] if i < 2 else int(rng.integers(-50, 50)) if i == 2 else dictionary[int(rng.integers(len(dictionary)))])
        out[g] = vals
    return out


UNUSED = ["0unused", "b-unused", "\U0001F601-unused"]  # imported ranks no row uses (ndict > ranks used)


def _winner_groups():
    """MIN / MAX winners across classes: one class mix per group."""
    mid = DICT_NE[len(DICT_NE) // 2]
    return {
        0: [False, M, None, False],                        # only FALSE
        1: [True, False, True, None],                      # FALSE and TRUE
        2: [True, 3, -2, False, M],                        # booleans and numbers
        3: [5, "abc", "Zeta", -9, None],                   # numbers and strings
        4: [mid, "abcdefgha", "abcdefgh", "abcdefgh\x01"],  # strings only, middle ranks
        5: [DICT_NE[0], DICT_NE[0], None],                 # the first rank only
        6: [DICT_NE[-1], M],                               # the last rank only
        7: [M, None, None],                                # nothing above NULL
    }


def _winners(groups, seed):
    """The class mixes repeated over many rows (each group spans many blocks)."""
    rng = np.random.default_rng(seed)
    return {g: [vs[i] for i in rng.integers(0, len(vs), 2000).tolist()] + vs for g, vs in groups.items()}


@functools.lru_cache(maxsize=None)
def fixture(name):
    rng = np.random.default_rng(FIXTURES.index(name) + 1)
    if name == "strings":
        return Fixture(name, shuffled(_string_groups(rng, DICT), 1), DICT, key_columns(6))
    if name == "strings_ne":
        return Fixture(name, shuffled(_string_groups(rng, DICT_NE), 2), DICT_NE, key_columns(6))
    if name == "mixed":
        return Fixture(name, shuffled(_mixed_groups(rng, DICT), 3), DICT, key_columns(6))
    if name == "winners":
        return Fixture(name, shuffled(_winners(_winner_groups(), 4), 4), DICT_NE, key_columns(8),
                       import_dict=utf8_sorted(DICT_NE + UNUSED))
    raise KeyError(name)


FIXTURES = ["strings", "strings_ne", "mixed", "winners"]


def _aggs(fx, layout):
    """Thread-private tables hold at most 48 words: with more classes that layout drops aggregates."""
    if layout == "dense-priv" and fx.name != "strings" and fx.name != "strings_ne":
        return AGGS if len(fx.keys["g"][0]) == 6 else ["count(*)", "min(%s)" % X, "max(%s)" % X]
    return NAGGS if any(isinstance(v, int) and not isinstance(v, bool) for v in fx.x) else AGGS


# (key columns, environment, mode, text the kernel must contain / must not contain)
LAYOUTS = {
    "ungrouped": ([], {}, "ungrouped", [], []),
    "dense-priv": (["g"], {}, "dense-shared-memory", ["s_priv"], []),
    "dense-shared": (["g"], {"N1GPU_NO_PRIV": "1"}, "dense-shared-memory", ["s_tab"], ["s_priv"]),
    "direct-cache256": (["gd"], {"N1GPU_CACHE_BLOCK": "256"}, "hbm-direct", ["cache_claim_1("], []),
    "direct-cache1024": (["gd"], {"N1GPU_CACHE_BLOCK": "1024"}, "hbm-direct", ["cache_claim_1("], []),
    "direct-nocache": (["gd"], {"N1GPU_NO_CACHE": "1"}, "hbm-direct", [], ["cache_claim"]),
    "direct-nopair": (["gd"], {"N1GPU_NO_MM_PAIR": "1"}, "hbm-direct", [], ["mmp"]),
    "hash64": (["gd"], {"N1GPU_NO_DIRECT": "1"}, "hbm-hash-64", [], []),
    "hash128": (["gd", "gw"], {}, "hbm-hash-128", [], []),
}


def _query(table, keys, aggs, env, monkeypatch, params=None, where=None):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    qq = q.Query(table, "d", where, [K(c) for c in keys], aggs, params=params)
    for k in env:
        monkeypatch.delenv(k)
    return qq


def _landed(fx, layout, monkeypatch):
    keys, env, mode, must, mustnot = LAYOUTS[layout]
    aggs = _aggs(fx, layout)
    qq = _query(fx.table, keys, aggs, env, monkeypatch)
    assert qq.info["mode"] == mode, (fx.name, layout, qq.info)
    src = qq.kernel_source
    assert all(m in src for m in must) and not any(m in src for m in mustnot), (fx.name, layout)
    if layout == "dense-priv":
        assert qq.info["slots"] == len(fx.keys["g"][0])  # mixed-radix: MISSING, NULL and the strings
    return qq, keys, aggs


# ---- GPU: every fixture through every layout ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def _device():
    q.init(0)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("name", FIXTURES)
def test_strings_through_every_layout(name, layout, _device, monkeypatch):
    fx = fixture(name)
    qq, keys, aggs = _landed(fx, layout, monkeypatch)
    assert_exact(fx.expected(keys, aggs), gpu_rows(qq.execute(), aggs), "%s via %s" % (name, layout))


DISTINCT_LAYOUTS = {
    "bitmap": ({"N1GPU_NO_PART": "1"}, lambda qq: not qq.part_source and "DISTINCT bitmap\n" in qq.kernel_source),
    "hashset": ({"N1GPU_NO_PART": "1", "N1GPU_NO_BITMAP": "1"}, lambda qq: not qq.part_source and "table_insert64(p.set_keys" in qq.kernel_source),
    "sliced-bitmap": ({"N1GPU_NO_PART": "1", "N1GPU_SET_PASSES": "2"}, lambda qq: not qq.part_source and "p.set_pass" in qq.kernel_source),
    "partitioned": ({"N1GPU_PART": "1"}, lambda qq: "NP " in qq.part_source),
}


def distinct_fixture(ndict):
    """A strings-only operand (no MISSING / NULL: one class, a plain rank) of `ndict` strings under an int key of 8192
    values: the partitioned DISTINCT aggregation takes a rank of at most 12 bits."""
    return _distinct_fixture(ndict)


@functools.lru_cache(maxsize=None)
def _distinct_fixture(ndict):
    rng = np.random.default_rng(ndict)
    d = utf8_sorted(["v%05dé" % i for i in range(ndict - len(EDGE_STRINGS))] + EDGE_STRINGS)
    assert len(d) == ndict
    n = 30000
    gid = np.concatenate([[0, 0, 1, 2, 3, 8191], rng.integers(4, 8191, n)]).tolist()
    vals = [d[0], d[0], d[-1], d[0], d[ndict // 2], d[-1]] + [d[i] for i in rng.integers(0, ndict, n).tolist()]
    keys = {"gk": (list(range(8192)), None)}
    return Fixture("distinct_%d" % ndict, list(zip(gid, vals)), d, keys, global_rows=1 << 20)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", list(DISTINCT_LAYOUTS))
def test_distinct_strings_in_every_set_layout(layout, _device, monkeypatch):
    fx = distinct_fixture(4096)
    env, check = DISTINCT_LAYOUTS[layout]
    qq = _query(fx.table, ["gk"], DAGGS, env, monkeypatch)
    assert qq.info["mode"] == "hbm-direct" and check(qq), layout
    assert_exact(fx.expected(["gk"], DAGGS), gpu_rows(qq.execute(), DAGGS), "distinct strings via " + layout)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["ungrouped", "dense-shared", "direct-cache1024", "hash64", "hash128"])
@pytest.mark.parametrize("name", ["mixed", "winners"])
def test_distinct_over_mixed_classes(name, layout, _device, monkeypatch):
    fx = fixture(name)
    keys, env, mode, _must, _mustnot = LAYOUTS[layout]
    qq = _query(fx.table, keys, DAGGS, env, monkeypatch)
    assert qq.info["mode"] == mode
    assert_exact(fx.expected(keys, DAGGS), gpu_rows(qq.execute(), DAGGS), "%s distinct via %s" % (name, layout))


# ---- GPU: WHERE over string columns against every constant position ----------------------------------------------------
def _where_table():
    """s: strings with "" in the dictionary; n: strings without it; m: strings, ints and booleans; k: a small int."""
    rng = np.random.default_rng(41)
    n = 4000
    absent = lambda i: M if i % 2 else None
    s = [DICT[i] if i < len(DICT) else absent(i) for i in rng.integers(0, len(DICT) + 3, n).tolist()]
    ne = [DICT_NE[i] if i < len(DICT_NE) else absent(i) for i in rng.integers(0, len(DICT_NE) + 3, n).tolist()]
    mix = []
    for i in rng.integers(0, 10, n).tolist():
        mix.append(DICT[int(rng.integers(len(DICT)))] if i < 5 else [False, True, M, None][i - 5] if i < 9 else int(rng.integers(-3, 4)))
    k = rng.integers(0, 6, n).tolist()
    s[:2], ne[:2] = [DICT[0], DICT[-1]], [DICT_NE[0], DICT_NE[-1]]
    cols = {"s": (s, DICT), "n": (ne, DICT_NE), "m": (mix, DICT), "k": (k, None)}
    t = q.Table(sorted(cols))
    for c, (vals, d) in cols.items():
        pay, tags = encode(vals, d or [])
        t.set_column(c, pay, tags=tags, dictionary=d)
    t.seal()
    docs = []
    for i in range(n):
        doc = {c: vals[i] for c, (vals, _d) in cols.items() if vals[i] is not M}
        docs.append(O.parse_document(json.dumps(doc, ensure_ascii=False)))
    return t, docs


def _lit(v):
    return json.dumps(v, ensure_ascii=False)


def _where_cases():
    """(id, WHERE text, array parameter or None)."""
    cases = []
    positions = {
        "s": {"first": DICT[0], "last": DICT[-1], "mid": "abcdefgha", "between": "abcdefgh0", "after": "\U0001F601", "empty_held": ""},
        "n": {"first": DICT_NE[0], "last": DICT_NE[-1], "mid": "zeta", "before": "0", "between": "abcdefghaa0", "after": "\U0001F600y",
              "empty_absent": ""},
        "m": {"first": DICT[0], "mid": "cafe", "between": "b", "after": "\U0001F601", "num": 1},
    }
    for c, pos in positions.items():
        f = K(c)
        for pid, v in pos.items():
            for op in ("=", "<", "<=", ">", ">="):
                cases.append(("%s %s %s" % (c, op, pid), "(%s %s %s)" % (f, op, _lit(v)), None))
            cases.append(("%s not= %s" % (c, pid), "(not (%s = %s))" % (f, _lit(v)), None))
        vals = list(pos.values())
        lo, hi = min(vals[:-1] if c == "m" else vals, key=lambda s: s.encode()), "\U0001F600z"
        cases.append(("%s between" % c, "(%s between %s and %s)" % (f, _lit(vals[1 if c != "m" else 0]), _lit(hi)), None))
        cases.append(("%s between absent" % c, "(%s between %s and %s)" % (f, _lit("abcdefgh0"), _lit("caf")), None))
        cases.append(("%s between low" % c, "(%s between %s and %s)" % (f, _lit(lo), _lit("A")), None))
        cases.append(("%s in literal" % c, "(%s in [%s])" % (f, ", ".join(_lit(v) for v in vals)), None))
        cases.append(("%s not in literal" % c, "(not (%s in [%s, %s]))" % (f, _lit(vals[0]), _lit(vals[-1])), None))
        cases.append(("%s in param" % c, "(%s in $1)" % f, vals))
        cases.append(("%s truth" % c, f, None))
        cases.append(("%s not truth" % c, "(not %s)" % f, None))
        cases.append(("%s and" % c, "(%s and ((`d`.`k`) < 3))" % f, None))
        cases.append(("%s or" % c, "(%s or ((`d`.`k`) = 5))" % f, None))
    cases.append(("m num lt", "((`d`.`m`) < 2)", None))
    cases.append(("m num between", "((`d`.`m`) between -1 and 2)", None))
    return cases


WHERE_CASES = _where_cases()


@pytest.fixture(scope="module")
def where_table():
    return _where_table()


@pytest.mark.gpu
def test_where_over_strings_against_every_constant_position(where_table, _device):
    """Every predicate over the three columns, counted per group of k and checked with the oracle: the constants'
    rank codes (2 * rank present, 2 * lower_bound - 1 absent) and the truth value's rank of ""."""
    t, docs = where_table
    aggs = ["count(*)", "min((`d`.`s`))", "max((`d`.`m`))"]
    for cid, where, param in WHERE_CASES:
        qq = q.Query(t, "d", where, [K("k")], aggs, params={"1": param} if param is not None else None)
        got = gpu_rows(qq.execute(), aggs)
        owhere = where.replace("$1", "[%s]" % ", ".join(_lit(v) for v in param)) if param is not None else where
        want = {}
        for r in O.run_chain(docs, "d", owhere, [K("k")], aggs):
            want[tuple(key_text(O.to_python(v)) for v in r.keys)] = ({a: O.to_python(r.aggregates[a]) for a in aggs}, False)
        assert_exact(want, got, "%s: %s" % (cid, where))


# ---- GPU: the device dictionary build against the host shredder ---------------------------------------------------------
def _many_strings(n):
    """n distinct strings: groups that share an 8-byte prefix (differing at byte 8, 9 or in length) and raw UTF-8 bytes
    >= 0x80 in every position."""
    rng = np.random.default_rng(51)
    out = set(EDGE_STRINGS)
    out.add("")
    pre = ["prefix%02d" % i for i in range(40)]
    for p in pre:
        out.add(p)
        for j in range(200):
            out.add(p + chr(0x61 + j % 26) + ("%d" % (j // 26) if j >= 26 else ""))
    alphabet = "aZ09~éÿĀ߿ࠀ€￿\U00010000\U0001F600"
    while len(out) < n:
        k = int(rng.integers(1, 14))
        out.add("".join(alphabet[i] for i in rng.integers(0, len(alphabet), k).tolist()))
    return utf8_sorted(out)[:n]


@pytest.fixture(scope="module")
def many_docs():
    strings = _many_strings(30000)
    rng = np.random.default_rng(52)
    docs, rows = [], []
    for i in range(90000):
        g = int(rng.integers(0, 7))
        v = strings[i] if i < len(strings) else strings[int(rng.integers(len(strings)))]
        r = int(rng.integers(0, 40))
        v = M if r == 0 else None if r == 1 else (r == 2) if r < 4 else v
        doc = {"g": g}
        if v is not M:
            doc["x"] = v
        docs.append(json.dumps(doc, ensure_ascii=False))
        rows.append((g, v))
    return docs, rows, strings


@pytest.mark.gpu
def test_device_dictionary_matches_the_host_shredder(many_docs, _device):
    docs, rows, strings = many_docs
    aggs = AGGS + ["count(distinct %s)" % X]
    tables = {}
    for threads in (-1, 1):
        t = q.Table(["g", "x"])
        t.append_json(docs, threads=threads)
        tables[threads] = t
    dev, host = tables[-1].dictionary("x"), tables[1].dictionary("x")  # (exported before seal)
    used = utf8_sorted(v for _g, v in rows if isinstance(v, str))
    assert len(used) >= 20000  # the sample sort of the device shredder's dictionary
    assert dev == host and [s.decode("utf-8") for s in dev] == used
    for t in tables.values():
        t.seal()
    fx = Fixture("many", rows, None, {"g": (list(range(7)), None)})
    for threads, t in tables.items():
        qq = q.Query(t, "d", None, [K("g")], aggs)
        assert_exact(fx.expected(["g"], aggs), gpu_rows(qq.execute(), aggs), "threads=%d" % threads)


# ---- GPU: partitions whose dictionaries and class mixes differ -----------------------------------------------------------
def _partition_cases():
    """{case: [rows of partition r]}: (group id, x value)."""
    a = ["alpha", "beta", "gammaé"]
    b = ["delta", "epsilon", "\U0001F600"]
    return {
        "disjoint": [[(g, a[g % 3]) for g in range(6)] * 50, [(g, b[g % 3]) for g in range(6)] * 40, [(g, None) for g in range(6)] * 3],
        "overlap": [[(g, a[g % 3]) for g in range(6)] * 50, [(g, (a + b)[g]) for g in range(6)] * 40, [(g, b[(g + 1) % 3]) for g in range(6)] * 7],
        "empty_dict": [[(g, a[g % 3]) for g in range(6)] * 50, [(g, M if g % 2 else None) for g in range(6)] * 9, [(g, b[g % 3]) for g in range(6)]],
        "empty_string": [[(g, a[g % 3]) for g in range(6)] * 50, [(g, "" if g < 3 else b[g % 3]) for g in range(6)] * 40, [(g, "zz") for g in range(6)]],
        "class_mix": [[(g, a[g % 3]) for g in range(6)] * 50, [(g, b[g % 3] if g % 2 else g * 7 - 20) for g in range(6)] * 40,
                      [(g, M if g % 2 else None) for g in range(6)] * 9],
    }


PART_KEY = lambda g: g << 40  # six groups spread over 43 bits: a hashed table, whose partial states travel as records


def _partition_table(rows, how):
    """One partition's table (unsealed): x and the group key g, host-staged, device-shredded or set_column_device."""
    import torch
    rows = [(PART_KEY(g), v) for g, v in rows]
    xs = [v for _g, v in rows]
    d = utf8_sorted([v for v in xs if isinstance(v, str)])
    t = q.Table(["g", "x"])
    if how == "docs":
        docs = []
        for g, v in rows:
            doc = {"g": g}
            if v is not M:
                doc["x"] = v
            docs.append(json.dumps(doc, ensure_ascii=False))
        t.append_json(docs, threads=-1)
        return t
    cols = {"g": encode([g for g, _v in rows], []), "x": encode(xs, d)}
    for c, (pay, tags) in cols.items():
        dd = (d or None) if c == "x" else None
        if how == "host":
            t.set_column(c, pay, tags=tags, dictionary=dd)
        else:
            p = torch.from_numpy(pay.view(np.int32) if pay.dtype == np.uint32 else pay).cuda()
            t.set_column_device(c, p, tags=torch.from_numpy(tags).cuda(), dictionary=dd)
    return t


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["host", "docs", "device"])
@pytest.mark.parametrize("nparts", [2, 3])
@pytest.mark.parametrize("case", list(_partition_cases()))
def test_partitions_agree_on_one_kernel(case, nparts, how, _device, monkeypatch):
    """Partitions of one keyspace whose dictionaries and classes differ compile the same kernel after the dictionary /
    statistics agreement (what DistributedQuery's digest check demands), and their merged groups equal one scan of all
    rows.  A device-resident column is sized by its own rows and widened at seal to the agreed classes."""
    import torch
    from query_b200 import dist as qd
    parts = _partition_cases()[case][:nparts]
    keys, env, mode, _must, _mustnot = LAYOUTS["hash64"]
    tables = [_partition_table(rows, how) for rows in parts]
    qd.agree_local(tables)
    allrows = [r for rows in parts for r in rows]
    union = Fixture("union", allrows, None, {"gd": ([PART_KEY(g) for g in range(6)], None)})
    qs = []
    for t in tables:
        t.seal()
        qq = _query(t, ["g"], NAGGS, env, monkeypatch)
        assert qq.info["mode"] == mode
        qq.scan_partial()
        qs.append(qq)
    assert len({x.kernel_source for x in qs}) == 1, "partitions compiled different kernels"
    n = len(qs)
    exported = []
    for qq in qs:
        ng, nd, rw = qq.partial_counts()
        recs = torch.zeros(max(1, ng) * rw, dtype=torch.int64, device="cuda")
        dents = torch.zeros(2, dtype=torch.int64, device="cuda")
        counts, _dcounts = qq.partial_export(n, recs.data_ptr(), ng, dents.data_ptr(), nd)
        exported.append((recs, counts, rw))
    got = {}
    for owner, qq in enumerate(qs):
        qq.partial_reset()
        for recs, counts, rw in exported:
            o = int(counts[:owner].sum())
            r = recs[o * rw:(o + int(counts[owner])) * rw].contiguous()
            qq.partial_import(r.data_ptr() if counts[owner] else 0, int(counts[owner]), 0, 0)
        part = gpu_rows(qq.finalize(), NAGGS)
        assert not (set(part) & set(got))
        got.update(part)
    assert_exact(union.expected(["gd"], NAGGS), got, "%s, %d partitions, %s" % (case, nparts, how))


# ---- CPU: the exact reference against the oracle ---------------------------------------------------------------------
def test_exact_reference_matches_the_oracle():
    fx = Fixture("oracle", shuffled(_winners(_winner_groups(), 61), 61) + shuffled(_mixed_groups(np.random.default_rng(62), DICT, 6), 62)[:3000],
                 DICT, key_columns(8))
    docs = []
    for g, v in zip(fx.gid, fx.x):
        doc = {}
        if fx.keys["g"][0][g] is not M:
            doc["g"] = fx.keys["g"][0][g]
        if v is not M:
            doc["x"] = v
        docs.append(O.parse_document(json.dumps(doc, ensure_ascii=False)))
    aggs = NAGGS + ["count(distinct %s)" % X]
    want = {}
    for r in O.run_chain(docs, "d", None, [K("g")], aggs):
        want[tuple(key_text(O.to_python(v)) for v in r.keys)] = {a: O.to_python(r.aggregates[a]) for a in aggs}
    exp = fx.expected(["g"], aggs)
    assert set(want) == set(exp)
    for k, (row, _approx) in exp.items():
        for a, v in row.items():
            assert type(want[k][a]) is type(v) and want[k][a] == v, (k, a, want[k][a], v)


def test_dictionaries_hold_the_edge_strings():
    assert DICT[0] == "" and DICT_NE[0] == "A"
    assert DICT.index("￿") + 1 == DICT.index("\U0001F600")  # bytewise: EF BF BF < F0 9F 98 80 (UTF-16 says otherwise)
    assert DICT.index("Zeta") < DICT.index("zeta") and DICT.index("abcdefgh") + 1 == DICT.index("abcdefgh\x01")
    assert "".join(sorted(["￿", "\U0001F600"], key=lambda s: s.encode("utf-16-be"))) == "\U0001F600￿"


# ---- CPU: which side of every threshold a fixture lands on --------------------------------------------------------------
def _key_table(ndict, extra=(), global_rows=None, ints=None):
    """A string key s over `ndict` strings with MISSING and NULL rows (and `extra` values), x strings; ints: (lo, hi)
    of a second key column i."""
    d = ["s%06d" % j for j in range(ndict)]
    svals = [M, None] + d + list(extra)
    cols = {"s": (svals, d), "x": ([d[j % ndict] if ndict else None for j in range(len(svals))], d or None)}
    if ints is not None:
        lo, hi = ints
        cols["i"] = ([lo + (j % 2) * (hi - lo) for j in range(len(svals))], None)
    t = q.Table(sorted(cols))
    for c, (vals, dd) in cols.items():
        pay, tags = encode(vals, dd or [])
        t.set_column(c, pay, tags=tags, dictionary=dd)
    if global_rows is not None:
        t.set_global_rows(global_rows)
    t.seal()
    return t


def _plan(t, keys, aggs, monkeypatch, env=None):
    qq = _query(t, keys, aggs, env or {}, monkeypatch)
    return qq.info, qq.kernel_source, qq.part_source


@pytest.mark.parametrize("b", [3, 5, 12])
def test_string_key_offset_packing_at_2_b_minus_2(b, monkeypatch):
    """MISSING + NULL + 2^b - 2 strings: b bits (bit-packed slots 2^b); one string more: b + 1 bits, numbered by the
    mixed radix (2^b + 1 slots).  At b = 12 one accumulator word (8 bytes x 2^12 = 32 KiB) still fits the 40 KiB shared
    table; 13 bits move to the direct-indexed HBM table."""
    n = (1 << b) - 2
    info_in, _src, _ = _plan(_key_table(n), ["s"], ["count(*)"], monkeypatch)
    info_out, _src, _ = _plan(_key_table(n + 1), ["s"], ["count(*)"], monkeypatch)
    assert info_in["mode"] == "dense-shared-memory" and info_in["slots"] == 1 << b
    if b < 12:
        assert info_out["mode"] == "dense-shared-memory" and info_out["slots"] == (1 << b) + 1
    else:
        assert info_out["mode"] == "hbm-direct"


def test_thread_private_table_up_to_48_cells(monkeypatch):
    """slots x words <= 48: thread-private copies; one string more (one slot more, mixed radix) crosses it."""
    aggs = ["count(*)", "min(%s)" % X, "max(%s)" % X, "count(%s)" % X]
    w = _plan(_key_table(6), ["s"], aggs, monkeypatch)[0]["words"]
    big = 48 // w  # the largest slot count that still fits
    info2, src2, _ = _plan(_key_table(big - 2), ["s"], aggs, monkeypatch)
    info3, src3, _ = _plan(_key_table(big - 1), ["s"], aggs, monkeypatch)
    assert info2["slots"] * w == 48 and "s_priv" in src2
    assert info3["slots"] == big + 1 and "s_priv" not in src3 and "s_tab" in src3


@pytest.mark.parametrize("b", [4, 6])
def test_cache_key32_at_31_and_32_bits(b, monkeypatch):
    """A string key of b bits next to an int key of 31 - b bits: u32 front-cache keys; one string more: 64-bit keys."""
    ints = (0, (1 << (31 - b)) - 1)
    n = (1 << b) - 2
    _i, src_in, _ = _plan(_key_table(n, ints=ints), ["s", "i"], ["count(*)"], monkeypatch)
    _i2, src_out, _ = _plan(_key_table(n + 1, ints=ints), ["s", "i"], ["count(*)"], monkeypatch)
    assert _i["mode"] == _i2["mode"] == "hbm-hash-64"
    assert "cache_claim_1(" in src_in and "cache_claim_n(" in src_out


def test_hash64_up_to_63_bits(monkeypatch):
    """String key of 4 bits + a biased int key of 59 bits: 63 bits, hash-64; one string more: 64 bits, hash-128."""
    ints = (-(1 << 58), (1 << 58) - 1)
    assert _plan(_key_table(14, ints=ints), ["s", "i"], ["count(*)"], monkeypatch)[0]["mode"] == "hbm-hash-64"
    assert _plan(_key_table(15, ints=ints), ["s", "i"], ["count(*)"], monkeypatch)[0]["mode"] == "hbm-hash-128"


@pytest.mark.parametrize("nd,rows,mode", [(14, 1 << 19, "hbm-direct"), (14, (1 << 19) - 1, "hbm-hash-64"), (15, 1 << 22, "hbm-hash-64")],
                         ids=["22bits", "22bits-rows-1", "23bits"])
def test_direct_table_up_to_22_bits_and_8_rows_a_slot(nd, rows, mode, monkeypatch):
    """String key of 4 bits + int key of 18 bits: 22 bits, direct-indexed when 2^22 <= 8 x declared rows."""
    t = _key_table(nd, ints=(0, (1 << 18) - 1), global_rows=rows)
    assert _plan(t, ["s", "i"], ["count(*)"], monkeypatch)[0]["mode"] == mode


@pytest.mark.parametrize("ndict,slots", [(12, 16), (13, 17)])
def test_boolean_key_counts_four_free_classes(ndict, slots, monkeypatch):
    """MISSING, NULL, FALSE, TRUE and strings: offset-packed as 4 + ndict values."""
    t = _key_table(ndict, extra=[False, True])
    info, _src, _ = _plan(t, ["s"], ["count(*)"], monkeypatch)
    assert info["mode"] == "dense-shared-memory" and info["slots"] == slots


def test_degenerate_string_keys(monkeypatch):
    """One string (bits_for(1) = 0 payload bits): the class index alone; no string at all: MISSING / NULL only."""
    t = _key_table(1)
    assert _plan(t, ["s"], ["count(*)"], monkeypatch)[0]["slots"] == 4  # classes MISSING, NULL, STRING: 2 bits, no offset pack
    t = q.Table(["s", "x"])
    for c in ("s", "x"):
        t.set_column(c, np.zeros(4, dtype=np.uint32), tags=np.array([0, 1, 0, 1], dtype=np.uint8), dictionary=["a", "b"])
    t.seal()
    info, _src, _ = _plan(t, ["s"], ["count(*)", "min(%s)" % X], monkeypatch)
    assert info["slots"] == 2
    t = q.Table(["s", "x"])
    for c in ("s", "x"):
        t.set_column(c, np.zeros(4, dtype=np.uint32), dictionary=["only"])
    t.seal()
    assert _plan(t, ["s"], ["count(*)"], monkeypatch)[0]["slots"] == 1


def test_string_and_int_key_without_offset_packing(monkeypatch):
    """A key of strings and ints packs the class index and the wider payload: no offset packing (two payload classes)."""
    t = _key_table(6, extra=[5, 6, 7, 8, False])  # classes M N F I S: 3 bits + max(int 2 bits, string 3 bits) = 6 bits
    info, src, _ = _plan(t, ["s"], ["count(*)"], monkeypatch)
    assert info["mode"] == "dense-shared-memory" and info["slots"] == 64


def test_min_max_seen_word(monkeypatch):
    """Over a single-class string operand MIN / MAX take the seen count; over a mixed operand the seen: OR word.  MIN and
    MAX rank cells of one operand pair (mmp) in a direct table unless N1GPU_NO_MM_PAIR."""
    seen_or = "OP_OR_U64, (1ULL << "
    fx = fixture("strings")
    for layout in ("ungrouped", "direct-cache1024"):
        src = _landed(fx, layout, monkeypatch)[0].kernel_source
        assert seen_or not in src
    src = _landed(fx, "direct-cache1024", monkeypatch)[0].kernel_source
    assert "cache_mm32" in src and "mmp" in src
    assert "mmp" not in _landed(fx, "direct-nopair", monkeypatch)[0].kernel_source
    for name in ("mixed", "winners"):
        assert seen_or in _landed(fixture(name), "direct-cache1024", monkeypatch)[0].kernel_source


@pytest.mark.parametrize("ndict,part", [(4096, True), (4097, False)])
def test_partitioned_distinct_needs_a_12_bit_rank(ndict, part, monkeypatch):
    fx = distinct_fixture(ndict)
    info, _src, psrc = _plan(fx.table, ["gk"], DAGGS, monkeypatch, {"N1GPU_PART": "1"})
    assert info["mode"] == "hbm-direct" and bool(psrc) == part


@pytest.mark.parametrize("layout", list(DISTINCT_LAYOUTS))
def test_distinct_strings_land_on_their_set_layouts(layout, monkeypatch):
    env, check = DISTINCT_LAYOUTS[layout]
    qq = _query(distinct_fixture(4096).table, ["gk"], DAGGS, env, monkeypatch)
    assert qq.info["mode"] == "hbm-direct" and check(qq), layout


def test_gpu_fixtures_land_on_their_layouts(monkeypatch):
    """Every fixture reaches the mode its GPU test asserts, so a planner change cannot move one elsewhere."""
    for name in FIXTURES:
        for layout in LAYOUTS:
            _landed(fixture(name), layout, monkeypatch)
