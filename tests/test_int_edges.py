"""Integer COUNT / SUM / AVG / MIN / MAX at the int64 limits and on both sides of every accumulator-layout threshold.

The planner (query_b200/csrc/codegen.cpp) reads column statistics and the declared keyspace row count to choose
narrower or fewer accumulators: one `isum` word instead of the `ilo` / `ihi` split, a float64 word carrying INT and
FLOAT addends (`fcarry`), one-cell 32-bit cached sums (`cache_add_carry`), 32-bit MIN / MAX cells holding
`value - lo + 1` (`cache_mm32`, paired as `mmp`), the sign mix of a SUM read off MIN / MAX, biased / offset-packed
keys and DISTINCT values, direct / hashed tables and the partitioned DISTINCT aggregation.  Every choice rests on a
range proof.  The fixtures here sit exactly on those proofs and just across them, and every result is compared
bit-exact, class included, with `exact_aggregates`: DESIGN.md section 4 restated with Python ints.

The CPU tests (no `gpu` mark) pin which side of each threshold every fixture lands on, from the generated kernel text.
"""
import functools
import math

import numpy as np
import pytest

import query_b200 as q
from oracle import n1ql_oracle as O
from util_n1 import gpu_rows

I64_MIN, I64_MAX = -(1 << 63), (1 << 63) - 1
T_MISSING, T_NULL, T_INT, T_FLOAT = 0, 1, 4, 5
MM32_SPAN = 0xfffffffc  # widest hi - lo a 32-bit MIN / MAX cell holds (value - lo + 1 stays below the empty value)

X = "(`d`.`x`)"
AGGS = ["count(*)", "count(%s)" % X, "countn(%s)" % X, "sum(%s)" % X, "avg(%s)" % X, "min(%s)" % X, "max(%s)" % X]
DAGGS = ["count(*)", "count(distinct %s)" % X, "sum(distinct %s)" % X, "avg(distinct %s)" % X]
K = lambda c: "(`d`.`%s`)" % c


# ---- exact reference -------------------------------------------------------------------------------------------------
def _py(tag, pay):
    if tag == T_INT:
        return int(pay)
    if tag == T_FLOAT:
        return float(np.array([pay], dtype=np.int64).view(np.float64)[0])
    return None if tag == T_NULL else O.MISSING


def _is_num(v):
    return isinstance(v, (int, float)) and not isinstance(v, bool)


def _int_sum(ints, from_zero):
    """SUM of ints (value/integer.go:266-277): an int when no sign mix (0 is non-negative) and the exact total fits,
    otherwise the correctly rounded float64 of the exact total.  SUM(DISTINCT) starts from int 0, so a negative member
    alone already mixes signs."""
    total = sum(ints)
    neg = any(v < 0 for v in ints)
    mixed = neg if from_zero else (neg and any(v >= 0 for v in ints))
    return total if not mixed and I64_MIN <= total <= I64_MAX else float(total)


def exact_aggregates(values, distinct=False):
    """{aggregate kind: value} of one group whose operand values are `values` (int / float / None / MISSING), and
    whether SUM / AVG involve a float addend (then only their class is exact; the float64 sum order is not specified)."""
    nums = [v for v in values if _is_num(v)]
    ints = [v for v in nums if isinstance(v, int)]
    flts = [v for v in nums if isinstance(v, float)]
    out = {"count*": len(values), "count": sum(1 for v in values if v is not None and v is not O.MISSING), "countn": len(nums)}
    if distinct:
        ints, flts = sorted(set(ints)), sorted(set(flts))
        nums = ints + flts
        out["dcount"] = len(nums)
    if not nums:
        out["sum"] = out["avg"] = out["min"] = out["max"] = None
        return out, False
    s = _int_sum(ints, distinct) if not flts else float(sum(ints)) + math.fsum(flts)
    out["sum"] = s
    out["avg"] = O.new_value(float(s) / len(nums))
    for kind, better in (("min", lambda a, b: a <= b), ("max", lambda a, b: a >= b)):
        pick = min if kind == "min" else max
        i = pick(ints) if ints else None
        f = pick(flts) if flts else None
        # intValue.Collate(floatValue) compares as float64 (value/integer.go:100-118); the fixtures never tie
        out[kind] = i if f is None else f if i is None else (i if better(float(i), f) else f)
    return out, bool(flts)


def _agg_kind(text):
    name = text.split("(", 1)[0]
    if text == "count(*)":
        return "count*"
    if "distinct" in text:
        return {"count": "dcount", "sum": "sum", "avg": "avg"}[name]
    return name


def assert_exact(exp, got, what):
    assert set(exp) == set(got), "%s group keys differ: only reference %s, only gpu %s" % (
        what, sorted(set(exp) - set(got))[:5], sorted(set(got) - set(exp))[:5])
    for k, (aggs, approx) in exp.items():
        for a, v in aggs.items():
            w = got[k][a]
            msg = "%s group %s %s: reference %r gpu %r" % (what, k, a, v, w)
            if approx and (a.startswith("sum(") or a.startswith("avg(")) and _is_num(v):
                assert type(w) is type(v) and abs(v - w) <= 1e-12 * max(abs(v), abs(w)), msg
            else:
                assert type(w) is type(v) and (v == w if not isinstance(v, float) else v.hex() == w.hex()), msg


# ---- fixtures: pre-shredded columns ----------------------------------------------------------------------------------
def ints(vals):
    a = np.array([int(v) for v in vals], dtype=np.int64)
    return np.full(len(a), T_INT, dtype=np.uint8), a


def floats(vals):
    a = np.array(vals, dtype=np.float64)
    assert not np.any(a == np.floor(a)), "integral floats would be canonicalised"
    return np.full(len(a), T_FLOAT, dtype=np.uint8), a.view(np.int64)


def absent(n):
    return np.where(np.arange(n) % 2 == 0, T_MISSING, T_NULL).astype(np.uint8), np.zeros(n, dtype=np.int64)


def rand_ints(rng, lo, hi, n):
    return ints(rng.integers(lo, hi, size=n, endpoint=True, dtype=np.int64).tolist())


# Group-key columns: the same six groups (ids 0..5) under keys that select each layout.  Group 0 has a MISSING key and
# group 1 a NULL key where the column allows them (offset packing; register groups).
def _tight(base):  # MISSING, NULL and four ints from `base`: six offset-packed values -> a six-slot mixed-radix table
    return [(T_MISSING, 0), (T_NULL, 0)] + [(T_INT, base + j) for j in range(4)]


KEY_COLUMNS = {
    "gd": [(T_MISSING, 0), (T_NULL, 0)] + [(T_INT, -4500 + 3000 * j) for j in range(4)],  # 14 bits: direct-indexed
    "gw1": [(T_INT, v) for v in (I64_MIN, I64_MAX, -1, 0, 1, 12345)],                      # 64 bits
    "gw2": [(T_INT, I64_MAX - ((1 << 62) - 2) + j * (((1 << 62) - 2) // 5)) for j in range(6)],  # 62 bits, biased
}


class Fixture:
    def __init__(self, name, gid, tags, pay, key_base=-2, global_rows=None, key_columns=None):
        """Rows (group id, x tag, x payload); the key columns map group ids to keys."""
        self.name, self.global_rows = name, global_rows
        self.gid, self.tags, self.pay = np.asarray(gid, dtype=np.int64), np.asarray(tags, dtype=np.uint8), np.asarray(pay, dtype=np.int64)
        self.keys = dict(KEY_COLUMNS, g=_tight(key_base)) if key_columns is None else key_columns

    @functools.cached_property
    def table(self):
        t = q.Table(["x"] + sorted(self.keys))
        t.set_column("x", self.pay, tags=self.tags)
        for c, spec in self.keys.items():
            kt = np.array([s[0] for s in spec], dtype=np.uint8)[self.gid]
            kv = np.array([s[1] for s in spec], dtype=np.int64)[self.gid]
            t.set_column(c, kv, tags=kt)
        if self.global_rows is not None:
            t.set_global_rows(self.global_rows)
        t.seal()
        return t

    def values(self, op=None):
        vals = [_py(t, p) for t, p in zip(self.tags.tolist(), self.pay.tolist())]
        return vals if op is None else [op(v) for v in vals]

    def expected(self, keys, aggs, op=None, distinct=False):
        vals = self.values(op)
        by = {}
        for g, v in zip(self.gid.tolist(), vals):
            by.setdefault(g if keys else 0, []).append(v)
        out = {}
        for g, vs in by.items():
            k = tuple("MISSING" if self.keys[c][g][0] == T_MISSING else "null" if self.keys[c][g][0] == T_NULL
                      else str(self.keys[c][g][1]) for c in keys)
            r, approx = exact_aggregates(vs, distinct)
            out[k] = ({a: r[_agg_kind(a)] for a in aggs}, approx)
        return out


def grouped(name, groups, seed, **kw):
    """groups: {group id: [(tags, payload), ...]}; rows are shuffled so that every group spans many blocks."""
    gid, tags, pay = [], [], []
    for g, parts in groups.items():
        for t, p in parts:
            gid.append(np.full(len(t), g, dtype=np.int64))
            tags.append(t)
            pay.append(p)
    perm = np.random.default_rng(seed).permutation(sum(len(t) for t in tags))
    return Fixture(name, np.concatenate(gid)[perm], np.concatenate(tags)[perm], np.concatenate(pay)[perm], **kw)


def _overflow_groups(rng, sign):
    """Six groups of one sign (x >= 0 for sign 1, x <= 0 for sign -1) at and just across the int64 limit."""
    lim = I64_MAX if sign > 0 else I64_MIN
    step = sign * ((1 << 47) - (1 if sign > 0 else 0))        # 65 536 of these + a remainder row reach the limit exactly
    rest = lim - (1 << 16) * step
    return {
        0: [ints([step] * (1 << 16) + [rest])],                 # sum == INT64_MAX / INT64_MIN: an int
        1: [ints([step] * (1 << 16) + [rest, sign])],           # one past it: float +-2^63 (+-(2^63 + 1) rounds there)
        2: [ints([lim]), absent(5)],                            # only the limit itself
        # low 32-bit word 0xffffffff: the low-word sum passes 2^32 inside one block while the high word is negative
        # (sign -1: -1 - 2^32 j) or positive (2^32 j + 0xffffffff)
        3: [ints([(j << 32) | 0xffffffff if sign > 0 else -1 - (j << 32) for j in rng.integers(0, 8, 70000).tolist()])],
        4: [ints([0] * 70000 + ([-1] if sign < 0 else []))],    # zeros, and (sign -1) exactly one negative: a float
        5: [ints(sign * rng.integers(0, 1 << 40, 80000).astype(np.int64)), absent(300)],
    }


def _mixed_groups(rng):
    return {
        0: [ints([(1 << 62) + 5, -(1 << 62) - 3] * 35000)],          # mixed signs, the total fits: a float
        1: [ints([I64_MAX, I64_MAX, I64_MIN, I64_MIN, 5] * 3)],      # partial sums leave int64, the total is back
        2: [ints([I64_MIN]), absent(3)],
        3: [ints([I64_MAX])],
        4: [rand_ints(rng, I64_MIN, I64_MAX, 70000)],                # |total| up to 2^79: int128 -> double rounding
        5: [ints([I64_MIN] * 3 + [7]), absent(2)],                   # below INT64_MIN with a positive member
    }


def _small_addend_groups(rng, lo, hi):
    n = 80000
    return {
        0: [ints([hi, lo] * (n // 2) + [hi])],                       # the 32-bit cell wraps both ways thousands of times
        1: [ints([hi] * n)],
        2: [ints([lo] * n)],
        3: [rand_ints(rng, lo, hi, n)],
        4: [ints([lo])],
        5: [ints([hi, 0, 0]), absent(4)],
    }


def _mm_groups(rng, lo, hi):
    return {
        0: [ints([lo] * 3)],                                         # only lo: the cell value 1
        1: [ints([hi] * 3)],                                         # only hi: the cell value hi - lo + 1
        2: [rand_ints(rng, lo, hi, 70000), ints([lo, hi])],
        3: [ints(hi - rng.integers(0, 1000, 70000))],
        4: [ints(lo + rng.integers(0, 1000, 70000))],
        5: [absent(6), ints([lo + 1])],
    }


def _largest_rows_below(mx, bound):
    """The largest row count R with mx * R < bound in float64 - the planner's proof, evaluated the same way."""
    r = int(bound / mx)
    while float(mx) * float(r) >= bound:
        r -= 1
    while float(mx) * float(r + 1) < bound:
        r += 1
    return r


ISUM34_ROWS = _largest_rows_below(float(1 << 34), 2.3e18)
ISUM50_ROWS = _largest_rows_below(float(1 << 50), 2.3e18)   # 2042
FCARRY_ROWS = _largest_rows_below(float(1 << 36), 9.0e15)


def _isum34_groups(rng):
    return {0: [ints([1 << 34] * 3)], 1: [ints([-(1 << 34)] * 3)], 2: [ints([1 << 34] * 150000)], 3: [ints([-(1 << 34)] * 70000)],
            4: [rand_ints(rng, -(1 << 34), 1 << 34, 70000)], 5: [absent(10)]}


def _isum50_groups(extra):
    return {0: [ints([1 << 50])], 1: [ints([-(1 << 50)])], 2: [ints([1 << 50] * (2030 + extra))], 3: [ints([-(1 << 50)] * 5)],
            4: [ints([(1 << 50), -(1 << 50), 7])], 5: [absent(2)]}


def _fcarry_groups(rng):
    n2 = FCARRY_ROWS - 1000 - 3
    return {
        0: [ints([-(1 << 36)] * 400)],
        1: [ints([0] * 50), absent(50)],
        2: [ints((1 << 36) - np.arange(n2) % 1000)],                  # int-only, the total just below 2^53: an exact INT
        3: [ints([1 << 36, -(1 << 36) + 1] * 100)],                   # int-only, mixed signs: an exact float
        4: [ints([1 << 30] * 100), floats(np.arange(100) + 0.25)],    # INT and FLOAT: a float (1e-12)
        5: [floats(np.arange(100) + 0.5)],
    }


@functools.lru_cache(maxsize=None)
def _fixtures():
    rng = lambda s: np.random.default_rng(s)
    fx = [
        grouped("pos", _overflow_groups(rng(1), 1), seed=1, key_base=I64_MAX - 3),
        grouped("neg", _overflow_groups(rng(2), -1), seed=2, key_base=I64_MIN),
        grouped("mixed", _mixed_groups(rng(3)), seed=3),
        grouped("wide1", _small_addend_groups(rng(4), -((1 << 31) - 1), (1 << 31) - 1), seed=4),
        grouped("wide", _small_addend_groups(rng(5), -(1 << 31), 1 << 31), seed=5),
        grouped("isum34_in", _isum34_groups(rng(6)), seed=6, global_rows=ISUM34_ROWS),
        grouped("isum34_out", _isum34_groups(rng(6)), seed=6, global_rows=ISUM34_ROWS + 1),
        grouped("isum50_in", _isum50_groups(0), seed=7, global_rows=ISUM50_ROWS),
        grouped("isum50_out", _isum50_groups(1), seed=7, global_rows=ISUM50_ROWS + 1),
        grouped("fcarry_in", _fcarry_groups(rng(8)), seed=8, global_rows=FCARRY_ROWS),
        grouped("fcarry_out", _fcarry_groups(rng(8)), seed=8, global_rows=FCARRY_ROWS + 1),
    ]
    return {f.name: f for f in fx}


def _mm_ranges():
    """(lo, hi) of the MIN / MAX fixtures: spans of 0xfffffffc (32-bit cells) and 0xfffffffd .. 0xffffffff, 2^32
    (64-bit cells), for lo in {INT64_MIN, -2^31, 0} and with hi == INT64_MAX."""
    out = []
    for lo in (I64_MIN, -(1 << 31), 0):
        out += [(lo, lo + s) for s in (MM32_SPAN, MM32_SPAN + 1, MM32_SPAN + 2, MM32_SPAN + 3, 1 << 32)]
    out += [(I64_MAX - s, I64_MAX) for s in (MM32_SPAN, MM32_SPAN + 1, MM32_SPAN + 3)]
    return out


def _mm_name(lo, hi):
    return "mm_%s_%x" % ({I64_MIN: "i64min", -(1 << 31): "m2p31", 0: "zero"}.get(lo, "i64max"), hi - lo)


@functools.lru_cache(maxsize=None)
def fixture(name):
    if name.startswith("mm_"):
        for i, (lo, hi) in enumerate(_mm_ranges()):
            if _mm_name(lo, hi) == name:
                return grouped(name, _mm_groups(np.random.default_rng(100 + i), lo, hi), seed=100 + i)
    return _fixtures()[name]


VALUE_FIXTURES = ["pos", "neg", "mixed", "wide1", "wide", "isum34_in", "isum34_out", "isum50_in", "isum50_out", "fcarry_in", "fcarry_out"]
MM_FIXTURES = [_mm_name(lo, hi) for lo, hi in _mm_ranges()]

# (id, key columns, environment, mode, text the kernel must contain / must not contain)
LAYOUTS = {
    "ungrouped": ([], {}, "ungrouped", [], []),
    "dense-priv": (["g"], {}, "dense-shared-memory", ["s_priv"], []),
    "dense-shared": (["g"], {"N1GPU_NO_PRIV": "1"}, "dense-shared-memory", ["s_tab"], ["s_priv"]),
    "direct-cache256": (["gd"], {"N1GPU_CACHE_BLOCK": "256"}, "hbm-direct", ["cache_claim_1("], []),
    "direct-cache1024": (["gd"], {"N1GPU_CACHE_BLOCK": "1024"}, "hbm-direct", ["cache_claim_1("], []),
    "direct-nocache": (["gd"], {"N1GPU_NO_CACHE": "1"}, "hbm-direct", [], ["cache_claim"]),
    "direct-nopair": (["gd"], {"N1GPU_NO_MM_PAIR": "1"}, "hbm-direct", [], ["mmp"]),
    "direct-nosign": (["gd"], {"N1GPU_NO_SIGN_FROM_MINMAX": "1"}, "hbm-direct", [], []),
    "hash64": (["gd"], {"N1GPU_NO_DIRECT": "1"}, "hbm-hash-64", [], []),
    "hash128": (["gw1", "gw2"], {}, "hbm-hash-128", [], []),
}
MM_LAYOUTS = ["ungrouped", "dense-priv", "direct-cache1024", "direct-nopair", "hash64"]


def _query(table, keys, aggs, env, monkeypatch, params=None, where=None):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    qq = q.Query(table, "d", where, [K(c) for c in keys], aggs, params=params)
    for k in env:
        monkeypatch.delenv(k)
    return qq


def _layout_aggs(fx, layout):
    """Thread-private tables hold at most 48 words: with FLOAT addends MIN / MAX need class words, so that layout leaves
    them out."""
    return ["count(*)", "sum(%s)" % X, "avg(%s)" % X] if layout == "dense-priv" and T_FLOAT in fx.tags else AGGS


def _run_layout(fx, layout, monkeypatch):
    keys, env, mode, must, mustnot = LAYOUTS[layout]
    aggs = _layout_aggs(fx, layout)
    qq = _query(fx.table, keys, aggs, env, monkeypatch)
    assert qq.info["mode"] == mode, (fx.name, layout, qq.info)
    src = qq.kernel_source
    assert all(m in src for m in must) and not any(m in src for m in mustnot), (fx.name, layout)
    if layout == "dense-priv":
        assert qq.info["slots"] == 6  # mixed-radix: MISSING, NULL and four ints
    assert_exact(fx.expected(keys, aggs), gpu_rows(qq.execute(), aggs), "%s via %s" % (fx.name, layout))


# ---- GPU: value fixtures through every layout ------------------------------------------------------------------------
@pytest.fixture(scope="module")
def _device():
    q.init(0)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("name", VALUE_FIXTURES)
def test_int64_limits_through_every_layout(name, layout, _device, monkeypatch):
    _run_layout(fixture(name), layout, monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", MM_LAYOUTS)
@pytest.mark.parametrize("name", MM_FIXTURES)
def test_min_max_cells_at_the_edge_of_their_range(name, layout, _device, monkeypatch):
    _run_layout(fixture(name), layout, monkeypatch)


# ---- DISTINCT: biased values near the int64 limits --------------------------------------------------------------------
def _distinct_fixture(near_min):
    rng = np.random.default_rng(11 if near_min else 12)
    lo = I64_MIN if near_min else I64_MAX - 4095
    n = 40000
    keys = np.concatenate([[0, 0, 1, 2, 2, 3, 8191], rng.integers(4, 8191, n)])
    vals = [lo, lo, lo + 5, lo, lo + 1, lo + 4095, lo + 4095] + (lo + rng.integers(0, 4096, n)).tolist()
    if not near_min:  # group 0: only INT64_MAX, group 2: INT64_MAX and one below (overflow)
        vals[:5] = [I64_MAX, I64_MAX, lo + 5, I64_MAX, I64_MAX - 1]
    t, p = ints(vals)
    return Fixture("distinct_" + ("min" if near_min else "max"), keys, t, p, global_rows=1 << 20,
                   key_columns={"gk": [(T_INT, k) for k in range(8192)]})


DISTINCT_LAYOUTS = {
    "bitmap": ({"N1GPU_NO_PART": "1"}, lambda qq: not qq.part_source and "DISTINCT bitmap\n" in qq.kernel_source),
    "hashset": ({"N1GPU_NO_PART": "1", "N1GPU_NO_BITMAP": "1"}, lambda qq: not qq.part_source and "table_insert64(p.set_keys" in qq.kernel_source),
    "sliced-bitmap": ({"N1GPU_NO_PART": "1", "N1GPU_SET_PASSES": "2"}, lambda qq: not qq.part_source and "p.set_pass" in qq.kernel_source),
    "partitioned": ({"N1GPU_PART": "1"}, lambda qq: "NP " in qq.part_source),
}


@pytest.mark.parametrize("layout", list(DISTINCT_LAYOUTS))
def test_distinct_fixtures_land_on_their_set_layouts(layout, monkeypatch):
    env, check = DISTINCT_LAYOUTS[layout]
    for near_min in (True, False):
        qq = _query(distinct_fixture(near_min).table, ["gk"], DAGGS, env, monkeypatch)
        assert qq.info["mode"] == "hbm-direct" and check(qq), (near_min, layout)


@functools.lru_cache(maxsize=None)
def distinct_fixture(near_min):
    return _distinct_fixture(near_min)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", list(DISTINCT_LAYOUTS))
@pytest.mark.parametrize("near_min", [True, False], ids=["int64_min", "int64_max"])
def test_distinct_sums_of_biased_values(near_min, layout, _device, monkeypatch):
    """A group whose only distinct value is near INT64_MIN sums to a float (SUM(DISTINCT) starts from int 0); near
    INT64_MAX a single value stays an int and two overflow.  The partitioned path rebuilds the sum from popcounts as
    bias * count + code sum, and counts the codes below -bias as negative values."""
    fx = distinct_fixture(near_min)
    env, check = DISTINCT_LAYOUTS[layout]
    qq = _query(fx.table, ["gk"], DAGGS, env, monkeypatch)
    assert qq.info["mode"] == "hbm-direct" and check(qq), layout
    exp = fx.expected(["gk"], DAGGS, distinct=True)
    got = gpu_rows(qq.execute(), DAGGS)
    assert_exact(exp, got, "%s via %s" % (fx.name, layout))
    k0 = ("0",)
    assert isinstance(got[k0][DAGGS[2]], float if near_min else int)


# ---- merges of partial states: no rank overflows, the union does --------------------------------------------------------
def _merge_rows():
    """(group id, rank class, value): class 0 rows go to rank 0, class 1 rows spread over the other ranks."""
    step, rest = (1 << 47) - 1, I64_MAX - (1 << 16) * ((1 << 47) - 1)
    rows = []
    rows += [(0, 0, step)] * (1 << 16) + [(0, 0, rest), (0, 1, 1)]                  # rank 0 holds INT64_MAX, the union 2^63
    rows += [(1, 0, -(1 << 47))] * (1 << 16) + [(1, 1, -1), (1, 1, 0)]              # rank 0 INT64_MIN, the others -1 and 0
    rows += [(2, 0, 5)] * 3000 + [(2, 1, -3)] * 3000                                # each rank one sign, the union mixed
    rows += [(3, 0, I64_MAX), (3, 1, I64_MIN)]
    rows += [(4, 0, -1)] * 40000 + [(4, 1, 0xffffffff)] * 40000                      # low words 0xffffffff, opposite signs
    rows += [(5, 0, I64_MIN), (5, 1, None)]
    return rows


def _merge_tables(nranks):
    rows = _merge_rows()
    parts = [[] for _ in range(nranks)]
    c1 = 0
    for g, cls, v in rows:
        if cls == 0:
            parts[0].append((g, v))
        else:
            parts[1 + c1 % (nranks - 1)].append((g, v))
            c1 += 1
    fxs = []
    for r, p in enumerate(parts):
        p = [p[i] for i in np.random.default_rng(r).permutation(len(p))]
        fxs.append(Fixture("merge_rank%d" % r, [g for g, _v in p], [T_NULL if v is None else T_INT for _g, v in p],
                           [0 if v is None else v for _g, v in p]))
    whole = Fixture("merge", np.concatenate([f.gid for f in fxs]), np.concatenate([f.tags for f in fxs]), np.concatenate([f.pay for f in fxs]))
    return fxs, whole


def _unsealed(fx):
    t = q.Table(["x"] + sorted(fx.keys))
    t.set_column("x", fx.pay, tags=fx.tags)
    for c, spec in fx.keys.items():
        t.set_column(c, np.array([s[1] for s in spec], dtype=np.int64)[fx.gid], tags=np.array([s[0] for s in spec], dtype=np.uint8)[fx.gid])
    return t


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["direct-cache1024", "hash64"])
def test_two_rank_export_import_of_overflowing_sums(layout, _device, monkeypatch):
    """The Intermediate -> Final exchange on one GPU: each rank's partial sums fit int64 and are of one sign; the owner's
    merge of the exported records must overflow / mix signs exactly as one scan of all rows does."""
    import torch
    from query_b200 import dist as qd
    fxs, whole = _merge_tables(2)
    keys, env, mode, _must, _mustnot = LAYOUTS[layout]
    tables = [_unsealed(f) for f in fxs]
    qd.agree_local(tables)
    qs = []
    for t in tables:
        t.seal()
        qq = _query(t, keys, AGGS, env, monkeypatch)
        assert qq.info["mode"] == mode
        qq.scan_partial()
        qs.append(qq)
    assert len({x.kernel_source for x in qs}) == 1
    exported = []
    for qq in qs:
        ng, nd, rw = qq.partial_counts()
        recs = torch.zeros(max(1, ng) * rw, dtype=torch.int64, device="cuda")
        dents = torch.zeros(2, dtype=torch.int64, device="cuda")
        counts, dcounts = qq.partial_export(2, recs.data_ptr(), ng, dents.data_ptr(), nd)
        exported.append((recs, counts, rw))
    got = {}
    for owner, qq in enumerate(qs):
        qq.partial_reset()
        for recs, counts, rw in exported:
            o = int(counts[:owner].sum())
            r = recs[o * rw:(o + int(counts[owner])) * rw].contiguous()
            qq.partial_import(r.data_ptr() if counts[owner] else 0, int(counts[owner]), 0, 0)
        part = gpu_rows(qq.finalize(), AGGS)
        assert not (set(part) & set(got))
        got.update(part)
    assert_exact(whole.expected(keys, AGGS), got, "two-rank merge via " + layout)


@pytest.mark.gpu
@pytest.mark.parametrize("nranks", [2, 3])
def test_peer_arena_merge_of_overflowing_sums(nranks, _device):
    """The collective-free merge of direct-indexed tables (all ranks driven by this process on one device): rank r
    finalises slot range r of every rank's table; sums that overflow or mix signs only in the union come out exact."""
    from query_b200 import dist as qd
    fxs, whole = _merge_tables(nranks)
    tables = [_unsealed(f) for f in fxs]
    qd.agree_local(tables)
    mbs = [q.Mailbox(nranks, r, 1024, arena_bytes=16 << 20) for r in range(nranks)]
    for r in range(nranks):
        for o in range(nranks):
            mbs[r].set_peer(o, mbs[o].base)
    qs = []
    for r in range(nranks):
        tables[r].seal()
        qq = q.Query(tables[r], "d", None, [K("gd")], AGGS)
        assert qq.info["mode"] == "hbm-direct"
        qq.set_mailbox(mbs[r])
        qs.append(qq)
    assert len({x.kernel_source for x in qs}) == 1
    exp = whole.expected(["gd"], AGGS)
    for step in range(2):
        for qq in qs:
            qq.launch()
        got = {}
        for qq in qs:
            part = gpu_rows(qq.collect(), AGGS)
            assert not (set(part) & set(got))
            got.update(part)
        assert_exact(exp, got, "peer merge, %d ranks, step %d" % (nranks, step))


# ---- prepared-statement parameters that move the operand's range across the thresholds --------------------------------
PX = "(%s + $1)" % X
PAGGS = ["sum(%s)" % PX, "avg(%s)" % PX, "min(%s)" % PX, "max(%s)" % PX, "count(*)"]
PARAM_ROWS = 1 << 21  # declared keyspace rows of the parameter fixtures


def _param_groups(rng, with_floats):
    top = 1 << 20
    body = rng.integers(0, top - 4096, 60000)  # no value in (2^20 - 4096, 2^20): x + $1 overflowing never ties with an int
    g = {0: [ints([0, 5])], 1: [ints([top])], 2: [ints(body)], 3: [ints([top] * 20000 + [0])], 4: [ints(body[:30000] + 1)], 5: [absent(5), ints([3])]}
    if with_floats:
        g[4].append(floats(np.arange(50) + 0.5))
    return g


@functools.lru_cache(maxsize=None)
def param_fixture(with_floats):
    return grouped("params" + ("_f" if with_floats else ""), _param_groups(np.random.default_rng(21), with_floats), seed=21,
                   global_rows=PARAM_ROWS)


def _param_bindings():
    top = 1 << 20
    c_isum = _largest_rows_below(float(PARAM_ROWS), 2.3e18) - top   # max(|lo|, |hi|) * rows < 2.3e18 with hi = 2^20 + $1
    c_fc = _largest_rows_below(float(PARAM_ROWS), 9.0e15) - top
    c_w1 = (1 << 31) - 1 - top                                       # hi + $1 == 2^31 - 1: one-cell sums
    c_mm = I64_MAX - top                                             # hi + $1 == INT64_MAX: still a ranged INT
    # (binding, fixture with floats, kernel text present, kernel text absent)
    return [
        ("isum", c_isum, False, [], [".b >> 32)"]), ("isum+1", c_isum + 1, False, [".b >> 32)"], []),
        ("wide1", c_w1, False, ["cache_add_carry("], ["cache_add_wide("]), ("wide1+1", c_w1 + 1, False, ["cache_add_wide("], ["cache_add_carry("]),
        ("mm32", c_mm, False, ["cache_mm32", "mmp"], []), ("mm32+1", c_mm + 1, False, [], ["cache_mm32"]),
        ("fcarry", c_fc, True, ["num_f("], []), ("fcarry+1", c_fc + 1, True, [], ["num_f("]),
    ]


PARAM_BINDINGS = _param_bindings()


def _binding_markers(binding, monkeypatch):
    _id, c, with_floats, must, mustnot = binding
    fx = param_fixture(with_floats)
    qq = _query(fx.table, ["gd"], PAGGS, {}, monkeypatch, params={"1": c})
    assert qq.info["mode"] == "hbm-direct"
    src = qq.kernel_source
    assert all(m in src for m in must) and not any(m in src for m in mustnot), (_id, must, mustnot)
    return fx, qq, c


@pytest.mark.gpu
@pytest.mark.parametrize("binding", PARAM_BINDINGS, ids=[b[0] for b in PARAM_BINDINGS])
def test_parameter_bindings_across_the_thresholds(binding, _device, monkeypatch):
    fx, qq, c = _binding_markers(binding, monkeypatch)
    op = lambda v: O.num_add(O.num_add(0, v), c) if _is_num(v) else v  # arith_add.go: an int overflow gives a float
    assert_exact(fx.expected(["gd"], PAGGS, op=op), gpu_rows(qq.execute(), PAGGS), "binding %s = %d" % (binding[0], c))


# ---- CPU: the exact reference against the oracle ---------------------------------------------------------------------
def test_exact_reference_matches_the_oracle_on_same_sign_fixtures():
    """Where every int has one sign no evaluation order can overflow differently, so the oracle's sequential SUM must
    equal the exact reference, class included."""
    rng = np.random.default_rng(31)
    groups = {0: [ints([I64_MAX - 10, 4, 6])], 1: [ints([I64_MIN + 10, -4, -6])], 2: [ints([I64_MAX - 10, 4, 7])],
              3: [ints([I64_MIN + 10, -4, -7])], 4: [ints([0, 0, -1])], 5: [ints(rng.integers(0, 1 << 56, 40)), absent(4)]}
    for key_base in (-2, I64_MIN, I64_MAX - 3):
        fx = grouped("oracle", groups, seed=31, key_base=key_base)
        docs = []
        for g, t, p in zip(fx.gid.tolist(), fx.tags.tolist(), fx.pay.tolist()):
            fields = []
            kt, kv = fx.keys["g"][g]
            if kt != T_MISSING:
                fields.append('"g": %s' % ("null" if kt == T_NULL else kv))
            if t != T_MISSING:
                fields.append('"x": %s' % ("null" if t == T_NULL else p))
            docs.append("{%s}" % ", ".join(fields))
        parsed = [O.parse_document(d) for d in docs]
        want = {}
        for r in O.run_chain(parsed, "d", None, [K("g")], AGGS):
            k = tuple("MISSING" if v is O.MISSING else "null" if v is None else str(O.to_python(v)) for v in r.keys)
            want[k] = dict(r.aggregates)
        exp = fx.expected(["g"], AGGS)
        assert set(want) == set(exp)
        for k, (aggs, _approx) in exp.items():
            for a, v in aggs.items():
                assert type(want[k][a]) is type(v) and want[k][a] == v, (key_base, k, a, want[k][a], v)


def test_exact_reference_semantics():
    r, _ = exact_aggregates([I64_MAX, 1])
    assert r["sum"] == 2.0 ** 63 and isinstance(r["sum"], float)
    r, _ = exact_aggregates([I64_MIN])
    assert r["sum"] == I64_MIN and r["avg"] == I64_MIN and isinstance(r["avg"], int)
    r, _ = exact_aggregates([I64_MIN], distinct=True)
    assert r["sum"] == -(2.0 ** 63) and isinstance(r["sum"], float)
    r, _ = exact_aggregates([0, 0, -1])
    assert r["sum"] == -1.0 and isinstance(r["sum"], float)
    r, _ = exact_aggregates([5, -3, None, O.MISSING])
    assert (r["count*"], r["count"], r["countn"], r["sum"], r["avg"]) == (4, 2, 2, 2.0, 1)
    assert isinstance(r["sum"], float) and isinstance(r["avg"], int)
    r, _ = exact_aggregates([(1 << 62)] * 4 + [1])  # 2^64 + 1 rounds to 2^64
    assert r["sum"] == 2.0 ** 64


# ---- CPU: which side of every threshold a fixture lands on --------------------------------------------------------------
def _cpu_table(x, keys=None, global_rows=None, xtags=None, key_tags=None):
    cols = {"x": (np.asarray(x, dtype=np.int64), xtags)}
    if keys is not None:
        cols["gd"] = (np.asarray(keys, dtype=np.int64), key_tags)
    t = q.Table(sorted(cols))
    for c, (p, tg) in cols.items():
        t.set_column(c, p, tags=tg)
    if global_rows is not None:
        t.set_global_rows(global_rows)
    t.seal()
    return t


def _cpu_plan(t, keys, aggs, monkeypatch, env=None, params=None):
    qq = _query(t, keys, aggs, env or {}, monkeypatch, params=params)
    return qq.info, qq.kernel_source, qq.part_source


_KEYS = [-4500, 4500, 0, 7]


def _isum_side(mx, rows, monkeypatch):
    t = _cpu_table([mx, -mx, 1, 0], _KEYS, global_rows=rows)
    info, src, _ = _cpu_plan(t, ["gd"], AGGS, monkeypatch)
    return info["words"], ".b >> 32)" in src


@pytest.mark.parametrize("mx,rows", [(1 << 34, ISUM34_ROWS), (1 << 50, ISUM50_ROWS)], ids=["2^34", "2^50"])
def test_one_word_int_sum_up_to_its_proof(mx, rows, monkeypatch):
    """max|x| * rows_bound < 2.3e18: one `isum` word; one row more: the ilo / ihi split (one word more)."""
    w_in, split_in = _isum_side(mx, rows, monkeypatch)
    w_out, split_out = _isum_side(mx, rows + 1, monkeypatch)
    assert (split_in, split_out) == (False, True) and w_out == w_in + 1
    for name in ("isum34_in", "isum50_in", "isum34_out", "isum50_out"):  # the GPU fixtures: same rows, same sides
        fx = fixture(name)
        src = _query(fx.table, ["gd"], AGGS, {}, monkeypatch).kernel_source
        assert (".b >> 32)" in src) == name.endswith("_out"), name


def test_float_carried_sum_up_to_its_proof(monkeypatch):
    """imax * rows_bound < 9e15 with INT and FLOAT addends: one float64 word (num_f); one row more: int words + fsum."""
    x = np.array([1 << 36, 0, 0, 0], dtype=np.int64)
    x[3] = np.array([0.5]).view(np.int64)[0]
    tags = np.array([T_INT, T_INT, T_NULL, T_FLOAT], dtype=np.uint8)
    sides = [("num_f(" in _cpu_plan(_cpu_table(x, _KEYS, rows, tags), ["gd"], AGGS, monkeypatch)[1]) for rows in (FCARRY_ROWS, FCARRY_ROWS + 1)]
    assert sides == [True, False]
    for name, want in (("fcarry_in", True), ("fcarry_out", False)):
        fx = fixture(name)
        assert ("num_f(" in _query(fx.table, ["gd"], AGGS, {}, monkeypatch).kernel_source) == want, name


@pytest.mark.parametrize("lo,hi,keys,env,carry", [
    (-((1 << 31) - 1), (1 << 31) - 1, "gd", {}, True),
    (-(1 << 31), (1 << 31) - 1, "gd", {}, False),
    (-((1 << 31) - 1), 1 << 31, "gd", {}, False),
    (-((1 << 31) - 1), (1 << 31) - 1, "gd", {"N1GPU_NO_DIRECT": "1"}, False),  # carries go to a direct-indexed word only
], ids=["pm2^31-1", "lo=-2^31", "hi=2^31", "hashed"])
def test_one_cell_sum_needs_addends_within_2_31(lo, hi, keys, env, carry, monkeypatch):
    info, src, _ = _cpu_plan(_cpu_table([lo, hi, 0, 1], _KEYS), [keys], ["count(*)", "sum(%s)" % X], monkeypatch, env)
    assert ("cache_add_carry(" in src, "cache_add_wide(" in src) == (carry, not carry), info
    for name, want in (("wide1", True), ("wide", False)):
        assert ("cache_add_carry(" in _query(fixture(name).table, ["gd"], AGGS, {}, monkeypatch).kernel_source) == want


@pytest.mark.parametrize("lo,hi", _mm_ranges(), ids=[_mm_name(lo, hi) for lo, hi in _mm_ranges()])
def test_min_max_cells_are_32_bit_only_within_their_span(lo, hi, monkeypatch):
    """hi - lo <= 0xfffffffc: MIN and MAX in 32-bit cells (value - lo + 1), interleaved in pairs; wider: 64-bit cells."""
    small = hi - lo <= MM32_SPAN
    src = _cpu_plan(_cpu_table([lo, hi, lo, hi], _KEYS), ["gd"], AGGS, monkeypatch)[1]
    assert ("cache_mm32" in src, "mmp" in src) == (small, small)
    src = _cpu_plan(_cpu_table([lo, hi, lo, hi], _KEYS), ["gd"], AGGS, monkeypatch, {"N1GPU_NO_MM_PAIR": "1"})[1]
    assert ("cache_mm32<" in src, "mmp" in src) == (small, False)
    src = _query(fixture(_mm_name(lo, hi)).table, ["gd"], AGGS, {}, monkeypatch).kernel_source
    assert ("cache_mm32" in src) == small


def test_sign_mix_read_off_min_and_max(monkeypatch):
    """A SUM over an INT operand of both signs counts its negative addends unless MIN and MAX of the same operand are in
    the query."""
    t = _cpu_table([-5, 5, 0, 1], _KEYS)
    neg = lambda aggs, env=None: ".b < 0)" in _cpu_plan(t, ["gd"], aggs, monkeypatch, env)[1]
    assert not neg(AGGS)
    assert neg(AGGS, {"N1GPU_NO_SIGN_FROM_MINMAX": "1"})
    assert neg(["sum(%s)" % X, "min(%s)" % X]) and neg(["sum(%s)" % X])
    for one_sign in ([5, 6, 0, 1], [-5, -6, -1, -1]):  # a range of one sign needs no counter at all
        assert ".b < 0)" not in _cpu_plan(_cpu_table(one_sign, _KEYS), ["gd"], ["sum(%s)" % X], monkeypatch)[1]


@pytest.mark.parametrize("span,biased", [((1 << 62) - 1, True), (1 << 62, False)], ids=["2^62-1", "2^62"])
def test_key_bias_needs_a_range_below_2_62(span, biased, monkeypatch):
    """A key component of range < 2^62 is packed as value - lo (62 bits: hash-64); 2^62 and more keep all 64 bits of
    the value (hash-128)."""
    t = q.Table(["a", "x"])
    t.set_column("a", np.array([I64_MIN, I64_MIN + span, I64_MIN + 5], dtype=np.int64))
    t.set_column("x", np.array([1, 2, 3], dtype=np.int64))
    t.seal()
    info, src, _ = _cpu_plan(t, ["a"], ["count(*)", "sum(%s)" % X], monkeypatch)
    assert info["mode"] == ("hbm-hash-64" if biased else "hbm-hash-128")
    assert ("(u64)col0.b - (u64)" in src) == biased


@pytest.mark.parametrize("nkeys,rows,mode,claim", [
    (1 << 12, None, "dense-shared-memory", None),
    ((1 << 12) + 1, None, "hbm-direct", "cache_claim_1("),
    (1 << 22, 1 << 19, "hbm-direct", "cache_claim_1("),
    ((1 << 22) + 1, 1 << 19, "hbm-hash-64", "cache_claim_1("),
    (1 << 31, None, "hbm-hash-64", "cache_claim_1("),
    ((1 << 31) + 1, None, "hbm-hash-64", "cache_claim_n("),
], ids=["12bits", "13bits", "22bits", "23bits", "31bits", "32bits"])
def test_key_range_selects_the_table(nkeys, rows, mode, claim, monkeypatch):
    """Key bits <= 13 and a table of at most 40 KiB (here one word: 12 bits): shared memory; <= 22 with enough declared rows: direct-indexed; more:
    hashed; <= 31: u32 front-cache keys, more: 64-bit keys."""
    t = _cpu_table([1, 2], [I64_MIN + 17, I64_MIN + 17 + nkeys - 1], global_rows=rows)
    info, src, _ = _cpu_plan(t, ["gd"], ["count(*)"], monkeypatch)
    assert info["mode"] == mode
    if claim:
        assert claim in src


@pytest.mark.parametrize("vrange,part", [(4096, True), (4097, False)])
@pytest.mark.parametrize("lo", [I64_MIN, I64_MAX - 4096], ids=["int64_min", "int64_max"])
def test_partitioned_distinct_needs_a_12_bit_value(lo, vrange, part, monkeypatch):
    keys = np.arange(8192, dtype=np.int64)
    x = lo + (np.arange(8192) % vrange)
    x[-1] = lo + vrange - 1
    t = _cpu_table(x.astype(np.int64), keys, global_rows=1 << 20)
    info, _src, psrc = _cpu_plan(t, ["gd"], DAGGS, monkeypatch)
    assert info["mode"] == "hbm-direct" and bool(psrc) == part
    if part:
        fx = distinct_fixture(lo == I64_MIN)
        assert _query(fx.table, ["gk"], DAGGS, {}, monkeypatch).part_source


def test_gpu_fixtures_land_on_their_layouts(monkeypatch):
    """Every value fixture reaches the mode its GPU test asserts, so a planner change cannot move one elsewhere."""
    for name in VALUE_FIXTURES + MM_FIXTURES[:3]:
        fx = fixture(name)
        for layout, (keys, env, mode, must, mustnot) in LAYOUTS.items():
            qq = _query(fx.table, keys, _layout_aggs(fx, layout), env, monkeypatch)
            assert qq.info["mode"] == mode, (name, layout)
            src = qq.kernel_source
            assert all(m in src for m in must) and not any(m in src for m in mustnot), (name, layout)
