"""Every way a table is filled gives the same column statistics and scan widths, and the entry points of a table accept
or refuse each other in one fixed order.

Statistics words (n1gpu_table_stats_get): class mask, has int, int min, int max, has float, dictionary size, rank of ""
(-1: absent), rows that are MISSING or NULL."""
import json
import math

import numpy as np
import pytest

import query_b200 as q

MISSING, NULL, FALSE, TRUE, INT, FLOAT, STRING, OTHER = range(8)
E_INVALID = -1

DOCS = [
    '{"i": 3, "f": 1.5, "s": "", "b": true, "n": null}',
    '{"i": -7, "f": 2.0, "s": "x", "b": false}',
    '{"i": 4.0, "s": "abc", "n": null, "f": "str", "b": 1}',
    'not json',
    '"a string"',
    '{"i": [1], "f": -0.25, "s": {"k": 1}, "n": null}',
    '{"i": 9223372036854775807, "s": "x", "b": false}',
    '{}',
]
COLS = ["i", "f", "s", "b", "n", "z"]  # z: never present


def _classify(v):
    if v is None:
        return NULL, None
    if v is True or v is False:
        return (TRUE if v else FALSE), None
    if isinstance(v, int):
        return INT, v
    if isinstance(v, float):
        return (INT, int(v)) if v == math.floor(v) and abs(v) < 2.0 ** 63 else (FLOAT, v)
    if isinstance(v, str):
        return STRING, v
    return OTHER, None


def _rows(docs, col):
    out = []
    for d in docs:
        try:
            o = json.loads(d)
        except ValueError:
            o = None
        out.append(_classify(o[col]) if isinstance(o, dict) and col in o else (MISSING, None))
    return out


def _expected(rows, dict_built=True):
    """the 8 statistics words of a column holding `rows` ((class, value) pairs, integral floats already INT)"""
    mask = 0
    ints = [v for c, v in rows if c == INT]
    strs = sorted({v.encode() for c, v in rows if c == STRING})
    for c, _v in rows:
        mask |= 1 << c
    ndict = len(strs) if dict_built else 0
    empty_rank = 0 if dict_built and strs and strs[0] == b"" else -1
    return [mask, int(bool(ints)), min(ints) if ints else 0, max(ints) if ints else 0, int(any(c == FLOAT for c, _ in rows)),
            ndict, empty_rank, sum(1 for c, _ in rows if c <= NULL)]


def _scan_bytes(stats):
    mask = stats[0]
    width = 8 if mask & ((1 << INT) | (1 << FLOAT)) else 4 if mask & (1 << STRING) else 0
    return width + (0 if mask and not mask & (mask - 1) else 1)


def _check(t, cols, rows_of, dict_built_before):
    """stats before seal (word 6 aside: see test_empty_rank_before_seal_is_the_sealed_one), then after seal, and scan_bytes"""
    for c in cols:
        got = list(t.stats(c))
        want = _expected(rows_of[c], dict_built_before)
        assert got[:6] + got[7:] == want[:6] + want[7:], (c, got, want)
    t.seal()
    for c in cols:
        want = _expected(rows_of[c])
        assert list(t.stats(c)) == want, (c, list(t.stats(c)), want)
        assert t.scan_bytes(c) == _scan_bytes(want), c


@pytest.mark.parametrize("threads", [1, 0])
def test_append_json_statistics(threads):
    t = q.Table(COLS)
    t.append_json(DOCS, threads=threads)
    _check(t, COLS, {c: _rows(DOCS, c) for c in COLS}, dict_built_before=False)


def test_load_ndjson_statistics(tmp_path):
    path = tmp_path / "docs.ndjson"
    path.write_text("\n".join(d for d in DOCS if "\n" not in d) + "\n")
    t = q.Table(COLS)
    t.load_ndjson(str(path), threads=2)
    _check(t, COLS, {c: _rows(DOCS, c) for c in COLS}, dict_built_before=False)


def test_load_segment_statistics(tmp_path):
    path = str(tmp_path / "seg.n1seg")
    w = q.Table(COLS)
    w.set_segment_output(path, "tag")
    w.append_json(DOCS, threads=1)
    w.seal()
    t = q.Table(COLS)
    assert t.load_segment(path, "tag")
    _check(t, COLS, {c: _rows(DOCS, c) for c in COLS}, dict_built_before=True)


def _host_columns():
    """(payload, tags, dictionary, rows) per column for set_column: integral floats tagged FLOAT, absent-only, booleans,
    "" in a dictionary"""
    f = np.array([2.0, 1.5, -3.0, 0.0, 7.25], dtype=np.float64)
    ftag = np.array([FLOAT, FLOAT, FLOAT, NULL, FLOAT], dtype=np.uint8)
    n = np.zeros(5, dtype=np.int64)
    ntag = np.array([MISSING, NULL, NULL, MISSING, MISSING], dtype=np.uint8)
    b = np.zeros(5, dtype=np.int64)
    btag = np.array([TRUE, FALSE, TRUE, MISSING, TRUE], dtype=np.uint8)
    words = ["", "k", "kk"]
    s = np.array([0, 2, 1, 0, 2], dtype=np.uint32)
    stag = np.array([STRING, STRING, STRING, NULL, STRING], dtype=np.uint8)
    i = np.array([5, -9, 12, 0, 3], dtype=np.int64)
    return {
        "f": (f, ftag, None, [_classify(float(v)) if c == FLOAT else (c, None) for v, c in zip(f, ftag)]),
        "n": (n, ntag, None, [(c, None) for c in ntag]),
        "b": (b, btag, None, [(c, None) for c in btag]),
        "s": (s, stag, words, [(STRING, words[v]) if c == STRING else (c, None) for v, c in zip(s, stag)]),
        "i": (i, None, None, [(INT, int(v)) for v in i]),
    }


def test_set_column_statistics():
    cols = _host_columns()
    t = q.Table(list(cols))
    for c, (pay, tags, words, _rows_) in cols.items():
        t.set_column(c, pay, tags=tags, dictionary=words)
    _check(t, list(cols), {c: v[3] for c, v in cols.items()}, dict_built_before=True)


def test_stats_leave_staged_rows_alone():
    """an integral FLOAT counts as INT in the statistics; the staged row stays what was set until seal canonicalises it"""
    f, ftag, _w, _r = _host_columns()["f"]
    t = q.Table(["f"])
    t.set_column("f", f, tags=ftag)
    assert list(t.stats("f")[:4]) == [(1 << INT) | (1 << FLOAT) | (1 << NULL), 1, -3, 2]
    pay, tags = t.peek("f")
    assert list(tags) == list(ftag)
    assert list(pay.view(np.float64)[ftag == FLOAT]) == list(f[ftag == FLOAT])


@pytest.mark.parametrize("fill", ["none", "append", "set_column"])
def test_empty_table_statistics(fill):
    t = q.Table(["a"])
    if fill == "append":
        t.append_json([], threads=1)
    elif fill == "set_column":
        t.set_column("a", np.zeros(0, dtype=np.int64))
    _check(t, ["a"], {"a": []}, dict_built_before=True)


def test_empty_rank_before_seal_is_the_sealed_one(tmp_path):
    """the rank of "" is read from the column's dictionary whether or not the table is sealed"""
    cols = _host_columns()
    t = q.Table(["s"])
    t.set_column("s", cols["s"][0], tags=cols["s"][1], dictionary=cols["s"][2])
    before = int(t.stats("s")[6])
    t.seal()
    assert before == int(t.stats("s")[6]) == 0
    t = q.Table(COLS)
    t.append_json(DOCS, threads=1)
    t.dictionary("s")  # builds the dictionary
    before = int(t.stats("s")[6])
    t.seal()
    assert before == int(t.stats("s")[6]) == 0


# ---- which entry point may follow which -------------------------------------------------------------------------------

def _segment(tmp_path):
    path = str(tmp_path / "ab.n1seg")
    w = q.Table(["a", "b"])
    w.set_segment_output(path, "tag")
    w.append_json(['{"a": 1, "b": "x"}', '{"a": 2.0, "b": ""}'], threads=1)
    w.seal()
    return path


def _blob(strings):
    enc = [s.encode() for s in strings]
    offs = np.zeros(len(enc) + 1, dtype=np.int64)
    if enc:
        np.cumsum([len(e) for e in enc], out=offs[1:])
    return np.frombuffer(b"".join(enc) or b"\0", dtype=np.uint8)[: int(offs[-1])].copy(), offs


def _ops(segment):
    return {
        "append_json": lambda t: t.append_json(['{"a": 1, "b": "x"}', '{"a": 2.5, "b": ""}'], threads=1),
        "set_column": lambda t: (t.set_column("a", np.array([1, 2], dtype=np.int64)),
                                 t.set_column("b", np.array([1, 0], dtype=np.uint32), dictionary=["", "x"])),
        "load_segment": lambda t: t.load_segment(segment, "tag"),
        "export": lambda t: t.dictionary("b"),
        "import": lambda t: t.import_dictionary("b", ["", "w", "x", "y"]),
        "merge": lambda t: t.merge_dictionaries("b", [_blob(["v", "x"])]),
        "set_stats": lambda t: t.set_stats("a", [1 << INT, 1, 1, 2, 0, 0, -1, 0]),
        "seal": lambda t: t.seal(),
    }


def _outcome(fn, t):
    try:
        r = fn(t)
    except q.N1GpuError as e:
        return e.code
    return "refused" if r is False else "ok"  # load_segment: False = the file was not loaded


# (first, second) -> outcome of the second; every pair not listed is accepted
REFUSED = {
    ("append_json", "set_column"): E_INVALID,
    ("append_json", "load_segment"): E_INVALID,
    ("set_column", "append_json"): E_INVALID,
    ("set_column", "load_segment"): E_INVALID,
    ("load_segment", "append_json"): E_INVALID,
    ("load_segment", "set_column"): E_INVALID,
    ("load_segment", "load_segment"): E_INVALID,
    ("export", "append_json"): E_INVALID,
    ("import", "append_json"): E_INVALID,
    ("merge", "append_json"): E_INVALID,
    ("merge", "import"): E_INVALID,  # the merged dictionary holds "v", the imported one does not
    ("seal", "append_json"): E_INVALID,
    ("seal", "set_column"): E_INVALID,
    ("seal", "load_segment"): E_INVALID,
    ("seal", "export"): E_INVALID,
    ("seal", "import"): E_INVALID,
    ("seal", "merge"): E_INVALID,
    ("seal", "set_stats"): E_INVALID,
}


def test_entry_point_order(tmp_path):
    ops = _ops(_segment(tmp_path))
    got = {}
    for first in ops:
        for second in ops:
            t = q.Table(["a", "b"])
            assert _outcome(ops[first], t) == "ok", first
            got[(first, second)] = _outcome(ops[second], t)
    want = {k: REFUSED.get(k, "ok") for k in got}
    assert got == want, {k: (got[k], want[k]) for k in got if got[k] != want[k]}


def test_bad_input_is_refused(tmp_path):
    def code(fn):
        with pytest.raises(q.N1GpuError) as e:
            fn()
        return e.value.code

    t = q.Table(["a", "b"])
    t.set_column("a", np.arange(3, dtype=np.int64))
    assert code(lambda: t.set_column("b", np.arange(4, dtype=np.int64))) == E_INVALID  # length mismatch
    t = q.Table(["a"])  # the width comes from the dtype: a bad one only through the C ABI
    pay = np.zeros(1, dtype=np.int64)
    assert q.lib().n1gpu_table_set_column(t._h, 0, 2, pay.ctypes.data, None, 1, None, None, 0) == E_INVALID
    t = q.Table(["s"])
    assert code(lambda: t.set_column("s", np.zeros(2, dtype=np.uint32), dictionary=["b", "a"])) == E_INVALID
    t = q.Table(["s"])
    assert code(lambda: t.import_dictionary("s", ["x", "x"])) == E_INVALID
    assert code(lambda: t.merge_dictionaries("s", [_blob(["b", "a"])])) == E_INVALID
    t = q.Table(["a"])
    t.set_column("a", np.arange(3, dtype=np.int64), tags=np.array([INT, 9, INT], dtype=np.uint8))
    assert code(t.seal) == E_INVALID  # bad class byte


# ---- the device routes ------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_device_shredder_statistics_match_host():
    from test_gpu_shredder import EDGE_DOCS
    q.init(0)
    cols = ["a", "s", "c", "n.a", "x"]
    th, td = q.Table(cols), q.Table(cols)
    th.append_json(EDGE_DOCS, threads=1)
    td.append_json(EDGE_DOCS, threads=-1)
    th.seal()
    td.seal()
    for c in cols:
        assert list(td.stats(c)) == list(th.stats(c)), c
        assert td.scan_bytes(c) == th.scan_bytes(c), c


@pytest.mark.gpu
def test_device_columns_refuse_host_input(tmp_path):
    import torch
    q.init(0)
    dev = torch.device("cuda:0")
    segment = _segment(tmp_path)
    ops = _ops(segment)
    for first in ("set_column_device", "append_json_device"):
        for second, fn in ops.items():
            t = q.Table(["a", "b"])
            if first == "set_column_device":
                t.set_column_device("a", torch.arange(2, dtype=torch.int64, device=dev))
                t.set_column_device("b", torch.tensor([1, 0], dtype=torch.int32, device=dev), dictionary=["", "x"])
            else:
                t.append_json(['{"a": 1, "b": "x"}', '{"a": 2.5, "b": ""}'], threads=-1)
            got = _outcome(fn, t)
            refused = second in ("append_json", "set_column", "load_segment")
            assert got == (E_INVALID if refused else "ok"), (first, second, got)
    t = q.Table(["a", "b"])
    t.set_column("a", np.arange(10, dtype=np.int64))
    with pytest.raises(q.N1GpuError) as e:
        t.set_column_device("b", torch.arange(10, dtype=torch.int64, device=dev))
    assert e.value.code == E_INVALID
    t = q.Table(["a", "b"])
    t.set_column_device("a", torch.arange(10, dtype=torch.int64, device=dev))
    with pytest.raises(q.N1GpuError) as e:
        t.set_column_device("b", torch.arange(11, dtype=torch.int64, device=dev))
    assert e.value.code == E_INVALID  # length mismatch
    with pytest.raises(q.N1GpuError) as e:
        t.seal()  # column b never set
    assert e.value.code == E_INVALID
    t = q.Table(["a"])
    with pytest.raises(q.N1GpuError) as e:
        t.set_column_device("a", torch.tensor([1, 2], dtype=torch.int64, device=dev), tags=torch.tensor([4, 9], dtype=torch.uint8, device=dev))
    assert e.value.code == E_INVALID  # bad class byte


@pytest.mark.gpu
def test_device_shredded_statistics_after_import():
    q.init(0)
    docs = ['{"s": "b", "a": 1}', '{"s": "", "a": 2.0}', '{"a": 0.5}', '{"s": "d"}']
    t = q.Table(["s", "a"])
    t.append_json(docs, threads=-1)
    before = list(t.stats("s"))
    t.import_dictionary("s", ["", "a", "b", "c", "d"])
    after = list(t.stats("s"))
    assert after == before[:5] + [5, 0] + before[7:]
    assert list(t.stats("a")) == _expected(_rows(docs, "a"))
    assert t.dictionary("s") == [b"", b"a", b"b", b"c", b"d"]
    t.seal()
    assert list(t.stats("s")) == after
    assert t.scan_bytes("s") == 5 and t.scan_bytes("a") == 9
