"""n1gpu_table_set_column_device: columns handed over in device memory give the same table (statistics, widths,
results) as the same columns handed over in host memory."""
import os

import numpy as np
import pytest

import query_b200 as q

pytestmark = pytest.mark.gpu

QUERIES = [
    ("((`d`.`n`) between 100 and 700)", [], ["count(*)", "sum((`d`.`n`))", "avg((`d`.`x`))", "min((`d`.`x`))", "max((`d`.`n`))"]),
    (None, ["(`d`.`s`)"], ["count(*)", "sum((`d`.`x`))", "min((`d`.`n`))", "max((`d`.`s`))", "count(distinct (`d`.`n`))"]),
    ("((`d`.`s`) >= \"k3\")", ["(`d`.`s`)", "(`d`.`n`)"], ["count((`d`.`x`))", "countn((`d`.`x`))"]),
]


def _columns(n, seed):
    rng = np.random.default_rng(seed)
    nn = rng.integers(-50, 1000, n, dtype=np.int64)
    ntag = np.full(n, 4, dtype=np.uint8)
    r = rng.integers(0, 10, n)
    ntag[r == 0] = 0  # MISSING
    ntag[r == 1] = 1  # NULL
    # x: floats, a third of them integral (must be canonicalised to ints), some booleans
    x = np.where(rng.integers(0, 3, n) == 0, rng.integers(-5, 5, n).astype(np.float64), rng.random(n) * 100 - 50)
    xtag = np.full(n, 5, dtype=np.uint8)
    r = rng.integers(0, 12, n)
    xtag[r == 0] = 1
    xtag[r == 1] = 2  # false
    xtag[r == 2] = 3  # true
    words = sorted("k%d" % i for i in range(40))
    s = rng.integers(0, len(words), n).astype(np.uint32)
    stag = np.full(n, 6, dtype=np.uint8)
    stag[rng.integers(0, 9, n) == 0] = 0
    return (nn, ntag), (x, xtag), (s, stag, words)


def _same(a, b):
    """same groups and values; float64 sums of a grouped scan are accumulated with atomics in arrival order, so
    floats are compared within the 1e-12 relative tolerance the path promises"""
    ra = sorted(a.rows(), key=lambda r: repr(r[0]))
    rb = sorted(b.rows(), key=lambda r: repr(r[0]))
    assert len(ra) == len(rb)
    for (ka, va), (kb, vb) in zip(ra, rb):
        assert repr(ka) == repr(kb)
        for x, y in zip(va, vb):
            if isinstance(x, float) and isinstance(y, float):
                assert abs(x - y) <= 1e-12 * max(abs(x), abs(y)), (ka, x, y)
            else:
                assert type(x) is type(y) and x == y, (ka, x, y)


@pytest.mark.parametrize("n", [0, 1, 4097, 200_000])
def test_device_columns_match_host_columns(n):
    import torch
    q.init(0)
    (nn, ntag), (x, xtag), (s, stag, words) = _columns(n, 7 + n)
    th = q.Table(["n", "x", "s"])
    th.set_column("n", nn, tags=ntag)
    th.set_column("x", x, tags=xtag)
    th.set_column("s", s, tags=stag, dictionary=words)
    th.seal()
    td = q.Table(["n", "x", "s"])
    dev = torch.device("cuda:0")
    td.set_column_device("n", torch.from_numpy(nn).to(dev), tags=torch.from_numpy(ntag).to(dev))
    td.set_column_device("x", torch.from_numpy(x).to(dev), tags=torch.from_numpy(xtag).to(dev))
    td.set_column_device("s", torch.from_numpy(s.astype(np.int32)).to(dev), tags=torch.from_numpy(stag).to(dev), dictionary=words)
    td.seal()
    assert td.num_rows == th.num_rows == n
    for c in ("n", "x", "s"):
        assert list(td.stats(c)[:5]) == list(th.stats(c)[:5]), c
    if n == 0:
        return
    for where, keys, aggs in QUERIES:
        a = q.Query(th, "d", where, keys, aggs).execute()
        b = q.Query(td, "d", where, keys, aggs).execute()
        _same(a, b)


def test_host_and_device_columns_do_not_mix():
    import torch
    q.init(0)
    t = q.Table(["a", "b"])
    t.set_column("a", np.arange(10, dtype=np.int64))
    with pytest.raises(q.N1GpuError):
        t.set_column_device("b", torch.arange(10, dtype=torch.int64, device="cuda:0"))
    t2 = q.Table(["a", "b"])
    t2.set_column_device("a", torch.arange(10, dtype=torch.int64, device="cuda:0"))
    with pytest.raises(q.N1GpuError):
        t2.seal()  # column b never set


def test_send_stop_aborts_a_running_scan(monkeypatch):
    """execution/base.go:313-338: SendStop may arrive from any goroutine at any time and must make the operator stop.  A scan
    in flight polls the cancel word (mapped pinned memory) once per 32 tiles per warp: n1gpu_query_cancel during a long scan
    makes collect fail with N1GPU_E_CANCELLED well before the scan would have finished."""
    import sys
    import time
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import torch
    import workloads as wl
    monkeypatch.setenv("N1GPU_NO_CACHE", "1")  # every row of a hot Zipf key is an L2 atomic on one address: a slow scan
    w = wl.Config5(scale=0.2)  # a scan of about 20 ms on a B200: long enough to stop well before its end
    t = w.sealed_table()
    qq = w.query(t)
    qq.execute()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    qq.execute()
    full = time.perf_counter() - t0
    qq.launch()
    time.sleep(min(0.002, full / 20))
    t0 = time.perf_counter()
    qq.cancel()
    with pytest.raises(q.N1GpuError) as e:
        qq.collect()
    stopped = time.perf_counter() - t0
    assert e.value.code == -6, e.value  # N1GPU_E_CANCELLED
    assert full > 0.01 and stopped < full / 3, (full, stopped)
