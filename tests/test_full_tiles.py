"""The cached GROUP BY scan runs phase 1 (filter, group key, front-cache probe) of a full 128-row warp tile without the
per-row bounds check; only the grid's last tile takes the checked copy.  The front cache's u32 keys and 32-bit cells are
addressed through 32-bit shared-memory addresses made once per kernel.  Pinned on the generated text (no GPU needed)."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import query_b200 as q  # noqa: E402

AGGS = ["count(*)", "count((`d`.`v`))", "sum((`d`.`v`))", "min((`d`.`v`))", "max((`d`.`v`))"]


def config5_table(n, seed=5, vocab=100000):
    """config 5's shape: k a dictionary string with MISSING and NULL rows, v an int64 with MISSING and NULL rows"""
    rng = np.random.default_rng(seed)
    t = q.Table(["k", "v"])
    r = rng.integers(0, 10, n)
    t.set_column("k", rng.integers(0, vocab, n).astype(np.uint32), tags=np.where(r == 0, 0, np.where(r == 1, 1, 6)).astype(np.uint8),
                 dictionary=["w%06d" % i for i in range(vocab)])
    r = rng.integers(0, 10, n)
    t.set_column("v", rng.integers(-1000, 1000000, n, dtype=np.int64), tags=np.where(r == 0, 0, np.where(r == 1, 1, 4)).astype(np.uint8))
    t.set_global_rows(1_000_000_000)
    t.seal()
    return t


def test_cached_scan_checks_bounds_only_on_the_last_tile():
    t = config5_table(200000)
    src = q.Query(t, "d", "((`d`.`v`) is not missing)", ["(`d`.`k`)"], AGGS).kernel_source
    assert "if (wbase + 128 <= nrows) {" in src
    assert src.count("bool pass = NQ_IN_RANGE(j);") == 2
    assert "#define NQ_IN_RANGE(j) true" in src and "#define NQ_IN_RANGE(j) (base + (j) < nrows)" in src
    # the probe is emitted once per copy; the update phases are emitted once
    assert src.count("cache_claim_1(") == 2 and src.count("__ballot_sync(0xffffffffu, cs[j] >= 0)") == 1
    # every cache access of the row loop goes through the hoisted shared addresses, none through s_ckey / s_c32
    assert "const u32 a_ckey = smem_addr(s_ckey), a_c32 = smem_addr(s_c32);" in src
    loop = src[src.index("for (i64 wbase"):src.index("    __syncthreads();\n    for (int i = threadIdx.x; i < NQ_CS")]
    assert "s_ckey" not in loop and "&s_c32[" not in loop and "cache_claim_1(a_ckey," in loop
    assert all("a_c32 + 4 * (" in line for line in src.splitlines() if line.startswith("#define ACCH_"))


@pytest.mark.parametrize("keys", [[], ["(`d`.`v`)"]])
def test_uncached_modes_keep_one_checked_row_loop(keys):
    """ungrouped and shared-memory dense scans have no front cache: their row loop is unchanged"""
    t = q.Table(["v"])
    t.set_column("v", np.arange(1000, dtype=np.int64) % 7)
    t.seal()
    src = q.Query(t, "d", "((`d`.`v`) > 2)", keys, ["count(*)", "sum((`d`.`v`))"]).kernel_source
    assert "NQ_IN_RANGE" not in src and "wbase + 128 <= nrows" not in src
    assert src.count("bool pass = base + j < nrows;") == 1

