#!/usr/bin/env python
"""Scan-kernel time of GROUP BY keys wider than 127 bits (the hbm-hash-wide table) next to the 128-bit hash table.

Device-resident columns of --rows rows (default 200 M; 1.6 GB each, far beyond the 126 MB L2): a, b, c hold int64 values
over the whole range (both limits occur, so every one packs as 64 bits) and d = b >> 2 (62 bits).  Each row takes one of
G key tuples, G = 10^3 and 10^6, drawn uniformly.  Three chains per G, all with count(*) and sum(a):
  wide3  GROUP BY a, b, c   192 bits, 3 key words
  wide2  GROUP BY a, b      128 bits, 2 key words (the narrowest wide key)
  h128   GROUP BY a, d      126 bits: the hbm-hash-128 table over the same groups
Kernel time: CUDA events around the scan (last_scan_ns), median of --reps runs after two warm-up runs (the first grows the
table to its final capacity).  One JSON line per measurement; the first names the GPU and its power limit.

Usage: python tools/wide_key_perf.py [--rows N] [--reps R] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import query_b200 as q  # noqa: E402

I64_MIN, I64_MAX = -(1 << 63), (1 << 63) - 1
CHAINS = {"wide3": ("a", "b", "c"), "wide2": ("a", "b"), "h128": ("a", "d")}


def gpu_line():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in out.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=200_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    q.init(0)
    sink = open(a.out, "w") if a.out else None

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        if sink:
            sink.write(line + "\n")
            sink.flush()

    emit(dict(gpu_line(), rows=a.rows, reps=a.reps))
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(7)
    for groups in (1_000, 1_000_000):
        pool = rng.integers(I64_MIN, I64_MAX, (groups, 3), dtype=np.int64, endpoint=True)
        pool[0, :], pool[1, :] = I64_MIN, I64_MAX
        pool_d = torch.from_numpy(pool).to(dev)
        g = torch.Generator(device=dev).manual_seed(groups)
        idx = torch.randint(0, groups, (a.rows,), generator=g, device=dev)
        idx[0], idx[1] = 0, 1
        t = q.Table(["a", "b", "c", "d"])
        for k, name in enumerate("abc"):
            t.set_column_device(name, pool_d[:, k][idx].contiguous())
        t.set_column_device("d", (pool_d[:, 1][idx] >> 2).contiguous())
        del idx
        t.seal()
        torch.cuda.synchronize()
        for chain, cols in CHAINS.items():
            qq = q.Query(t, "d", None, ["(`d`.`%s`)" % c for c in cols], ["count(*)", "sum((`d`.`a`))"])
            qq.execute()
            r = qq.execute()
            ns = []
            for _ in range(a.reps):
                r = qq.execute()
                ns.append(qq.last_scan_ns)
            med = float(np.median(ns))
            info = qq.info
            emit({"chain": chain, "keys": list(cols), "groups": groups, "found_groups": r.num_groups, "mode": info["mode"],
                  "registers": info["registers"], "grid": info["grid"], "block": info["block"], "slots": info["slots"],
                  "kernel_us_median": med / 1e3, "kernel_us_all": [x / 1e3 for x in ns], "ns_per_row": med / a.rows,
                  "rows_per_s": a.rows / (med * 1e-9)})
            del qq
        del t
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
