#!/usr/bin/env python
"""Scan-kernel time of `x IN <list>` as the unrolled in_arg chain and as the device-resident set (NqInSet).

Two 200 M-row columns, larger than the 126 MB L2 together and each alone: `n` (int64, uniform in [0, 10^9)) and `k`
(dictionary ranks of 100 000 words).  For list lengths 1-64 every statement is timed twice: with the list written out
as a literal (the chain up to codegen.hpp's IN_CHAIN_MAX, the set beyond) and bound to `$p` (always the set); lengths
10^3-10^6 are timed on the set alone, and the same scan without a filter as the floor.  Only count(*) is aggregated, so
each scan reads its filter column and nothing else.  Kernel time: CUDA events around the scan (last_scan_ns), median of
--reps runs after one warm-up run.  One JSON line per measurement; the first line names the GPU and its power limit.

Usage: python tools/in_set_perf.py [--rows N] [--reps R] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import query_b200 as q  # noqa: E402


def gpu_line():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in out.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=200_000_000)
    ap.add_argument("--reps", type=int, default=7)
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
    g = torch.Generator(device=dev).manual_seed(1)
    words = sorted("w%06d" % i for i in range(100_000))
    t = q.Table(["n", "k"])
    t.set_column_device("n", torch.randint(0, 1_000_000_000, (a.rows,), generator=g, device=dev, dtype=torch.int64))
    t.set_column_device("k", torch.randint(0, len(words), (a.rows,), generator=g, device=dev, dtype=torch.int32), dictionary=words)
    t.seal()
    torch.cuda.synchronize()
    rng = np.random.default_rng(2)

    def time_query(where, params):
        qq = q.Query(t, "d", where, [], ["count(*)"], params=params)
        qq.execute()
        ns = []
        for _ in range(a.reps):
            qq.execute()
            ns.append(qq.last_scan_ns)
        form = "set" if "in_set(" in qq.kernel_source else ("chain" if "in_arg(" in qq.kernel_source else "none")
        return form, float(np.median(ns)) / 1e3, float(min(ns)) / 1e3

    def elements(col, n):
        if col == "n":
            return rng.integers(0, 1_000_000_000, n).tolist()
        return [words[i] for i in rng.choice(len(words), min(n, len(words)), replace=False)]

    for col in ("n", "k"):
        form, us, best = time_query(None, None)
        emit(dict(col=col, length=0, how="no_filter", form=form, median_us=us, min_us=best))
        for length in (1, 2, 4, 6, 8, 12, 16, 20, 24, 32, 48, 64):
            el = elements(col, length)
            lst = "[" + ", ".join(json.dumps(x) for x in el) + "]"
            for how, where, params in (("literal", "((`d`.`%s`) in %s)" % (col, lst), None), ("param", "((`d`.`%s`) in $p)" % col, {"p": el})):
                form, us, best = time_query(where, params)
                emit(dict(col=col, length=length, how=how, form=form, median_us=us, min_us=best))
        for length in (1_000, 10_000, 100_000, 1_000_000):
            if col == "k" and length > len(words):
                continue
            form, us, best = time_query("((`d`.`%s`) in $p)" % col, {"p": elements(col, length)})
            emit(dict(col=col, length=length, how="param", form=form, median_us=us, min_us=best))


if __name__ == "__main__":
    main()
