"""Refresh of a resident directory keyspace after document writes, against a load from scratch (B200 only).

Builds a file-datastore keyspace of N config-2-shaped documents ({"n": int, "f": float}, one file each), loads it once
through the operator, then for every k rewrites k documents in place and times the operator build + run_once that
follows (the refresh: k documents read, the columns spliced in HBM).  The baseline is a load from scratch of the same
files under another path (a symbolic link: another keyspace to the resident-table cache, the same page-cached files).
Phases come from the library's N1GPU_TRACE lines ("[n1gpu load|refresh] <phase> <ms>").  Writes JSONL to --out with the
card name and power limit."""
import argparse
import json
import os
import random
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
os.environ["N1GPU_TRACE"] = "1"

import query_b200 as q  # noqa: E402
from plans_n1 import explain_plan  # noqa: E402

WHERE = "((`d`.`n`) between 250000 and 749999)"
AGGS = ["count(*)", "count((`d`.`n`))", "sum((`d`.`n`))", "avg((`d`.`n`))", "min((`d`.`n`))", "max((`d`.`n`))", "sum((`d`.`f`))"]
PHASE = re.compile(r"^\[n1gpu (load|refresh)\] (\S+)\s+([0-9.]+) ms$")


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True)
    name, power = out.stdout.strip().splitlines()[0].split(", ")
    return name, power


def doc(rnd):
    return '{"n": %d, "f": %.6f}' % (rnd.randrange(1_000_000), rnd.randrange(1, 1_000_000) / 1e6)


def timed_build(plan, root):
    """operator build + run_once, wall time after the device is idle again; the trace lines of this build"""
    err = tempfile.TemporaryFile(mode="w+")
    saved = os.dup(2)
    os.dup2(err.fileno(), 2)
    try:
        t0 = time.perf_counter()
        op = q.Operator(plan, root)
        op.run_once()
        ms = (time.perf_counter() - t0) * 1e3
    finally:
        os.dup2(saved, 2)
        os.close(saved)
    err.seek(0)
    phases = {}
    for line in err.read().splitlines():
        m = PHASE.match(line.strip())
        if m:
            key = m.group(1) + "." + m.group(2)
            phases[key] = round(phases.get(key, 0.0) + float(m.group(3)), 3)
    return ms, op.marshal_json().get("#stats", {}).get("#docsRead", 0), phases


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="100000,1000000")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_refresh.jsonl"))
    ap.add_argument("--workdir", default=None, help="where the keyspaces are written (default: a temporary directory)")
    a = ap.parse_args()
    q.init(0)
    name, power = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    work = tempfile.mkdtemp(prefix="n1refresh", dir=a.workdir)
    plan = explain_plan("default", "d", "d", WHERE, [], AGGS)
    with open(a.out, "a") as out:
        for n in [int(s) for s in a.sizes.split(",")]:
            rnd = random.Random(n)
            root = os.path.join(work, "n%d" % n)
            d = os.path.join(root, "default", "d")
            try:
                os.makedirs(d)
                for i in range(n):
                    with open(os.path.join(d, "k%08d.json" % i), "w") as f:
                        f.write(doc(rnd))
            except OSError as e:  # the file system holds no more files
                out.write(json.dumps({"N": n, "measured": False, "why": str(e), "card": name, "power_limit": power}) + "\n")
                continue
            time.sleep(0.05)
            first_ms, first_read, first_phases = timed_build(plan, root)
            out.write(json.dumps({"N": n, "k": "initial load", "ms": round(first_ms, 3), "docsRead": first_read, "phases": first_phases,
                                  "card": name, "power_limit": power}) + "\n")
            for j, k in enumerate(sorted({0, 1, 100, 10_000, n // 2, n})):
                if k > n:
                    continue
                for i in rnd.sample(range(n), k):
                    with open(os.path.join(d, "k%08d.json" % i), "w") as f:
                        f.write(doc(rnd))
                time.sleep(0.05)  # past the racily-clean margin
                ms, read, phases = timed_build(plan, root)
                cold_root = os.path.join(work, "cold%d_%d" % (n, j))
                os.symlink(root, cold_root)
                cold_ms, cold_read, cold_phases = timed_build(plan, cold_root)
                rec = {"N": n, "k": k, "refresh_ms": round(ms, 3), "docsRead": read, "phases": phases,
                       "cold_ms": round(cold_ms, 3), "cold_docsRead": cold_read, "cold_phases": cold_phases, "card": name, "power_limit": power}
                out.write(json.dumps(rec) + "\n")
                out.flush()
                print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
