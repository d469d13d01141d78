#!/usr/bin/env python
"""Variant sweep of the config-5 scan kernel (Zipf string keys, direct-indexed HBM table behind the front cache):
the table is generated once on the device, then the query is compiled under each set of N1GPU_* knobs (they are
read at compile time), timed, and every variant's groups are checked against torch reductions over the same tensors.

Usage: ROWS=200000000 python tools/sweep_config5.py            (one JSON line per variant)"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import full_size as fs  # noqa: E402
import workloads as wl  # noqa: E402
import query_b200 as q  # noqa: E402

# the knobs of the cached scan that the library reads; a variant naming anything else is refused, since the library
# would ignore it and the default kernel would be timed under the variant's name
KNOBS = ["N1GPU_NO_PACK", "N1GPU_CACHE_BLOCK", "N1GPU_MIN_BLOCKS", "N1GPU_CACHE_KB", "N1GPU_NO_CACHE", "N1GPU_NO_KEY32",
         "N1GPU_NO_COMPLEMENT", "N1GPU_NO_WIDE1", "N1GPU_NO_SIGN_FROM_MINMAX", "N1GPU_NO_MM_PAIR"]

VARIANTS = [
    ("default", {}),
    ("default, 4 blocks x 256", {"N1GPU_MIN_BLOCKS": "4"}),
    ("default, 2 blocks x 512", {"N1GPU_CACHE_BLOCK": "512"}),
    ("default, 1 block x 1024", {"N1GPU_CACHE_BLOCK": "1024"}),
    ("default, 6 blocks x 192", {"N1GPU_CACHE_BLOCK": "192", "N1GPU_MIN_BLOCKS": "6"}),
]


def main():
    if os.environ.get("EXTRA"):  # ad-hoc variants: EXTRA='[["name", {"N1GPU_...": "..."}], ...]' replaces the list
        VARIANTS[:] = [(n_, e_) for n_, e_ in json.loads(os.environ["EXTRA"])]
    for name, env in VARIANTS:
        unknown = sorted(set(env) - set(KNOBS))
        if unknown:
            sys.exit("variant %r sets %s: not a knob the library reads (%s)" % (name, ", ".join(unknown), ", ".join(KNOBS)))
    q.init(0)
    n = int(os.environ.get("ROWS", "200000000"))
    w = wl.Config5(rows=n)
    t = w.sealed_table()
    ref = w.reference()
    only = os.environ.get("ONLY")
    for name, env in VARIANTS:
        if only and only not in name:
            continue
        for k in KNOBS:
            os.environ.pop(k, None)
        os.environ.update(env)
        qq = w.query(t)
        res, scan_ns, wall, ng = fs.timed(qq, reps=5)
        w.check(res, ref)
        info = qq.info
        gbs = info["scan_bytes_per_row"] * n / scan_ns
        print(json.dumps({"variant": name, "knobs": env, "rows": n, "words": info["words"], "registers": info["registers"], "grid": info["grid"],
                          "block": info["block"], "scan_us": round(scan_ns / 1e3, 1), "rows_per_s": n / (scan_ns * 1e-9), "gb_per_s": round(gbs, 1),
                          "roofline_frac": round(gbs / fs.PEAK, 3), "groups": ng, "check": "every group exact vs torch"}))
        sys.stdout.flush()
        del qq, res


if __name__ == "__main__":
    main()
