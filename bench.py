#!/usr/bin/env python
"""bench.py — filter + GROUP BY throughput of the B200-native path (BASELINE.json metric) and of the CPU arm.

  python bench.py --gpus N --steps K --warmup W            our arm (one rank per GPU; torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  the CPU arm: the reference-shaped C restatement of the
                                                            Go chain (oracle/oracle_ref.c; the Go reference itself
                                                            cannot be built in this image), all host cores

Headline workload (config.workload = "config5", the north-star 1 B-row GROUP BY, BASELINE.json configs[4]):
  1 B documents {"k": Zipf(s=1.1) string over a 100 k vocabulary, "v": int64 U[-1e3,1e6)}, 10 % of k and of v MISSING
  and 10 % null;  SELECT k,COUNT(*),COUNT(v),SUM(v),MIN(v),MAX(v) FROM d WHERE v IS NOT MISSING GROUP BY k
  STRONG scaling: the same 1 B-row keyspace is range-partitioned over the N ranks (tools/workloads.py generates the
  shredded columns on the device, chunk-seeded, so the data does not depend on N).
A step = one pass of the whole chain over the whole keyspace: every rank's scan of its row range, the
Intermediate -> Final merge across ranks, and the finalisation of all groups into host result arrays.
  value : rows/s, columns resident in HBM (14 GB / N per GPU, far beyond the 126 MB L2), K steps between two CUDA
          events on the launching stream, max over ranks; the merged result is checked in the run at every N against
          torch reductions over the same data (exact).
  e2e   : the same chain through the public API from HOST buffers every step: raw JSON documents of the same shape in
          pinned host memory -> H2D -> device shredder -> seal -> compile (cached) -> scan -> merge -> result on the host.
  roofline : the scan kernel nq_scan - column bytes it must read / its mean CUDA-event duration over the timed steps,
          against MEASURED_PEAKS.json hbm_gbs.
  configs : the other BASELINE configs at full size (2: 10 M ungrouped, 3: 60 M TPC-H Q1, 4: 200 M rows / 1 M groups with
          COUNT+SUM DISTINCT), sharded over the same ranks, each with scan time, rows/s, roofline fraction and check.
  cpu_baseline : oracle_ref.c (kind "port") on a bounded sample of config-5 documents, all host cores (N = 1 only).
  --dump-outputs DIR : the groups of the last timed config-5 step as DIR/<name>.npy (see dump_arrays); the keyspace is
          seeded, so two builds run with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import collections
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

# the config-5 chain in the reference's serialised form (Stringer text, as plan JSON carries it)
ALIAS = "d"
WHERE = "((`d`.`v`) is not missing)"
KEYS = ["(`d`.`k`)"]
AGGS = ["count(*)", "count((`d`.`v`))", "sum((`d`.`v`))", "min((`d`.`v`))", "max((`d`.`v`))"]
METRIC = "filter+GROUP BY rows/sec (columns resident in HBM)"
UNIT = "rows/s"
ROWS = 1_000_000_000
# identical in both arms (the reference arm states its per-step sample under cpu_baseline.sample)
CONFIG = {"workload": "config5", "rows": ROWS,
          "query": "SELECT k,COUNT(*),COUNT(v),SUM(v),MIN(v),MAX(v) FROM d WHERE v IS NOT MISSING GROUP BY k",
          "documents": "k: Zipf(s=1.1) string over a 100k vocabulary, v: int64 U[-1e3,1e6); 10% MISSING + 10% null on each, independently",
          "groups": 100002, "partitioning": "contiguous row ranges of one keyspace, one per GPU (strong scaling)",
          "step": "scan of every row range + Intermediate->Final merge across ranks + finalisation of all groups to host arrays; "
                  "--inflight steps overlap (the next scan runs while the step before it is merged, finalised and copied out), results collected in order",
          "l2": "inputs larger than L2: 14 GB of columns / N per GPU vs 126 MB"}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                 "--format=csv,noheader,nounits", "-lms", "100"], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            rows = [l.strip().split(", ") for l in open(self.path) if l.strip()]
            sm = sorted(float(r[0]) for r in rows if r[0].replace(".", "").isdigit())
            if sm:
                out["sm_mhz"] = sm[len(sm) // 2]
                out["sm_max_mhz"] = float(rows[0][1])
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            seen = set()
            for r in rows:
                for i, nm in enumerate(names):
                    if len(r) > 3 + i and r[3 + i].strip().lower() == "active":
                        seen.add(nm)
            out["reasons"] = sorted(seen)
            out["samples"] = len(rows)
            os.unlink(self.path)
        except Exception:
            pass
        return out


def gen_docs_parallel(cref, config, seed, first, n, threads=8, newline=True):
    """documents [first, first + n) of a config from the C generator, on several host threads (deterministic per row); every
    document ends with a line end, so the buffer is also a packed NDJSON keyspace file as it stands"""
    import numpy as np
    parts = [None] * threads
    bounds = [first + n * i // threads for i in range(threads + 1)]

    def work(i):
        parts[i] = cref.gen_docs(config, seed, bounds[i], bounds[i + 1] - bounds[i], newline)

    ts = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    total = sum(int(o[-1]) for _b, o in parts)
    buf = np.empty(total + 1, dtype=np.uint8)
    offs = np.empty(n + 1, dtype=np.int64)
    at, row = 0, 0
    for b, o in parts:
        m = len(o) - 1
        buf[at:at + int(o[-1])] = b[: int(o[-1])]
        offs[row:row + m] = o[:-1] + at
        at += int(o[-1])
        row += m
    offs[n] = at
    buf[at] = 0
    return buf, offs


DUMP_NAMES = ["count", "count_v", "sum_v", "min_v", "max_v"]  # file names of AGGS, in order


def dump_arrays(w, res):
    """The groups of a config-5 result, ordered by group id, as float arrays: group_id (0 = MISSING key, 1 = NULL key,
    2 + i = the i-th word of the workload's sorted vocabulary), one array per aggregate (float64, exact while |value| < 2^53,
    NaN for NULL), and agg_class (the N1QL class of every aggregate value: an integer SUM and a float SUM differ)."""
    import numpy as np
    rows = res.rows()
    gid = np.array(w.group_ids(res), dtype=np.float64)
    val = np.array([[np.nan if v is None else float(v) for v in a] for _k, a in rows], dtype=np.float64).reshape(len(rows), len(AGGS))
    cls = res.arrays()[2].astype(np.float32).reshape(len(rows), len(AGGS))
    return gid, val, cls


def write_dump(path, gid, val, cls):
    import numpy as np
    order = np.argsort(gid, kind="stable")
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "group_id.npy"), gid[order])
    for j, name in enumerate(DUMP_NAMES):
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(val[order, j]))
    np.save(os.path.join(path, "agg_class.npy"), cls[order])


def same_value(a, b, tol=1e-12):
    """bit-exact, the int / float class of a value included; float64 sums within the north-star tolerance"""
    if isinstance(a, float) and isinstance(b, float):
        return a == b or abs(a - b) <= tol * max(abs(a), abs(b))
    return type(a) is type(b) and a == b


CONFIG1 = [  # BASELINE.json configs[0] (SURVEY.md 8d.1): the reference's own CPU-runnable case, data/sampledb/dimestore
    ("product", "SELECT color, COUNT(*), SUM(unitPrice), AVG(unitPrice), MIN(unitPrice), MAX(unitPrice) FROM product WHERE unitPrice > 10 GROUP BY color",
     "(10 < (`product`.`unitPrice`))", ["(`product`.`color`)"],
     ["count(*)", "sum((`product`.`unitPrice`))", "avg((`product`.`unitPrice`))", "min((`product`.`unitPrice`))", "max((`product`.`unitPrice`))"]),
    ("review", "SELECT rating, COUNT(*) FROM review WHERE rating > 1 GROUP BY rating", "(1 < (`review`.`rating`))", ["(`review`.`rating`)"], ["count(*)"]),
]


def config1_entry(q, cref, np):
    """Config 1 through the reference-facing operator: the two sampledb statements over the file-datastore layout (one file
    per document; the documents are the fixture tests/golden/keyspaces.json.gz extracted from the reference's data/sampledb),
    timed cold (files read + shredded + kernel compiled or fetched) and warm (resident table), checked against oracle_ref.c.
    A latency figure: 900 / 10 000 documents do not fill a GPU."""
    import gzip
    import shutil
    with gzip.open(os.path.join(ROOT, "tests", "golden", "keyspaces.json.gz"), "rb") as f:
        ks = json.loads(f.read().decode("utf-8"))
    root = tempfile.mkdtemp(prefix="n1gpu_config1_")
    out = {}
    try:
        for name, sql, where, keys, aggs in CONFIG1:
            docs = ks["sampledb/dimestore/" + name]
            d = os.path.join(root, "dimestore", name)
            os.makedirs(d)
            for key, text in docs:
                with open(os.path.join(d, key + ".json"), "w", encoding="utf-8") as f:
                    f.write(text)
            term = {"keyspace": name, "namespace": "dimestore"}
            aggs_sorted = sorted(set(aggs))
            plan = {"#operator": "Sequence", "~children": [{"#operator": "Sequence", "~children": [
                dict({"#operator": "PrimaryScan", "index": "#primary", "using": "default"}, **term), dict({"#operator": "Fetch"}, **term),
                {"#operator": "Parallel", "~child": {"#operator": "Sequence", "~children": [
                    {"#operator": "Filter", "condition": where}, {"#operator": "InitialGroup", "aggregates": aggs_sorted, "group_keys": keys}]}},
                {"#operator": "IntermediateGroup", "aggregates": aggs_sorted, "group_keys": keys},
                {"#operator": "FinalGroup", "aggregates": aggs_sorted, "group_keys": keys},
                {"#operator": "Parallel", "~child": {"#operator": "Sequence", "~children": [
                    {"#operator": "InitialProject", "result_terms": [{"expr": a} for a in aggs_sorted]}, {"#operator": "FinalProject"}]}}]},
                {"#operator": "Stream"}]}

            def once():
                t0 = time.perf_counter()
                r = q.Operator(plan, root).run_once()
                r.num_groups
                return r, (time.perf_counter() - t0) * 1e3

            r, cold_ms = once()
            warm = sorted(once()[1] for _ in range(20))
            enc = [t.encode("utf-8") for _k, t in sorted(docs)]
            offs = np.zeros(len(enc) + 1, dtype=np.int64)
            np.cumsum([len(e) for e in enc], out=offs[1:])
            groups, cpu_s, _p = cref.run(np.frombuffer(b"".join(enc), dtype=np.uint8).copy(), offs, name, where, keys, aggs_sorted, threads=1)
            from oracle import n1ql_oracle as O
            exp = {tuple("\0MISSING" if k is O.MISSING else k for k in kk): a for kk, a in groups}
            got = {tuple("\0MISSING" if k is q.MISSING else k for k in kk): a for kk, a in r.rows()}
            ok = exp.keys() == got.keys() and all(all(same_value(x, y) for x, y in zip(exp[k], got[k])) for k in exp)
            out[name] = {"query": sql, "documents": len(docs), "groups": len(got), "cold_ms": cold_ms, "warm_ms_median": warm[len(warm) // 2],
                         "cpu_port_ms_one_thread": cpu_s * 1e3, "check": "every group equals oracle_ref.c" if ok else "MISMATCH"}
    finally:
        shutil.rmtree(root, ignore_errors=True)
    return out


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import query_b200 as q
    import workloads as wl
    from query_b200 import dist as qd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout (one JSON line only)
        dist.init_process_group("nccl", device_id=dev)
    q.init(local)
    K, W = args.steps, max(args.warmup, 3)
    peak, peak_src = peaks()
    trace = bool(os.environ.get("N1GPU_TRACE"))

    def log(msg):
        if trace and rank == 0:
            sys.stderr.write("[bench] %s\n" % msg)

    def maxrank(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def timed_steps(step, k, streams=()):
        """k steps between two CUDA events on the current stream, barrier + synchronize on both sides; max over ranks (ms).
        `streams`: other streams the steps run on - they start after the first event and the second waits for them."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        cur = torch.cuda.current_stream()
        sync_all()
        ev0.record()
        for s_ in streams:
            s_.wait_event(ev0)
        res = None
        for _ in range(k):
            res = step()
        for s_ in streams:
            e_ = torch.cuda.Event()
            e_.record(s_)
            cur.wait_event(e_)
        ev1.record()
        sync_all()
        return maxrank(ev0.elapsed_time(ev1)), res

    # one peer mailbox + arena per process: small states are merged by peer stores fused into the scan, direct-indexed
    # tables are folded owner-sharded by the finalisation kernel over NVLink; NCCL only moves hash / DISTINCT records
    mailbox = qd.make_mailbox(max_words=8192, arena_bytes=(1536 << 20)) if world > 1 else None

    def make(w):
        """table + compiled chain + distributed wrapper of a workload, on torch's current stream"""
        t = w.sealed_table()
        qq = w.query(t)
        qq.set_stream(torch.cuda.current_stream().cuda_stream)
        qq.set_timing(True)
        return t, qq, qd.DistributedQuery(qq, stream=torch.cuda.current_stream(), mailbox=mailbox)

    def checked(w, dq, res):
        ref = w.reference()
        how = w.check(res, ref)
        if world > 1 and not dq.replicated:
            w.check_partition(res, ref["cnt"] > 0)
            how += "; every group finalised by exactly one of the %d ranks" % world
        elif world > 1:
            how += "; merged result replicated on every rank, each rank checked its copy"
        return how

    # ---- headline: config 5, the whole keyspace over the ranks ----------------------------------------------------------
    t_setup = time.perf_counter()
    w5 = wl.Config5(rows=args.rows, dev=dev)
    assert (w5.alias, w5.where, list(w5.keys), list(w5.aggs)) == (ALIAS, WHERE, KEYS, AGGS)
    t5, q5, dq5 = make(w5)
    info = q5.info
    bytes_per_row = info["scan_bytes_per_row"]
    log("config5 table of %d rows on this rank in %.1f s" % (w5.n, time.perf_counter() - t_setup))

    # Steps are pipelined: --inflight prepared instances of the chain (one compiled kernel, one table; each instance owns its
    # stream, group table and result buffers), a step is launched while the one before it is merged, finalised and copied to
    # the host - results are collected in order.  The scan of a 1024-thread block leaves room on every SM for those small
    # kernels (56 registers per thread), so the GPU never waits for the host or for a peer's flag between scans.
    D = max(1, args.inflight)
    q5s, dq5s, streams5 = [q5], [dq5], []
    for _ in range(D - 1):
        s_ = torch.cuda.Stream()
        with torch.cuda.stream(s_):
            qq_ = w5.query(t5)
            qq_.set_stream(s_.cuda_stream)
            qq_.set_timing(True)
            q5s.append(qq_)
            dq5s.append(qd.DistributedQuery(qq_, stream=s_, mailbox=mailbox))
        streams5.append(s_)

    def run5(k, scans=None):
        """k steps, at most D in flight, collected in launch order; returns the last result"""
        fly, res = collections.deque(), None

        def collect():
            j = fly.popleft()
            r = dq5s[j].collect()
            r.num_groups  # the groups are finalised and on the host
            if scans is not None:
                scans.append(q5s[j].last_scan_ns)
            return r

        for i in range(k):
            if len(fly) == D:
                res = collect()
            dq5s[i % D].launch()
            fly.append(i % D)
        while fly:
            res = collect()
        return res

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    res = run5(W)
    # soak: keep stepping (untimed, under its own key) so that clocks are ramped and nvidia-smi has samples under load
    soak_steps, t_soak = 0, time.perf_counter()
    while args.soak > 0:
        res = run5(5)
        soak_steps += 5
        done = time.perf_counter() - t_soak >= args.soak
        if world > 1:  # every rank must run the same number of (collective) steps: rank 0 decides
            flag = torch.tensor([1 if done else 0], device=dev)
            dist.broadcast(flag, 0)
            done = bool(flag.item())
        if done:
            break
    launches0 = q.launch_count()
    res = None
    ms, res = timed_steps(lambda: run5(K), 1, streams5)
    launches = q.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    value = w5.rows * K / (ms / 1e3)
    check5 = checked(w5, dq5, res)
    dump = None
    if args.dump_outputs:
        dump = dump_arrays(w5, res)
        if world > 1:  # rank 0 writes every rank's groups (a replicated merge leaves all of them on rank 0)
            parts = [None] * world
            dist.gather_object(dump, parts if rank == 0 else None, dst=0)
            if rank == 0 and not dq5.replicated:
                import numpy as np
                dump = tuple(np.concatenate(x) for x in zip(*parts))
    # the kernel's own duration (roofline) and the latency of one step: K more steps, one at a time, CUDA events around every
    # nq_scan launch on its stream (with two steps in flight an event pair would also time the wait for the SMs)
    scan_ns = []
    res = None
    D_saved, D = D, 1
    ms_seq, res = timed_steps(lambda: run5(K, scan_ns), 1, streams5)
    D = D_saved
    mean_scan_ns = maxrank(sum(scan_ns) / len(scan_ns))
    merge5 = dq5.describe()
    groups5 = res.num_groups
    if world > 1:
        g = torch.tensor([0 if dq5.replicated and rank else groups5], device=dev)
        dist.all_reduce(g)
        groups5 = int(g.item())
    log("config5: %.3f ms/step, scan %.3f ms" % (ms / K, mean_scan_ns / 1e6))

    # ---- the other configs at full size, sharded over the same ranks ----------------------------------------------------------
    configs = {"config5": {"rows": w5.rows, "rows_per_gpu": w5.n, "mode": info["mode"], "scan_us": mean_scan_ns / 1e3, "step_ms": ms / K,
                           "rows_per_s": value, "scan_bytes_per_row": bytes_per_row,
                           "roofline_frac": bytes_per_row * w5.n / mean_scan_ns / peak, "groups": groups5, "check": check5}}
    del dq5, q5, t5, res, dq5s, q5s
    torch.cuda.empty_cache()
    for name in [c for c in args.configs.split(",") if c and c != "config1"]:  # (config 1 runs through the operator, below)
        t0 = time.perf_counter()
        w = wl.CONFIGS[name](dev=dev, scale=args.configs_scale)
        t, qq, dq = make(w)
        r = dq.execute()
        r.num_groups
        sns = []

        def step():
            rr = dq.execute()
            rr.num_groups
            sns.append(qq.last_scan_ns)
            return rr

        for _ in range(3):  # like the timed loop: the previous step's result is still alive while the next one is built
            r = step()      # (results live in pooled pinned memory; a third live result would mean a fresh cudaHostAlloc)
        sns.clear()
        r = None
        cms, r = timed_steps(step, args.configs_steps)
        cscan = maxrank(sum(sns) / len(sns))
        inf = qq.info
        entry = {"rows": w.rows, "rows_per_gpu": w.n, "mode": inf["mode"], "scan_us": cscan / 1e3, "step_ms": cms / args.configs_steps,
                 "rows_per_s": w.rows * args.configs_steps / (cms / 1e3), "scan_rows_per_s": w.rows / (cscan * 1e-9),
                 "scan_bytes_per_row": inf["scan_bytes_per_row"], "survey_bytes_per_row": w.survey_bytes_per_row,
                 "roofline_frac": inf["scan_bytes_per_row"] * w.n / cscan / peak, "query": w.sql, "check": checked(w, dq, r)}
        # The same launches queued back to back on one stream, elapsed / launches (each = table re-arm + scan kernel(s) of this
        # rank's rows, no merge): a 26 us kernel between two events mostly measures the events, and - measured - a scan that
        # follows an idle gap (one step at a time: the host turns every step around) runs ~10 % slower than one that follows
        # another kernel.
        entry["scan_us_back_to_back"] = maxrank(kernel_back_to_back(q, torch, w, t, 32 if name == "config2" else 6))
        entry["roofline_frac_back_to_back"] = inf["scan_bytes_per_row"] * w.n / (entry["scan_us_back_to_back"] * 1e3) / peak
        groups = r.num_groups
        if world > 1:
            g = torch.tensor([0 if dq.replicated and rank else groups], device=dev)
            dist.all_reduce(g)
            groups = int(g.item())
        entry["groups"] = groups
        configs[name] = entry
        log("%s: %.3f ms/step, scan %.3f ms (%.1f s with setup and check)" % (name, entry["step_ms"], cscan / 1e6, time.perf_counter() - t0))
        del dq, qq, t, r, w
        torch.cuda.empty_cache()

    # ---- end to end from host JSON, config-5 shaped documents ---------------------------------------------------------------------
    from oracle import cref  # document generator + CPU baseline only (never the measured path of this arm)
    e2e_total = args.e2e_rows * world  # --e2e-rows documents per GPU: every rank ingests at its own PCIe rate (weak scaling of the ingest)
    lo, hi = qd.row_range(e2e_total, rank, world)
    buf, offs = gen_docs_parallel(cref, 5, 42, lo, hi - lo)
    pinned = torch.from_numpy(buf).pin_memory()   # the step's inputs live in pinned host memory
    hbuf = pinned.numpy()
    pinned_offs = torch.from_numpy(offs).pin_memory()
    hoffs = pinned_offs.numpy()
    e2e_steps = max(1, min(args.e2e_steps, K))
    phases = []

    def e2e_step():
        ts = [time.perf_counter()]
        t = q.Table(["k", "v"])
        t.append_json((hbuf, hoffs), threads=args.shred_threads)
        ts.append(time.perf_counter())
        if world > 1:
            qd.agree_dictionaries_and_stats(t)
        else:
            t.set_global_rows(t.num_rows)
        t.seal()
        qq = q.Query(t, ALIAS, WHERE, KEYS, AGGS)
        ts.append(time.perf_counter())
        dq = qd.DistributedQuery(qq, mailbox=mailbox if args.e2e_peer else None)
        r = dq.execute()
        ng = r.num_groups
        ts.append(time.perf_counter())
        phases.append([(b - a) * 1e3 for a, b in zip(ts, ts[1:])])
        return r, ng, dq.replicated

    r_e2e, ng_e2e, rep_e2e = e2e_step()  # warm-up (JIT cache, allocator)
    phases.clear()
    sync_all()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        r_e2e, ng_e2e, rep_e2e = e2e_step()
    sync_all()
    e2e_s = maxrank(time.perf_counter() - t0)
    e2e_value = e2e_total * e2e_steps / e2e_s
    h2d = int(hoffs[-1]) + 8 * (len(hoffs))                       # raw JSON + document offsets of this rank
    d2h = ng_e2e * (1 + len(w5.aggs)) * 9                         # class byte + 8-byte payload per key / aggregate value
    ph = [sum(p[i] for p in phases) / len(phases) for i in range(3)]
    if world > 1:
        tt = torch.tensor([float(h2d), float(d2h)] + ph, device=dev, dtype=torch.float64)
        mx = tt.clone()
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        h2d, d2h = int(tt[0].item()), int(tt[1].item())
        ph = [float(x) for x in mx[2:].tolist()]
    # parity of the e2e result against the CPU restatement over the very same documents (rank 0 regenerates all of them)
    mine = [(k[0] if k[0] is not q.MISSING else "\0MISSING", a) for k, a in r_e2e.rows()]
    if world > 1:
        allrows = [None] * world
        dist.gather_object(mine, allrows if rank == 0 else None, dst=0)
        if rank == 0:
            merged = {}
            for i, part in enumerate(allrows):
                if rep_e2e and i:
                    continue  # a replicated merge leaves the complete result on every rank
                for k, a in part:
                    assert k not in merged, "group %r finalised by two ranks" % (k,)
                    merged[k] = a
    else:
        merged = dict(mine)
    parity = None
    cpu = None
    if rank == 0:
        cores = os.cpu_count() or 1
        if world > 1:
            buf_all, offs_all = gen_docs_parallel(cref, 5, 42, 0, e2e_total)
        else:
            buf_all, offs_all = buf, offs
        groups, cpu_s, _passed = cref.run(buf_all, offs_all, ALIAS, WHERE, KEYS, AGGS, threads=cores)
        from oracle import n1ql_oracle as O
        exp = {(k[0] if k[0] is not O.MISSING else "\0MISSING"): a for k, a in groups}
        bad = [k for k in exp if k not in merged or not all(same_value(x, y) for x, y in zip(exp[k], merged[k]))]
        parity = "ok: %d groups of the e2e result equal oracle_ref.c over the same %d documents" % (len(exp), e2e_total) \
            if not bad and len(exp) == len(merged) else "MISMATCH %d groups, e.g. %r: %r vs %r" % (len(bad), bad[:1], [exp[k] for k in bad[:1]], [merged.get(k) for k in bad[:1]])
        if world == 1:
            sample = min(args.cpu_sample, e2e_total)
            sbuf, soffs = (buf_all, offs_all) if sample == e2e_total else gen_docs_parallel(cref, 5, 42, 0, sample)
            if sample != e2e_total:
                groups, cpu_s, _passed = cref.run(sbuf, soffs, ALIAS, WHERE, KEYS, AGGS, threads=cores)
            cpu = {"value": sample / cpu_s, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": "%d config5-shaped JSON documents, oracle/oracle_ref.c (reference-shaped C restatement of the Go chain), %d threads" % (sample, cores)}

    if rank == 0 and "config1" in args.configs.split(","):
        configs["config1"] = config1_entry(q, cref, np)
    # ---- the same end to end through the reference-facing operator (plan JSON + datastore root), one GPU ----------------------------
    e2e_op = None
    if world == 1 and args.e2e_operator:
        import shutil
        root = tempfile.mkdtemp(prefix="n1gpu_bench_")
        try:
            os.makedirs(os.path.join(root, "default"))
            packed = os.path.join(root, "default", "d.ndjson")  # the packed form of the keyspace default:d (one document per line)
            buf[: int(offs[-1])].tofile(packed)
            term = {"keyspace": "d", "namespace": "default"}
            aggs_sorted = sorted(set(AGGS))
            plan = {"#operator": "Sequence", "~children": [{"#operator": "Sequence", "~children": [
                dict({"#operator": "PrimaryScan", "index": "#primary", "using": "default"}, **term), dict({"#operator": "Fetch"}, **term),
                {"#operator": "Parallel", "~child": {"#operator": "Sequence", "~children": [
                    {"#operator": "Filter", "condition": WHERE}, {"#operator": "InitialGroup", "aggregates": aggs_sorted, "group_keys": KEYS}]}},
                {"#operator": "IntermediateGroup", "aggregates": aggs_sorted, "group_keys": KEYS},
                {"#operator": "FinalGroup", "aggregates": aggs_sorted, "group_keys": KEYS},
                {"#operator": "Parallel", "~child": {"#operator": "Sequence", "~children": [
                    {"#operator": "InitialProject", "result_terms": [{"expr": a} for a in aggs_sorted]}, {"#operator": "FinalProject"}]}}]},
                {"#operator": "Stream"}]}

            def op_step():
                os.utime(packed)  # a changed keyspace: the operator's resident table is stale, the documents are read and shredded again
                op = q.Operator(plan, root)
                r = op.run_once()
                return r, r.num_groups

            r_op, ng_op = op_step()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                r_op, ng_op = op_step()
            torch.cuda.synchronize()
            op_s = time.perf_counter() - t0
            order = [aggs_sorted.index(a) for a in AGGS]
            got_op = {(k[0] if k[0] is not q.MISSING else "\0MISSING"): [a[i] for i in order] for k, a in r_op.rows()}
            same = got_op.keys() == merged.keys() and all(all(same_value(x, y) for x, y in zip(got_op[k], merged[k])) for k in merged)
            e2e_op = {"value": e2e_total * e2e_steps / op_s, "unit": UNIT, "steps": e2e_steps, "rows_per_step": e2e_total,
                      "includes": "n1gpu_plan_build on the reference's plan JSON + a packed NDJSON keyspace file read into pinned memory by all cores + "
                                  "chunked H2D overlapped with the device shredder + scan + finalisation (the resident-table cache is invalidated every step)",
                      "same_groups_as_e2e": bool(same)}
        finally:
            shutil.rmtree(root, ignore_errors=True)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel ----------------------------------------------------------------------------------------
    # the kernel's average launch duration: per-launch events in the one-at-a-time pass, or - when smaller - the timed region
    # divided by its launches (one scan per step, and scans cannot overlap each other: one block per SM fills its shared memory),
    # which still contains everything else a step does
    kernel_ns = min(mean_scan_ns, ms / K * 1e6)
    achieved = bytes_per_row * w5.n / kernel_ns  # bytes/ns == GB/s
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        per_row = tj.get("nq_scan_config5_dram_bytes_per_row")
        if per_row:
            traffic = per_row * w5.n
            traffic_src = "static: %s (dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture, per row, scaled to this launch)" % tj.get("nq_scan_config5_source")
    except Exception:
        pass
    merge = "none (one rank)" if world == 1 else merge5
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup, "warmup_run": W, "soak_steps": soak_steps,
        "ms_per_step": ms / K, "steps_in_flight": D, "ms_per_step_one_at_a_time": ms_seq / K,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "int64 (u32 dictionary ranks, u8 classes)", "data": "synthetic", "config": CONFIG,
        "result_check": check5, "groups": groups5,
        "kernel": {"mode": info["mode"], "registers": info["registers"], "grid": info["grid"], "block": info["block"],
                   "scan_bytes_per_row": bytes_per_row, "survey_bytes_per_row": 14, "rows_per_launch": w5.n, "merge": merge},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                "rows_per_step": e2e_total, "rows_per_gpu_per_step": args.e2e_rows, "scaling": "weak (--e2e-rows documents per GPU)",
                "json_bytes_per_step": h2d - 8 * (e2e_total + world),
                "includes": ("H2D of the raw JSON from pinned host memory + device shredder (shred.cu)" if args.shred_threads < 0 else "JSON shredding on host threads + column H2D")
                + " + dictionary / statistics agreement across ranks + seal + compile (cached) + scan + merge + finalisation to host arrays",
                "phase_ms_max_over_ranks": {"shred": ph[0], "agree+seal+compile": ph[1], "scan+merge+finalize": ph[2]},
                "parity_vs_cpu_baseline": parity, "through_operator": e2e_op},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "traffic_source": traffic_src, "kernel": "nq_scan (filter + group key + hash aggregation of config 5)", "peak_source": peak_src,
                     "mean_kernel_us": kernel_ns / 1e3, "mean_kernel_us_one_at_a_time": mean_scan_ns / 1e3,
                     "timed_region_us_per_launch": ms / K * 1e3, "algorithmic_bytes_per_launch": bytes_per_row * w5.n,
                     "timing": "min(CUDA events around every nq_scan launch on its stream, mean over %d steps run one at a time right after the timed region; "
                               "CUDA events around the timed region / its %d launches - one scan per step, scans cannot overlap each other), max over ranks" % (K, K),
                     "accumulator_updates_per_s": None},
        "cpu_baseline": cpu,
        "configs": configs,
    }
    if dump is not None:
        write_dump(args.dump_outputs, *dump)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def kernel_back_to_back(q, torch, w, table, nk):
    """mean duration (us) of nk launches of the scan queued back to back on one stream between two CUDA events"""
    s = torch.cuda.Stream()
    kq = []
    for _ in range(nk):
        qq = w.query(table)
        qq.set_stream(s.cuda_stream)
        qq.set_timing(False)
        kq.append(qq)
    for qq in kq:
        qq.execute()
    ka, kb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = []
    for _ in range(5):
        torch.cuda.synchronize()
        ka.record(s)
        for qq in kq:
            qq.launch()
        kb.record(s)
        for qq in kq:
            qq.collect()
        torch.cuda.synchronize()
        best.append(ka.elapsed_time(kb) * 1e3 / nk)
    return sorted(best)[len(best) // 2]


def run_reference(args):
    """The CPU arm: the reference's own algorithm for the path (document-at-a-time interpreter over raw JSON, string
    group keys, 3-phase merge) restated in C because Go is not in this image; all host threads; each step a bounded
    sample of the same workload (config-5 shaped documents), sized so that the whole run ends within ~90 s."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cref
    cores = os.cpu_count() or 1
    K, W = args.steps, max(1, args.warmup)
    sample = args.cpu_sample
    buf, offs = gen_docs_parallel(cref, 5, 42, 0, sample)
    t0 = time.perf_counter()
    cref.run(buf, offs, ALIAS, WHERE, KEYS, AGGS, threads=cores)
    rate = sample / max(time.perf_counter() - t0, 1e-9)
    fit = int(rate * 90.0 / max(K + W, 1))
    if fit < sample:
        sample = max(50_000, fit)
        buf, offs = gen_docs_parallel(cref, 5, 42, 0, sample)
    for _ in range(W):
        cref.run(buf, offs, ALIAS, WHERE, KEYS, AGGS, threads=cores)
    t0 = time.perf_counter()
    for _ in range(K):
        groups, _s, _p = cref.run(buf, offs, ALIAS, WHERE, KEYS, AGGS, threads=cores)
    el = time.perf_counter() - t0
    value = sample * K / el
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": args.warmup,
        "ms_per_step": el / K * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "int64 (u32 dictionary ranks, u8 classes)", "data": "synthetic", "config": CONFIG,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d config5-shaped JSON documents per step (a bounded sample of the 1 B-document workload), oracle/oracle_ref.c with %d threads "
                                   "(the Go reference is not buildable here)" % (sample, cores)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "groups": len(groups),
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=ROWS, help="documents of the config-5 keyspace (all ranks together)")
    ap.add_argument("--configs", default="config1,config2,config3,config4", help="other BASELINE configs reported in the `configs` block")
    ap.add_argument("--configs-scale", type=float, default=1.0)
    ap.add_argument("--configs-steps", type=int, default=5)
    ap.add_argument("--inflight", type=int, default=3, help="steps of the headline config in flight (prepared instances of the chain on their own streams)")
    ap.add_argument("--e2e-rows", type=int, default=16_000_000, help="config-5 shaped JSON documents per e2e step and GPU")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-sample", type=int, default=16_000_000)
    ap.add_argument("--shred-threads", type=int, default=-1, help="-1: device shredder (shred.cu); >= 0: host threads (0 = all cores)")
    ap.add_argument("--e2e-operator", type=int, default=1, help="0: skip the operator-level e2e figure (N = 1)")
    ap.add_argument("--e2e-peer", type=int, default=1, help="0: the e2e steps merge with NCCL instead of the peer arena")
    ap.add_argument("--soak", type=float, default=1.0, help="seconds of untimed stepping before the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the groups of the last timed config-5 step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of --impl ours")
    # stdout carries exactly ONE JSON line: libraries that print banners to fd 1 (NCCL's version line) are sent to
    # stderr for the duration of the run, and the JSON line goes to the real stdout at the end.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
