"""Thin Python handles over the C ABI (include/n1gpu.h).  Everything that computes is in libn1gpu.so."""
from __future__ import annotations

import ctypes as C
import json
import struct

import numpy as np

from . import _lib
from ._lib import C_FALSE, C_FLOAT, C_INT, C_MISSING, C_NULL, C_STRING, C_TRUE, check, lib

PATH_SEP = "\x1f"


class Missing:
    """N1QL MISSING as a Python value (distinct from None == NULL)."""
    _inst = None

    def __new__(cls):
        if cls._inst is None:
            cls._inst = super().__new__(cls)
        return cls._inst

    def __repr__(self):
        return "MISSING"

    def __bool__(self):
        return False


MISSING = Missing()


def _path(p):
    if isinstance(p, (list, tuple)):
        return PATH_SEP.join(p)
    return p.replace(".", PATH_SEP) if PATH_SEP not in p else p


def init(device=-1):
    check(lib().n1gpu_init(int(device)))


def launch_count():
    return int(lib().n1gpu_launch_count())


def jit_stats():
    """(kernels compiled by NVRTC, requests served from the in-process kernel caches) since load"""
    c, r = C.c_uint64(), C.c_uint64()
    check(lib().n1gpu_jit_stats(C.byref(c), C.byref(r)))
    return int(c.value), int(r.value)


def set_segment_dir(path):
    """Directory in which plan-level operators keep persistent columnar segments ("" = none)."""
    check(lib().n1gpu_set_segment_dir(path.encode("utf-8") if path else None))


class Table:
    """A shredded keyspace resident in HBM (n1gpu_table)."""

    def __init__(self, columns=()):
        self._h = C.c_void_p()
        check(lib().n1gpu_table_create(C.byref(self._h)))
        self.columns = []
        for c in columns:
            self.add_column(c)
        self._keep = []

    def add_column(self, path):
        p = _path(path)
        idx = check(lib().n1gpu_table_add_column(self._h, p.encode("utf-8")))
        if p not in self.columns:
            self.columns.append(p)
        return idx

    def find_column(self, path):
        return lib().n1gpu_table_find_column(self._h, _path(path).encode("utf-8"))

    def append_json(self, docs, threads=0):
        """docs: iterable of JSON texts (str/bytes) in primary-key order, or (buffer, offsets)."""
        if isinstance(docs, tuple):
            buf, offsets = docs
            offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        else:
            parts = [d.encode("utf-8") if isinstance(d, str) else bytes(d) for d in docs]
            offsets = np.zeros(len(parts) + 1, dtype=np.int64)
            if parts:
                np.cumsum([len(p) for p in parts], out=offsets[1:])
            buf = b"".join(parts)
        if isinstance(buf, np.ndarray):
            bufp = buf.ctypes.data_as(C.c_char_p)
        else:
            bufp = C.c_char_p(buf)
        check(lib().n1gpu_table_append_json(self._h, bufp, offsets.ctypes.data_as(_lib._I64P), len(offsets) - 1, threads))
        return self

    def load_dir(self, path, threads=0):
        check(lib().n1gpu_table_load_dir(self._h, path.encode("utf-8"), threads))
        return self

    def set_column(self, col, payload, tags=None, dictionary=None):
        """Pre-shredded column: payload int64/float64 (width 8) or uint32 ranks (width 4); tags uint8 or None."""
        idx = col if isinstance(col, int) else self.find_column(col)
        a = np.ascontiguousarray(payload)
        if a.dtype == np.float64 or a.dtype == np.int64 or a.dtype == np.uint64:
            width = 8
        elif a.dtype == np.uint32 or a.dtype == np.int32:
            width = 4
        else:
            raise TypeError("payload dtype %s" % a.dtype)
        t = None
        if tags is not None:
            t = np.ascontiguousarray(tags, dtype=np.uint8)
        blob, offs, nd = None, None, 0
        if dictionary is not None:
            enc = [s.encode("utf-8") if isinstance(s, str) else s for s in dictionary]
            offs = np.zeros(len(enc) + 1, dtype=np.int64)
            if enc:
                np.cumsum([len(e) for e in enc], out=offs[1:])
            blob = b"".join(enc)
            nd = len(enc)
        check(lib().n1gpu_table_set_column(
            self._h, idx, width, a.ctypes.data_as(C.c_void_p), t.ctypes.data_as(C.c_void_p) if t is not None else None,
            a.shape[0], blob, offs.ctypes.data_as(_lib._I64P) if offs is not None else None, nd))
        return self

    def set_column_device(self, col, payload, tags=None, dictionary=None):
        """Pre-shredded column held in device memory: payload / tags are CUDA tensors (torch) of dtype int64 / float64
        (width 8) or int32 (width 4: string ranks) and uint8; copied device-to-device, no host staging."""
        idx = col if isinstance(col, int) else self.find_column(col)
        if not payload.is_cuda or not payload.is_contiguous():
            raise TypeError("payload must be a contiguous CUDA tensor")
        width = {8: 8, 4: 4}.get(payload.element_size())
        if width is None:
            raise TypeError("payload dtype %s" % payload.dtype)
        if tags is not None and (not tags.is_cuda or not tags.is_contiguous() or tags.element_size() != 1):
            raise TypeError("tags must be a contiguous CUDA uint8 tensor")
        blob, offs, nd = None, None, 0
        if dictionary is not None:
            enc = [s.encode("utf-8") if isinstance(s, str) else s for s in dictionary]
            offs = np.zeros(len(enc) + 1, dtype=np.int64)
            if enc:
                np.cumsum([len(e) for e in enc], out=offs[1:])
            blob = b"".join(enc)
            nd = len(enc)
        import torch
        torch.cuda.current_stream().synchronize()  # the producer of the tensors has finished
        check(lib().n1gpu_table_set_column_device(
            self._h, idx, width, C.c_void_p(payload.data_ptr()), C.c_void_p(tags.data_ptr()) if tags is not None else None,
            payload.shape[0], blob, offs.ctypes.data_as(_lib._I64P) if offs is not None else None, nd))
        return self

    def peek(self, col):
        """(payload int64[nrows], tags uint8[nrows]) of a staged column (before seal)."""
        idx = col if isinstance(col, int) else self.find_column(col)
        n = self.num_rows
        pay = np.zeros(n, dtype=np.int64)
        tg = np.zeros(n, dtype=np.uint8)
        check(lib().n1gpu_table_column_peek(self._h, idx, pay.ctypes.data_as(_lib._I64P), tg.ctypes.data_as(_lib._U8P), n))
        return pay, tg

    def dictionary(self, col):
        idx = col if isinstance(col, int) else self.find_column(col)
        nd, nb = C.c_int64(), C.c_int64()
        check(lib().n1gpu_table_dict_export(self._h, idx, None, 0, None, 0, C.byref(nd), C.byref(nb)))
        blob = C.create_string_buffer(max(1, nb.value))
        offs = np.zeros(nd.value + 1, dtype=np.int64)
        check(lib().n1gpu_table_dict_export(self._h, idx, blob, nb.value, offs.ctypes.data_as(_lib._I64P), nd.value + 1,
                                            C.byref(nd), C.byref(nb)))
        raw = blob.raw
        return [raw[offs[i]:offs[i + 1]] for i in range(nd.value)]

    def dictionary_raw(self, col):
        """(blob uint8[bytes], offsets int64[n + 1]) of the column's sorted dictionary - no Python object per string"""
        idx = col if isinstance(col, int) else self.find_column(col)
        nd, nb = C.c_int64(), C.c_int64()
        check(lib().n1gpu_table_dict_export(self._h, idx, None, 0, None, 0, C.byref(nd), C.byref(nb)))
        blob = np.zeros(max(1, nb.value), dtype=np.uint8)
        offs = np.zeros(nd.value + 1, dtype=np.int64)
        check(lib().n1gpu_table_dict_export(self._h, idx, blob.ctypes.data_as(C.c_char_p), nb.value, offs.ctypes.data_as(_lib._I64P), nd.value + 1,
                                            C.byref(nd), C.byref(nb)))
        return blob[: nb.value], offs

    def merge_dictionaries(self, col, parts):
        """parts: [(blob uint8 array, offsets int64 array)] - sorted dictionaries (every rank's export): merged natively with
        the column's own into the global sorted dictionary, ranks remapped (on the device when the column lives there)."""
        idx = col if isinstance(col, int) else self.find_column(col)
        n = len(parts)
        blobs = [np.ascontiguousarray(b, dtype=np.uint8) for b, _o in parts]
        offs = [np.ascontiguousarray(o, dtype=np.int64) for _b, o in parts]
        bp = (C.c_char_p * n)(*[C.cast(b.ctypes.data_as(C.c_void_p), C.c_char_p) if b.size else C.c_char_p(b"") for b in blobs])
        op = (_lib._I64P * n)(*[o.ctypes.data_as(_lib._I64P) for o in offs])
        nd = np.array([len(o) - 1 for o in offs], dtype=np.int64)
        check(lib().n1gpu_table_dict_merge(self._h, idx, n, bp, op, nd.ctypes.data_as(_lib._I64P)))

    def import_dictionary(self, col, strings):
        idx = col if isinstance(col, int) else self.find_column(col)
        enc = [s.encode("utf-8") if isinstance(s, str) else s for s in strings]
        offs = np.zeros(len(enc) + 1, dtype=np.int64)
        if enc:
            np.cumsum([len(e) for e in enc], out=offs[1:])
        check(lib().n1gpu_table_dict_import(self._h, idx, b"".join(enc), offs.ctypes.data_as(_lib._I64P), len(enc)))

    def stats(self, col):
        idx = col if isinstance(col, int) else self.find_column(col)
        s = np.zeros(8, dtype=np.int64)
        check(lib().n1gpu_table_stats_get(self._h, idx, s.ctypes.data_as(_lib._I64P)))
        return s

    def set_stats(self, col, stats):
        idx = col if isinstance(col, int) else self.find_column(col)
        s = np.ascontiguousarray(stats, dtype=np.int64)
        check(lib().n1gpu_table_stats_set(self._h, idx, s.ctypes.data_as(_lib._I64P)))

    def load_ndjson(self, path, threads=0):
        """One JSON document per line, in primary-key order (threads=-1: device shredder)."""
        check(lib().n1gpu_table_load_ndjson(self._h, path.encode("utf-8"), threads))
        return self

    def set_segment_output(self, path, source_tag=""):
        """seal() also writes the shredded columns to `path` (persistent columnar segment)."""
        check(lib().n1gpu_table_set_segment_output(self._h, path.encode("utf-8"), source_tag.encode("utf-8")))
        return self

    def load_segment(self, path, source_tag=""):
        """True when the segment was written for the same columns under the same tag and is now loaded (then seal())."""
        ok = C.c_int()
        check(lib().n1gpu_table_load_segment(self._h, path.encode("utf-8"), source_tag.encode("utf-8"), C.byref(ok)))
        return bool(ok.value)

    def set_global_rows(self, rows):
        """Rows of the whole keyspace over all partitions whose partial states get merged (include/n1gpu.h)."""
        check(lib().n1gpu_table_set_global_rows(self._h, int(rows)))
        return self

    def seal(self):
        check(lib().n1gpu_table_seal(self._h))
        return self

    @property
    def num_rows(self):
        return int(lib().n1gpu_table_num_rows(self._h))

    def scan_bytes(self, col):
        idx = col if isinstance(col, int) else self.find_column(col)
        return lib().n1gpu_table_column_scan_bytes(self._h, idx)

    def close(self):
        if self._h:
            lib().n1gpu_table_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _bits_to_float(b):
    return struct.unpack("<d", struct.pack("<q", int(b)))[0]


class Result:
    """What FinalGroup sends downstream: per group the key values and the final aggregate values."""

    def __init__(self, handle):
        self._h = handle
        self._fetched = False

    def _fetch(self):
        """Values are copied out of the library on first use (a pipelined caller may never look at most results)."""
        if self._fetched:
            return
        handle = self._h
        L = lib()
        self._num_groups = int(L.n1gpu_result_num_groups(handle))
        self.num_keys = L.n1gpu_result_num_keys(handle)
        self.num_aggregates = L.n1gpu_result_num_aggregates(handle)
        g, k, a = self._num_groups, self.num_keys, self.num_aggregates
        kc = np.zeros(max(1, g * k), dtype=np.uint8)
        kv = np.zeros(max(1, g * k), dtype=np.int64)
        ac = np.zeros(max(1, g * a), dtype=np.uint8)
        av = np.zeros(max(1, g * a), dtype=np.int64)
        check(L.n1gpu_result_fetch(handle, kc.ctypes.data_as(_lib._U8P), kv.ctypes.data_as(_lib._I64P),
                                   ac.ctypes.data_as(_lib._U8P), av.ctypes.data_as(_lib._I64P)))
        self.key_cls, self.key_val = kc[:g * k].reshape(g, k), kv[:g * k].reshape(g, k)
        self.agg_cls, self.agg_val = ac[:g * a].reshape(g, a), av[:g * a].reshape(g, a)
        st = np.zeros(8, dtype=np.int64)
        check(L.n1gpu_result_stats(handle, st.ctypes.data_as(_lib._I64P)))
        self._stats = {"rows": int(st[0]), "groups": int(st[1]), "scan_ns": int(st[2]), "shred_upload_ns": int(st[3]),
                       "scan_bytes": int(st[4]), "launches": int(st[5])}
        self._fetched = True

    @property
    def num_groups(self):
        return int(lib().n1gpu_result_num_groups(self._h))

    @property
    def stats(self):
        self._fetch()
        return self._stats

    def _value(self, cls, val):
        if cls == C_MISSING:
            return MISSING
        if cls == C_NULL:
            return None
        if cls == C_FALSE:
            return False
        if cls == C_TRUE:
            return True
        if cls == C_INT:
            return int(val)
        if cls == C_FLOAT:
            return _bits_to_float(val)
        if cls == C_STRING:
            p, n = C.c_char_p(), C.c_int64()
            check(lib().n1gpu_result_string(self._h, int(val), C.byref(p), C.byref(n)))
            return C.string_at(p, n.value).decode("utf-8", "surrogateescape")
        raise ValueError(cls)

    def arrays(self):
        """(key_cls, key_val, agg_cls, agg_val, strings): the flat result arrays and the string table (utf-8 bytes) that
        string payloads index - what Operator.import_arrays takes.  (Inside the library a string payload may be a
        (dictionary column, rank) reference; here every distinct one gets an index of the returned table.)"""
        self._fetch()
        kc, kv, ac, av = self.key_cls.copy(), self.key_val.copy(), self.agg_cls.copy(), self.agg_val.copy()
        strings, index = [], {}
        for cls, val in ((kc, kv), (ac, av)):
            if not (cls.size and (cls == C_STRING).any()):
                continue
            mask = cls == C_STRING
            uniq, inv = np.unique(val[mask], return_inverse=True)
            remap = np.empty(len(uniq), dtype=np.int64)
            for i, u in enumerate(uniq.tolist()):
                if u not in index:
                    p, n = C.c_char_p(), C.c_int64()
                    check(lib().n1gpu_result_string(self._h, int(u), C.byref(p), C.byref(n)))
                    index[u] = len(strings)
                    strings.append(C.string_at(p, n.value))
                remap[i] = index[u]
            val[mask] = remap[inv]
        return kc, kv, ac, av, strings

    def rows(self):
        """[(keys list, aggregates list)] with python values (int / float / str / bool / None / MISSING)."""
        self._fetch()
        out = []
        for g in range(self._num_groups):
            ks = [self._value(self.key_cls[g, k], self.key_val[g, k]) for k in range(self.num_keys)]
            ag = [self._value(self.agg_cls[g, a], self.agg_val[g, a]) for a in range(self.num_aggregates)]
            out.append((ks, ag))
        return out

    def to_json(self):
        n = C.c_int64()
        check(lib().n1gpu_result_to_json(self._h, None, 0, C.byref(n)))
        buf = C.create_string_buffer(n.value + 1)
        check(lib().n1gpu_result_to_json(self._h, buf, n.value + 1, C.byref(n)))
        return json.loads(buf.value.decode("utf-8"))

    def close(self):
        if self._h:
            lib().n1gpu_result_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


MODES = {0: "ungrouped", 1: "dense-shared-memory", 2: "hbm-hash-64", 3: "hbm-hash-128", 4: "hbm-direct", 5: "hbm-hash-wide"}


class Query:
    """A compiled Filter + InitialGroup/IntermediateGroup/FinalGroup chain (n1gpu_query)."""

    def __init__(self, table, alias, where, group_keys, aggregates, params=None):
        """params: {name or position: python scalar} for the `$name` / `$1` parameters of a prepared statement; a list of
        scalars is accepted as the right operand of IN / NOT IN (`x IN $ids`) and is probed as a device-resident set"""
        self.table = table
        self.aggregates = list(aggregates)
        self.group_keys = list(group_keys)
        self._h = C.c_void_p()
        karr = (C.c_char_p * max(1, len(self.group_keys)))(*[k.encode("utf-8") for k in self.group_keys])
        aarr = (C.c_char_p * max(1, len(self.aggregates)))(*[a.encode("utf-8") for a in self.aggregates])
        if params:
            names = [str(k).encode("utf-8") for k in params]
            values = [json.dumps(v).encode("utf-8") for v in params.values()]
            narr = (C.c_char_p * len(names))(*names)
            varr = (C.c_char_p * len(values))(*values)
            check(lib().n1gpu_query_compile_params(table._h, alias.encode("utf-8"), where.encode("utf-8") if where else None, karr,
                                                   len(self.group_keys), aarr, len(self.aggregates), narr, varr, len(names), C.byref(self._h)))
            return
        check(lib().n1gpu_query_compile(table._h, alias.encode("utf-8"), where.encode("utf-8") if where else None,
                                        karr, len(self.group_keys), aarr, len(self.aggregates), C.byref(self._h)))

    def execute(self):
        r = C.c_void_p()
        check(lib().n1gpu_query_execute(self._h, C.byref(r)))
        return Result(r)

    def launch(self):
        check(lib().n1gpu_query_launch(self._h))

    def collect(self):
        r = C.c_void_p()
        check(lib().n1gpu_query_collect(self._h, C.byref(r)))
        return Result(r)

    def cancel(self):
        check(lib().n1gpu_query_cancel(self._h))

    def rebind(self, table):
        check(lib().n1gpu_query_rebind(self._h, table._h))
        self.table = table

    def set_timing(self, enable):
        check(lib().n1gpu_query_set_timing(self._h, 1 if enable else 0))

    def set_stream(self, cuda_stream):
        """cuda_stream: a cudaStream_t as int (torch.cuda.current_stream().cuda_stream; 0 = the legacy default
        stream), or None for the query's own non-blocking stream."""
        check(lib().n1gpu_query_set_stream(self._h, C.c_void_p(-1 if cuda_stream is None else int(cuda_stream))))

    @property
    def kernel_source(self):
        return lib().n1gpu_query_kernel_source(self._h).decode("utf-8")

    @property
    def part_source(self):
        return lib().n1gpu_query_part_source(self._h).decode("utf-8")

    @property
    def info(self):
        a = np.zeros(8, dtype=np.int64)
        check(lib().n1gpu_query_info(self._h, a.ctypes.data_as(_lib._I64P)))
        return {"mode": MODES[int(a[0])], "words": int(a[1]), "registers": int(a[2]), "grid": int(a[3]), "block": int(a[4]),
                "scan_bytes_per_row": int(a[5]), "static_smem": int(a[6]), "slots": int(a[7])}

    @property
    def last_scan_ns(self):
        return int(lib().n1gpu_query_last_scan_ns(self._h))

    # ---- multi-GPU partial state (device pointers as ints) ----
    def scan_partial(self):
        check(lib().n1gpu_query_scan_partial(self._h))

    def partial_counts(self):
        g, d, w = C.c_int64(), C.c_int64(), C.c_int()
        check(lib().n1gpu_query_partial_counts(self._h, C.byref(g), C.byref(d), C.byref(w)))
        return g.value, d.value, w.value

    def partial_export(self, nranks, dev_records, cap_records, dev_distinct, cap_distinct):
        counts = np.zeros(nranks, dtype=np.int64)
        dcounts = np.zeros(nranks, dtype=np.int64)
        check(lib().n1gpu_query_partial_export(self._h, nranks, C.c_void_p(dev_records), cap_records,
                                               counts.ctypes.data_as(_lib._I64P), C.c_void_p(dev_distinct), cap_distinct,
                                               dcounts.ctypes.data_as(_lib._I64P)))
        return counts, dcounts

    def partial_reset(self):
        check(lib().n1gpu_query_partial_reset(self._h))

    def partial_import(self, dev_records, n, dev_distinct, nd):
        check(lib().n1gpu_query_partial_import(self._h, C.c_void_p(dev_records), n, C.c_void_p(dev_distinct), nd))

    def finalize(self):
        r = C.c_void_p()
        check(lib().n1gpu_query_finalize(self._h, C.byref(r)))
        return Result(r)

    def state_words(self):
        """(device pointer, nwords) of the whole partial state of a small-state chain (ungrouped / dense, no DISTINCT)."""
        p, n = C.c_void_p(), C.c_int64()
        check(lib().n1gpu_query_state_words(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def word_ops(self):
        """combine operation of every accumulator word (0 add u64, 1 add f64, 2 min i64, 3 max i64, 4 min u64, 5 max u64, 6 or)"""
        ops = (C.c_int * 64)()
        n = lib().n1gpu_query_word_ops(self._h, ops, 64)
        return [int(ops[i]) for i in range(n)]

    def merge_words(self, dev_all_words, nranks):
        check(lib().n1gpu_query_merge_words(self._h, C.c_void_p(dev_all_words), nranks))

    def set_mailbox(self, mailbox):
        check(lib().n1gpu_query_set_mailbox(self._h, mailbox._h if mailbox is not None else None))
        self._mailbox = mailbox

    @property
    def peer_mode(self):
        """0: no arena merge, 1: direct-indexed table folded owner-sharded, 2: partitioned DISTINCT aggregation over peers"""
        return check(lib().n1gpu_query_peer_mode(self._h))

    def close(self):
        if self._h:
            lib().n1gpu_query_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Mailbox:
    """Peer mailbox for the fused small-state multi-GPU merge, optionally with an arena for peer-readable direct-indexed
    group tables (owner-sharded, collective-free merge + finalisation): n1gpu_mailbox_*."""

    def __init__(self, nranks, rank, max_words=8192, arena_bytes=0):
        self._h = C.c_void_p()
        self.nranks, self.rank, self.arena_bytes = nranks, rank, int(arena_bytes)
        check(lib().n1gpu_mailbox_create_arena(nranks, rank, max_words, int(arena_bytes), C.byref(self._h)))

    @property
    def base(self):
        return lib().n1gpu_mailbox_base(self._h)

    def set_peer(self, rank, dev_base):
        """in-process wiring: the device base pointer of another rank's mailbox (same process)"""
        check(lib().n1gpu_mailbox_set_peer(self._h, rank, C.c_void_p(dev_base)))

    def ipc_handle(self):
        buf = C.create_string_buffer(64)
        check(lib().n1gpu_mailbox_ipc_handle(self._h, buf))
        return buf.raw

    def open_peers(self, handles):
        """handles: list of nranks 64-byte handles in rank order (the own one is ignored)."""
        blob = b"".join(handles)
        assert len(blob) == 64 * self.nranks
        check(lib().n1gpu_mailbox_open_peers(self._h, blob))

    def close(self):
        if self._h:
            lib().n1gpu_mailbox_free(self._h)
            self._h = C.c_void_p()


class Operator:
    """execution.Operator handle built from the reference's plan JSON (n1gpu_plan_build)."""

    def __init__(self, plan_json, datastore_root, tail=False):
        """tail=True also takes over the eligible operators behind FinalGroup (n1gpu_plan_build_tail)."""
        if not isinstance(plan_json, str):
            plan_json = json.dumps(plan_json)
        self._h = C.c_void_p()
        rest, outer = C.c_int(), C.c_int()
        if tail:
            check(lib().n1gpu_plan_build_tail(plan_json.encode("utf-8"), datastore_root.encode("utf-8"), C.byref(self._h), C.byref(rest), C.byref(outer)))
        else:
            check(lib().n1gpu_plan_build(plan_json.encode("utf-8"), datastore_root.encode("utf-8"), C.byref(self._h), C.byref(rest)))
        self.rest_index = rest.value
        self.outer_rest_index = outer.value

    @property
    def tail_operators(self):
        n = C.c_int64()
        check(lib().n1gpu_operator_tail_operators(self._h, None, 0, C.byref(n)))
        buf = C.create_string_buffer(n.value + 1)
        check(lib().n1gpu_operator_tail_operators(self._h, buf, n.value + 1, C.byref(n)))
        text = buf.value.decode("utf-8")
        return text.split(",") if text else []

    def import_result(self, groups):
        """groups: list of (key values, aggregate values) as Result.rows() yields them (MISSING / None / bool / int /
        float / str; aggregates in the order given to the group operators) -> a Result the tail can run over
        (n1gpu_operator_import_result)."""
        strings, index = [], {}

        def enc(v):
            if v is MISSING:
                return 0, 0
            if v is None:
                return 1, 0
            if v is False:
                return 2, 0
            if v is True:
                return 3, 0
            if isinstance(v, int):
                return 4, v
            if isinstance(v, float):
                return 5, int(np.float64(v).view(np.int64))
            if isinstance(v, str):
                if v not in index:
                    index[v] = len(strings)
                    strings.append(v.encode("utf-8"))
                return 6, index[v]
            raise TypeError("not a scalar value: %r" % (v,))
        n = len(groups)
        nk = len(groups[0][0]) if n else 0
        na = len(groups[0][1]) if n else 0
        kc, kv = np.zeros(n * nk, dtype=np.uint8), np.zeros(n * nk, dtype=np.int64)
        ac, av = np.zeros(n * na, dtype=np.uint8), np.zeros(n * na, dtype=np.int64)
        for g, (ks, ag) in enumerate(groups):
            for k, v in enumerate(ks):
                kc[g * nk + k], kv[g * nk + k] = enc(v)
            for a, v in enumerate(ag):
                ac[g * na + a], av[g * na + a] = enc(v)
        return self.import_arrays(kc, kv, ac, av, strings)

    def import_arrays(self, key_cls, key_val, agg_cls, agg_val, strings):
        """The same from flat arrays in n1gpu_result_fetch layout ([ngroups * nkeys] / [ngroups * naggs], row-major; string
        payloads index `strings`, a list of utf-8 bytes) - what Result.arrays() returns, e.g. gathered from several ranks."""
        kc = np.ascontiguousarray(key_cls, dtype=np.uint8).reshape(-1)
        kv = np.ascontiguousarray(key_val, dtype=np.int64).reshape(-1)
        ac = np.ascontiguousarray(agg_cls, dtype=np.uint8).reshape(-1)
        av = np.ascontiguousarray(agg_val, dtype=np.int64).reshape(-1)
        nk, na = self.num_keys, self.num_aggregates
        n = len(kc) // nk if nk else (len(ac) // na if na else 0)
        if len(kc) != n * nk or len(ac) != n * na or len(kv) != len(kc) or len(av) != len(ac):
            raise ValueError("array sizes do not describe %d groups of %d keys and %d aggregates" % (n, nk, na))
        offs = np.zeros(len(strings) + 1, dtype=np.int64)
        if strings:
            np.cumsum([len(b) for b in strings], out=offs[1:])
        r = C.c_void_p()
        check(lib().n1gpu_operator_import_result(self._h, n, kc.ctypes.data_as(_lib._U8P), kv.ctypes.data_as(_lib._I64P),
                                                 ac.ctypes.data_as(_lib._U8P), av.ctypes.data_as(_lib._I64P), b"".join(strings),
                                                 offs.ctypes.data_as(_lib._I64P), len(strings), C.byref(r)))
        return Result(r)

    @property
    def num_keys(self):
        return int(lib().n1gpu_operator_num_keys(self._h))

    @property
    def num_aggregates(self):
        return int(lib().n1gpu_operator_num_aggregates(self._h))

    def run_tail(self, result):
        """The rows FinalProject sends (HAVING / projection / ORDER BY / OFFSET / LIMIT applied): list of dicts."""
        n, rows = C.c_int64(), C.c_int64()
        check(lib().n1gpu_operator_run_tail(self._h, result._h, None, 0, C.byref(n), C.byref(rows)))
        buf = C.create_string_buffer(n.value + 1)
        check(lib().n1gpu_operator_run_tail(self._h, result._h, buf, n.value + 1, C.byref(n), C.byref(rows)))
        return json.loads(buf.value.decode("utf-8"))

    def run_once(self):
        r = C.c_void_p()
        check(lib().n1gpu_operator_run_once(self._h, C.byref(r)))
        return Result(r)

    def send_stop(self):
        check(lib().n1gpu_operator_send_stop(self._h))

    def marshal_json(self):
        n = C.c_int64()
        check(lib().n1gpu_operator_marshal_json(self._h, None, 0, C.byref(n)))
        buf = C.create_string_buffer(n.value + 1)
        check(lib().n1gpu_operator_marshal_json(self._h, buf, n.value + 1, C.byref(n)))
        return json.loads(buf.value.decode("utf-8"))

    def close(self):
        if self._h:
            lib().n1gpu_operator_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
