"""The per-document fingerprints the operator keeps with a resident directory keyspace (execution.cpp): which builds read
documents ("#docsRead") and which reuse the table.  Without a device every change is a load from scratch."""
import os
import time

import query_b200 as q
from gen_n1 import F, make_docs
from plans_n1 import explain_plan
from util_n1 import write_keyspace


def docs_read(plan, root):
    return q.Operator(plan, root).marshal_json().get("#stats", {}).get("#docsRead")


def test_docs_read_on_load_reuse_and_touch(tmp_path):
    root = str(tmp_path)
    d = write_keyspace(root, "default", "d", [("k%03d" % i, t) for i, t in enumerate(make_docs(40, seed=5))])
    open(os.path.join(d, "k003.txt"), "w").write("a second row of k003.json")
    time.sleep(0.06)  # past the racily-clean margin: the fingerprints of this load hold
    plan = explain_plan("default", "d", "d", None, [F("t")], ["count(*)", "sum(%s)" % F("p")])
    assert docs_read(plan, root) == 41
    assert docs_read(plan, root) is None  # reused
    os.utime(d, None)
    assert docs_read(plan, root) is None  # a touched directory: the same rows under a new tag
    open(os.path.join(d, "k007.json"), "w").write('{"t": "x"}')
    time.sleep(0.06)
    n = docs_read(plan, root)
    assert n == (1 if q_has_device() else 41)
    assert docs_read(plan, root) is None


def test_racy_document_is_read_again(tmp_path):
    root = str(tmp_path)
    write_keyspace(root, "default", "d", [("k%03d" % i, '{"t": "t%d"}' % (i % 3)) for i in range(10)])
    plan = explain_plan("default", "d", "d", None, [F("t")], ["count(*)"])
    assert docs_read(plan, root) == 10  # every file written just now: racily clean
    time.sleep(0.06)
    assert docs_read(plan, root) == 10  # read again, with or without a device
    assert docs_read(plan, root) is None


def q_has_device():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False
