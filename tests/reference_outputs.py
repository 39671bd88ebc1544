"""What the unmodified reference computed for the tests' inputs, kept so that the comparisons run where it is not built.

The reference tools (oracle/_ref, compiled from the original project's sources by `make -C oracle ref`) exist only
where those sources do.  Every call a test makes to one of them is keyed by a SHA-1 of the tool, its arguments and
all its input bytes, and tests/golden/reference_outputs.json holds the length and SHA-1 of every output the tool gave
for that key.  Where the tool is built it runs and must still give the stored digests; elsewhere the stored digests
are the reference's answer.

To add or refresh entries, run the tests where oracle/_ref is built with VP8GPU_RECORD_REFERENCE=<file>: every call
appends its key and digests to <file> (JSON lines), and `python tests/reference_outputs.py merge <file>...` folds them
into the golden file."""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_outputs.json")
_store = None


def tool(name):
    """path of the reference tool `name`, or None where it is not built"""
    p = os.path.join(REF_DIR, name)
    return p if os.path.exists(p) else None


def digest(b):
    return [len(b), hashlib.sha1(bytes(b)).hexdigest()]


def digests(chunks):
    return [digest(c) for c in chunks]


def key(name, *inputs):
    h = hashlib.sha1(name.encode())
    for x in inputs:
        if isinstance(x, np.ndarray):
            b = repr((x.shape, x.dtype.str)).encode() + np.ascontiguousarray(x).tobytes()
        elif isinstance(x, (bytes, bytearray, memoryview)):
            b = bytes(x)
        elif isinstance(x, (list, tuple)):
            b = key("", *x).encode()
        else:
            b = repr(x).encode()
        h.update(len(b).to_bytes(8, "little"))
        h.update(b)
    return h.hexdigest()


def stored(k):
    """the reference's output digests for key `k`; fails when they were never recorded"""
    global _store
    if _store is None:
        _store = json.load(open(GOLDEN)) if os.path.exists(GOLDEN) else {}
    assert k in _store, "no stored reference output for these inputs (key %s): record it where oracle/_ref is built" % k
    return _store[k]


def check(k, outputs):
    """`outputs` of a reference tool run for key `k`: recorded when asked to, compared with the stored digests when
    there are any; returns `outputs`"""
    got = digests(outputs)
    rec = os.environ.get("VP8GPU_RECORD_REFERENCE")
    if rec:
        with open(rec, "a") as f:
            f.write(json.dumps({"key": k, "out": got}) + "\n")
    else:
        assert got == stored(k), "the reference tool's output differs from the digests stored in %s" % GOLDEN
    return outputs


def expected(k, run):
    """digests of the reference's outputs for key `k`: from the tool (`run()` returns its outputs) where it is built,
    else the stored ones"""
    return digests(check(k, run())) if run is not None else stored(k)


def merge(paths):
    store = json.load(open(GOLDEN)) if os.path.exists(GOLDEN) else {}
    for p in paths:
        for line in open(p):
            r = json.loads(line)
            assert store.setdefault(r["key"], r["out"]) == r["out"], "the reference gave two answers for key %s" % r["key"]
    with open(GOLDEN, "w") as f:
        json.dump(store, f, indent=0, sort_keys=True)
        f.write("\n")


if __name__ == "__main__" and sys.argv[1:2] == ["merge"]:
    merge(sys.argv[2:])
