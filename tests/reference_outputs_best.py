"""What the unmodified reference encoder computed at BEST_QUALITY for tests/test_gpu_encoder_best_quality.py
(oracle/_ref/ref_encode_best, ref_reencode_best), kept in tests/golden/reference_outputs_best.json so that those tests
run where the reference is not built.  Keys and digests are reference_outputs.py's; the file is a store of its own.

To add or refresh entries, run the tests where oracle/_ref is built with VP8GPU_RECORD_REFERENCE_BEST=<file>: every call
appends its key and digests to <file> (JSON lines), and `python tests/reference_outputs_best.py merge <file>...` folds
them into the golden file (new keys only)."""
import json
import os
import sys

import reference_outputs as R

GOLDEN = os.path.join(R.ROOT, "tests", "golden", "reference_outputs_best.json")
_store = None


def stored(k):
    """the reference's output digests for key `k`; fails when they were never recorded"""
    global _store
    if _store is None:
        _store = json.load(open(GOLDEN)) if os.path.exists(GOLDEN) else {}
    assert k in _store, "no stored reference output for these inputs (key %s): record it where oracle/_ref is built" % k
    return _store[k]


def check(k, outputs):
    """`outputs` of a reference tool run for key `k`: recorded when asked to, else compared with the stored digests"""
    got = R.digests(outputs)
    rec = os.environ.get("VP8GPU_RECORD_REFERENCE_BEST")
    if rec:
        with open(rec, "a") as f:
            f.write(json.dumps({"key": k, "out": got}) + "\n")
    else:
        assert got == stored(k), "the reference tool's output differs from the digests stored in %s" % GOLDEN
    return outputs


def expected(k, run):
    """digests of the reference's outputs for key `k`: from the tool (`run()`) where it is built, else the stored ones"""
    return R.digests(check(k, run())) if run is not None else stored(k)


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
