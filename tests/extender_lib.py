"""cudaextender test infrastructure (TEST ONLY): ctypes bindings of the CPU oracle (oracle/liboracle_extender.so) and of the
unmodified reference cudaextender (oracle/_ref/libgwref_ext.so), both built by oracle/extender.mk, and the reference's outputs on the
tests' inputs, stored in tests/golden/extender_reference_outputs.json.gz so that the GPU tests compare against the reference kernels
without the reference present.

Stored results are keyed like tests/reference_outputs.py keys its own (digest of function name, arguments and input arrays) and
hold the number of scored segment pairs and a digest of all of them in order. To record them again, where oracle/_ref/ is built
and a GPU is present:
    GWB200_RECORD_EXTENDER_REFERENCE=/tmp/ext.jsonl python -m pytest tests/test_gpu_extender.py
    python tests/extender_lib.py /tmp/ext.jsonl
"""
import ctypes as C
import gzip
import json
import os
import subprocess
import sys

import numpy as np

from reference_outputs import _key, digest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_LIB = os.path.join(ORACLE_DIR, "_ref", "libgwref_ext.so")
GOLDEN = os.path.join(ROOT, "tests", "golden", "extender_reference_outputs.json.gz")
RECORD_ENV = "GWB200_RECORD_EXTENDER_REFERENCE"
_oracle = None
_ref = None
_table = None


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _inputs(query, target, score_mat, seeds):
    return (np.ascontiguousarray(query, dtype=np.int8), np.ascontiguousarray(target, dtype=np.int8),
            np.ascontiguousarray(score_mat, dtype=np.int32).reshape(-1), np.ascontiguousarray(seeds, dtype=np.uint32).reshape(-1, 2))


def _records(out, k):
    rec = out[:k].astype(np.int64)
    rec[:, :2] &= 0xFFFFFFFF
    return rec


def oracle_run(query, target, score_mat, xdrop, no_entropy, score_threshold, seeds):
    """oracle_extender_run: encoded query / target (int8), 64 scores, seeds as (n, 2) rows of {query, target} ->
    (records: (m, 4) int64 array of query, target, length, score; segments kept before deduplication)."""
    global _oracle
    if _oracle is None:
        path = os.path.join(ORACLE_DIR, "liboracle_extender.so")
        src = os.path.join(ORACLE_DIR, "extender_oracle.cpp")
        if not os.path.exists(path) or os.path.getmtime(src) > os.path.getmtime(path):
            subprocess.check_call(["make", "-C", ORACLE_DIR, "-f", "extender.mk", "oracle_ext"], stdout=subprocess.DEVNULL)
        _oracle = C.CDLL(path)
        _oracle.oracle_extender_run.restype = C.c_int64
    q, t, m, s = _inputs(query, target, score_mat, seeds)
    out = np.zeros((max(len(s), 1), 4), dtype=np.int32)
    stats = np.zeros(2, dtype=np.int64)
    k = _oracle.oracle_extender_run(_p(q), C.c_int32(len(q)), _p(t), C.c_int32(len(t)), _p(m), C.c_int32(xdrop),
                                    C.c_int32(1 if no_entropy else 0), C.c_int32(score_threshold), _p(s), C.c_int32(len(s)), _p(out),
                                    _p(stats))
    return _records(out, k), int(stats[0])


def have_reference():
    return os.path.exists(REF_LIB)


def reference_run(query, target, score_mat, xdrop, no_entropy, score_threshold, seeds, device_api=False):
    """The unmodified reference (create_extender + extend_async + sync, host or device pointer API) ->
    dict(records=(m, 4) int64 array, timings=[device ms (device API), host ms of the call, host ms of create_extender])."""
    global _ref
    if _ref is None:
        _ref = C.CDLL(REF_LIB)
    q, t, m, s = _inputs(query, target, score_mat, seeds)
    out = np.zeros((max(len(s), 1), 4), dtype=np.int32)
    n_out = C.c_int32(0)
    timings = np.zeros(3, dtype=np.float64)
    err = C.create_string_buffer(1024)
    rc = _ref.ref_extender_run(_p(q), C.c_int32(len(q)), _p(t), C.c_int32(len(t)), _p(m), C.c_int32(xdrop), C.c_int32(1 if no_entropy else 0),
                               C.c_int32(score_threshold), _p(s), C.c_int32(len(s)), C.c_int32(1 if device_api else 0), _p(out),
                               C.byref(n_out), _p(timings), err, C.c_int32(1024))
    if rc != 0:
        raise RuntimeError("reference cudaextender failed: " + err.value.decode())
    return dict(records=_records(out, n_out.value), timings=timings)


def stored_reference_run(query, target, score_mat, xdrop, no_entropy, score_threshold, seeds, device_api=False):
    """reference_run's output on these inputs as stored: dict(count, records = digest of the records in order)."""
    args = _inputs(query, target, score_mat, seeds)
    args = (args[0], args[1], args[2], xdrop, bool(no_entropy), score_threshold, args[3])
    key = _key("ref_extender_run", args, {"device_api": device_api})
    rec = os.environ.get(RECORD_ENV)
    if rec:
        r = reference_run(*args, device_api=device_api)["records"]
        out = {"count": int(len(r)), "records": digest(r.reshape(-1))}
        with open(rec, "a") as f:
            f.write(json.dumps({"key": key, "fn": "ref_extender_run", "result": out}) + "\n")
        return out
    global _table
    if _table is None:
        with gzip.open(GOLDEN, "rt") as f:
            _table = json.load(f)
    if key not in _table:
        raise AssertionError("ref_extender_run: no stored reference output for these inputs (key %s); record it as %s describes"
                             % (key, os.path.relpath(__file__)))
    return _table[key]["result"]


def merge(record_paths):
    """Adds recorded entries to the stored table; a key recorded twice must have the same result."""
    table = {}
    if os.path.exists(GOLDEN):
        with gzip.open(GOLDEN, "rt") as f:
            table = json.load(f)
    for p in record_paths:
        with open(p) as f:
            for line in f:
                e = json.loads(line)
                new = {"fn": e["fn"], "result": e["result"]}
                if e["key"] in table and table[e["key"]] != new:
                    raise SystemExit("%s: recorded twice with different results" % e["key"])
                table[e["key"]] = new
    with open(GOLDEN, "wb") as raw, gzip.GzipFile(fileobj=raw, mode="wb", mtime=0) as f:
        f.write(json.dumps(table, sort_keys=True, separators=(",", ":")).encode())
    print("%d entries -> %s" % (len(table), GOLDEN))


if __name__ == "__main__":
    merge(sys.argv[1:])
