"""Outputs of the unmodified reference implementation (GenomeWorks' cudapoa and cudaaligner kernels, 3rdparty/spoa) on the inputs
the tests generate, stored in tests/golden/reference_outputs.json.gz so that the tests compare this engine against the reference
without its sources or the libraries built from them (oracle/_ref/).

The functions take the arguments of their namesakes in ref_lib.py. Each stored result is keyed by a digest of the call: function,
arguments and input arrays, leaving out those that only size the reference's batches (memory, threads). A test whose inputs change
finds no entry and fails instead of comparing against the output of other inputs. Per-window outputs of the GPU reference are
stored as digests (digest() below); spoa's consensus strings and MSA rows are stored in full.

To record them again, where oracle/_ref/ is built and a GPU is present:
    GWB200_RECORD_REFERENCE=/tmp/ref.jsonl python -m pytest tests
    python tests/reference_outputs.py /tmp/ref.jsonl
"""
import gzip
import hashlib
import json
import os
import sys

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.json.gz")
RECORD_ENV = "GWB200_RECORD_REFERENCE"
_RESOURCE_ARGS = {"mem_fraction", "max_windows_per_batch", "max_device_memory", "n_threads"}
_table = None


def digest(x):
    """64-bit prefix of SHA-256 over one window's output: a string, a list of strings (MSA rows) or a sequence of integers."""
    h = hashlib.sha256()
    if isinstance(x, str):
        h.update(b"s" + x.encode())
    elif isinstance(x, (list, tuple)) and len(x) and all(isinstance(r, str) for r in x):
        h.update(b"r" + "\n".join(x).encode())
    else:
        h.update(b"i" + np.asarray(x, dtype=np.int64).tobytes())
    return h.hexdigest()[:16]


def _key(fn, args, kwargs):
    h = hashlib.sha256(fn.encode())
    for name, a in [("", a) for a in args] + sorted((k, v) for k, v in kwargs.items() if k not in _RESOURCE_ARGS):
        h.update(("|" + name + "=").encode())
        if isinstance(a, np.ndarray):
            a = np.ascontiguousarray(a)
            h.update(("%s%s" % (a.dtype.str, a.shape)).encode() + a.tobytes())
        elif isinstance(a, (list, tuple)):
            h.update(json.dumps(list(a)).encode())
        else:
            h.update(repr(a).encode())
    return h.hexdigest()[:32]


def _ints(a):
    return [int(x) for x in a]


def _stored_form(fn, r):
    if fn == "ref_poa_run":
        out = {"status": _ints(r["status"]), "consensus": [digest(c) for c in r["consensus"]],
               "coverage": [digest(c) for c in r["coverage"]]}
        if "msa" in r:
            out["msa"] = [digest(rows) for rows in r["msa"]]
        return out
    if fn in ("ref_aligner_run", "ref_global_aligner_run"):
        return {"status": _ints(r["status"]), "is_optimal": _ints(r["is_optimal"]), "edit_distance": _ints(r["edit_distance"]),
                "cigar_basic": [digest(c) for c in r["cigar_basic"]], "cigar_extended": [digest(c) for c in r["cigar_extended"]]}
    if fn == "spoa_consensus":
        return {"consensus": r["consensus"], "cells": r["cells"]}
    if fn == "spoa_msa":
        return r
    raise ValueError(fn)


def _lookup(fn, *args, **kwargs):
    key = _key(fn, args, kwargs)
    rec = os.environ.get(RECORD_ENV)
    if rec:
        import ref_lib
        out = _stored_form(fn, getattr(ref_lib, fn)(*args, **kwargs))
        with open(rec, "a") as f:
            f.write(json.dumps({"key": key, "fn": fn, "result": out}) + "\n")
        return out
    global _table
    if _table is None:
        with gzip.open(GOLDEN, "rt") as f:
            _table = json.load(f)
    if key not in _table:
        raise AssertionError("%s: no stored reference output for these inputs (key %s); record it as %s describes"
                             % (fn, key, os.path.relpath(__file__)))
    return _table[key]["result"]


def ref_poa_run(*args, **kwargs):
    """ref_lib.ref_poa_run: status per window; consensus, coverage and (msa=True) MSA rows as per-window digests."""
    return _lookup("ref_poa_run", *args, **kwargs)


def ref_aligner_run(*args, **kwargs):
    """ref_lib.ref_aligner_run: status, is_optimal, edit_distance per pair; CIGARs as per-pair digests."""
    return _lookup("ref_aligner_run", *args, **kwargs)


def ref_global_aligner_run(*args, **kwargs):
    """ref_lib.ref_global_aligner_run: as ref_aligner_run."""
    return _lookup("ref_global_aligner_run", *args, **kwargs)


def spoa_consensus(*args, **kwargs):
    """ref_lib.spoa_consensus: consensus strings and DP cell count."""
    return _lookup("spoa_consensus", *args, **kwargs)


def spoa_msa(*args, **kwargs):
    """ref_lib.spoa_msa: the MSA rows."""
    return _lookup("spoa_msa", *args, **kwargs)


def merge(record_paths):
    """Adds the recorded entries to the stored table (a key recorded twice must have the same result)."""
    table = {}
    if os.path.exists(GOLDEN):
        with gzip.open(GOLDEN, "rt") as f:
            table = json.load(f)
    for p in record_paths:
        with open(p) as f:
            for line in f:
                e = json.loads(line)
                new = {"fn": e["fn"], "result": e["result"]}
                old = table.get(e["key"])
                if old is not None and old["fn"] == new["fn"] and old["result"] != new["result"]:
                    raise SystemExit("%s: recorded twice with different results" % e["key"])
                table[e["key"]] = new
    with open(GOLDEN, "wb") as raw, gzip.GzipFile(fileobj=raw, mode="wb", mtime=0) as f:
        f.write(json.dumps(table, sort_keys=True, separators=(",", ":")).encode())
    print("%d entries -> %s (%d bytes)" % (len(table), GOLDEN, os.path.getsize(GOLDEN)))


if __name__ == "__main__":
    merge(sys.argv[1:])
