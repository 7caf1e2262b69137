"""What the reference's own HOST build computed in the parity tests, stored so that they compare against the original
without it: tests/golden/reference/<test module>.json holds, per test id, the fingerprints of the reference's results in
the order the test asked for them.

A fingerprint keeps scalars as they are and replaces arrays and byte strings by a SHA-256 digest of their bytes, so that
comparing fingerprints is comparing the bytes.  A QueryResult keeps its group count and digests of its rows and measures
in output order, ordered by row and ordered by the 32-bit group hash (see assert_same_result).

Re-recording needs the reference's HOST build in oracle/_ref (ARESDB_REFERENCE=<reference tree> bash oracle/build_ref.sh):
    ARESDB_RECORD_REFERENCE=1 python -m pytest -m "not gpu" tests
replaces the stored results of the tests that run and keeps those of the others.  A test module that uses expected()
imports the autouse fixture reference_results, which restarts a test's count of results at every run of it.
"""
from __future__ import annotations

import atexit
import hashlib
import json
import os
from pathlib import Path

import numpy as np
import pytest

STORE = Path(__file__).resolve().parent / "golden" / "reference"
RECORD = os.environ.get("ARESDB_RECORD_REFERENCE") == "1"

_stores: dict = {}
_cursor: dict = {}
_recorded: set = set()


@pytest.fixture(autouse=True)
def reference_results():
    """Every run of a test asks for its stored results from the first one on (reruns and repeats included)."""
    _cursor.clear()
    yield


def _digest(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()[:32]


def _float_key(m: np.ndarray) -> bytes:
    """Measure bytes with -0.0 folded into +0.0 (a dict of python floats does not tell them apart)."""
    return (m + 0).tobytes() if m.dtype.kind == "f" else m.tobytes()


def fingerprint(x):
    from aresdb_b200.query import QueryResult
    if isinstance(x, QueryResult):
        import hashes
        rows = x.packed_rows()
        by_row = np.lexsort(rows.T[::-1]) if rows.shape[1] else np.arange(x.groups)
        fp = {"groups": int(x.groups), "rows": _digest(rows.tobytes()), "measures": _digest(x.measures.tobytes()),
              "counts": None if x.counts is None else _digest(x.counts.tobytes()),
              "by_row": _digest(rows[by_row].tobytes() + _float_key(x.measures[by_row])), "by_hash": None}
        if x.groups and rows.shape[1] % 4 == 0:    # rows the hash-reduce mode keys by murmur3-32
            h = hashes.murmur3_32(rows)
            by_hash = np.argsort(h, kind="stable")
            fp["by_hash"] = _digest(h[by_hash].tobytes() + _float_key(x.measures[by_hash]))
        return fp
    if isinstance(x, np.ndarray):
        return "sha256:" + _digest(x.tobytes())
    if isinstance(x, (bytes, bytearray)):
        return "sha256:" + _digest(bytes(x))
    if isinstance(x, np.generic):
        return x.item()
    if isinstance(x, dict):
        if all(isinstance(k, str) for k in x):
            return {k: fingerprint(v) for k, v in x.items()}
        return "sha256:" + _digest(repr(sorted(((k, fingerprint(v)) for k, v in x.items()), key=repr)).encode())
    if isinstance(x, (list, tuple)):
        return [fingerprint(v) for v in x]
    return x


def _test_id() -> tuple[str, str]:
    cur = os.environ["PYTEST_CURRENT_TEST"].rsplit(" ", 1)[0]       # tests/test_x.py::test_name[params]
    path, name = cur.split("::", 1)
    return Path(path).stem, name


def _store(module: str) -> dict:
    if module not in _stores:
        f = STORE / f"{module}.json"
        _stores[module] = json.loads(f.read_text()) if f.exists() else {}
    return _stores[module]


def _compact(fp) -> str:
    return "fp:" + _digest(json.dumps(fp, sort_keys=True).encode())[:16]


def expected(compute, compact=False):
    """The fingerprint of compute(<the reference's HOST build backend>): computed and stored when recording, else the
    stored one (the n-th call of a test gets the n-th result it stored).  compact: only a digest of the fingerprint is
    stored (for tests that compare thousands of small results and need nothing but equality)."""
    module, name = _test_id()
    store = _store(module)
    n = _cursor[(module, name)] = _cursor.get((module, name), -1) + 1
    if RECORD:
        import harness
        fp = json.loads(json.dumps(fingerprint(compute(harness.get_backend("ref")))))
        if compact:
            fp = _compact(fp)
        if n == 0:
            store[name] = []
        store[name][n:] = [fp]
        _recorded.add(module)
        return json.loads(json.dumps(fp))
    assert name in store and n < len(store[name]), \
        f"no stored reference result #{n} for {module}::{name}: re-record tests/golden/reference/ (see reference_golden.py)"
    return store[name][n]


def assert_same(got, exp, ctx=""):
    """`got` (a live result) against `exp` (a fingerprint from expected())."""
    fp = json.loads(json.dumps(fingerprint(got)))
    if isinstance(exp, str) and exp.startswith("fp:"):
        fp = _compact(fp)
    if isinstance(fp, dict) and isinstance(exp, dict):
        diff = sorted(k for k in set(fp) | set(exp) if fp.get(k) != exp.get(k))
        assert not diff, f"{ctx}: {diff} differ from the reference's"
    assert fp == exp, f"{ctx}: differs from the reference's"


def assert_same_result(got, exp: dict, ordered=True, ctx=""):
    """A QueryResult against the reference's fingerprint: group count, rows and measures in output order; unordered
    (hash-reduce mode, where which member of a set of 32-bit colliding rows names the group is unspecified): the groups
    as a map row -> measure, or failing that as a map hash -> measure."""
    fp = fingerprint(got)
    assert fp["groups"] == exp["groups"], f"{ctx}: {fp['groups']} groups vs {exp['groups']}"
    if ordered:
        assert fp["rows"] == exp["rows"], f"{ctx}: dimension rows / order differ"
        assert fp["measures"] == exp["measures"], f"{ctx}: measures differ"
    else:
        assert fp["by_row"] == exp["by_row"] or (fp["by_hash"] is not None and fp["by_hash"] == exp["by_hash"]), \
            f"{ctx}: group map differs"
    assert fp["counts"] == exp["counts"], f"{ctx}: counts differ"


@atexit.register
def _save():
    if _recorded:
        STORE.mkdir(parents=True, exist_ok=True)
        for module in _recorded:
            store = _stores[module]
            (STORE / f"{module}.json").write_text(json.dumps(store, indent=0, sort_keys=True) + "\n")
