"""Per-node parity on seeded random inputs.

`impl` is the implementation under test: the C restatement (CPU run — this is what pins the
oracle against the reference build) or the B200 engine (`-m gpu`).  The checker of the C restatement
is what the reference's own HOST build computed on the same inputs (stored, tests/reference_golden.py);
the checker of the B200 engine is the C restatement.  Integer /
byte / index outputs must be bit-exact; float outputs of these element-wise ops too (same
IEEE operations in the same order).
"""
import numpy as np
import pytest

import harness as H
import parity_cases as P
import reference_golden as R
from reference_golden import reference_results  # noqa: F401  (autouse fixture)
from aresdb_b200 import cabi as A


def checker_for(impl):
    """None: the reference's stored results."""
    return None if impl.name == "oracle" else H.get_backend("oracle")


def check(chk, got: dict, run, ctx):
    """`got` against run(chk), or against the reference's stored result of run when chk is None."""
    if chk is None:
        R.assert_same(got, R.expected(run, compact=True), ctx)
    else:
        assert_same(got, run(chk), ctx)


def assert_same(a: dict, b: dict, ctx):
    assert a.keys() == b.keys()
    for k in a:
        if isinstance(a[k], np.ndarray):
            assert a[k].tobytes() == b[k].tobytes(), f"{ctx}: '{k}' differs\n got {a[k][:64]}\n exp {b[k][:64]}"
        else:
            assert a[k] == b[k], f"{ctx}: '{k}' differs: {a[k]} vs {b[k]}"


def _sink_ok(sink, result_class):
    """Avoid float -> integer sinks with negative / fractional surprises only where C leaves the
    conversion undefined (negative float -> unsigned)."""
    dt = sink[1]
    if result_class == "f" and dt in (A.Uint8, A.Uint16, A.Uint32):
        return False
    return True


def _random_sink(rng):
    r = rng.integers(0, 3)
    if r == 0:
        return ("scratch", P.SCRATCH_TYPES[rng.integers(0, 3)])
    if r == 1:
        return ("dim", P.DIM_TYPES[rng.integers(0, len(P.DIM_TYPES))])
    # aggregate family consistent with the element type, as the AQL compiler guarantees
    # (query/aql_compiler.go:1139-1250); mismatched pairs hit undefined float->int identities.
    dt = P.MEASURE_TYPES[rng.integers(0, len(P.MEASURE_TYPES))]
    choices = {A.Int32: [A.AGGR_SUM_SIGNED, A.AGGR_MIN_SIGNED, A.AGGR_MAX_SIGNED],
               A.Uint32: [A.AGGR_SUM_UNSIGNED, A.AGGR_MIN_UNSIGNED, A.AGGR_MAX_UNSIGNED],
               A.Float32: [A.AGGR_SUM_FLOAT, A.AGGR_MIN_FLOAT, A.AGGR_MAX_FLOAT],
               A.Int64: [A.AGGR_SUM_SIGNED, A.AGGR_SUM_UNSIGNED],
               A.Float64: [A.AGGR_SUM_FLOAT, A.AGGR_AVG_FLOAT]}[dt]
    agg = choices[rng.integers(0, len(choices))]
    return ("measure", dt, agg)


def _rle(rng, n_rows):
    """Cumulative counts of a random RLE column covering n_rows rows."""
    cuts = np.sort(rng.choice(np.arange(1, n_rows), size=min(n_rows - 1, max(1, n_rows // 3)), replace=False))
    return np.concatenate([[0], cuts, [n_rows]]).astype(np.uint32)


@pytest.mark.parametrize("seed", range(6))
def test_unary_transform_matrix(impl, seed):
    chk = checker_for(impl)
    rng = np.random.default_rng(1000 + seed)
    for fn in P.UNARY_FNS:
        for trial in range(6):
            n = int(rng.integers(1, 70))
            rle = _rle(rng, n + 5) if n > 2 else None
            spec = P.random_input(rng, n, small=fn in P.DATE_FNS, rle=rle)
            cls = P.input_kind_class(spec)
            sink = _random_sink(rng)
            result_cls = "u" if fn in P.DATE_FNS or fn in (A.Not, A.IsNull, A.IsNotNull, A.GetHLLValue) else cls
            if fn == A.GetHLLValue and cls == "f":
                result_cls = "f"
            if not _sink_ok(sink, result_cls):
                continue
            index = rng.permutation(n).astype(np.uint32) if rng.integers(0, 2) else None
            use_bc = rle is not None and rng.integers(0, 2)
            base_counts = _rle(rng, n + 5)[: n + 1] if False else None
            if use_bc:
                # baseCounts: cumulative row numbers of the batch's first (RLE) column, n runs
                steps = rng.integers(1, 3, n)
                base_counts = np.concatenate([[0], np.cumsum(steps)]).astype(np.uint32)
                if spec.kind == "column" and spec.mode == 3:
                    spec.counts = _rle(rng, int(base_counts[-1]) + 1)
                    runs = len(spec.counts) - 1
                    spec.values = P.random_values(rng, spec.data_type, runs, small=fn in P.DATE_FNS)
                    spec.valid = rng.integers(0, 4, runs) != 0
            kw = dict(index=index, base_counts=base_counts, start_count=int(rng.integers(0, 3)))
            got = P.run_transform(impl, [spec], fn, sink, n, **kw)
            check(chk, got, lambda be: P.run_transform(be, [spec], fn, sink, n, **kw), f"unary fn={fn} sink={sink} in={spec.kind}/{spec.data_type}/mode{spec.mode}")


@pytest.mark.parametrize("seed", range(6))
def test_binary_transform_matrix(impl, seed):
    chk = checker_for(impl)
    rng = np.random.default_rng(2000 + seed)
    for fn in P.BINARY_FNS:
        for trial in range(8):
            n = int(rng.integers(1, 70))
            divides = fn in (A.Divide, A.Mod, A.Floor)
            lhs = P.random_input(rng, n, allow_const=False, small=divides)
            rhs = P.random_input(rng, n, nonzero=divides, small=divides)
            ca, cb = P.input_kind_class(lhs), P.input_kind_class(rhs)
            common = "f" if "f" in (ca, cb) else ("s" if "s" in (ca, cb) else "u")
            if common == "f" and fn in P.INT_ONLY_BIN:
                continue  # "return t1": a pass-through of the float lhs, covered by Noop
            sink = _random_sink(rng)
            result_cls = "u" if fn <= A.GreaterThanOrEqual else common
            if not _sink_ok(sink, result_cls):
                continue
            if fn == A.Minus and common == "u":
                sink = ("scratch", A.Uint32)  # wrapped differences only make sense as raw bits
            index = rng.permutation(n).astype(np.uint32) if rng.integers(0, 2) else None
            got = P.run_transform(impl, [lhs, rhs], fn, sink, n, index=index)
            check(chk, got, lambda be: P.run_transform(be, [lhs, rhs], fn, sink, n, index=index), f"binary fn={fn} sink={sink} lhs={lhs.kind}/{lhs.data_type} rhs={rhs.kind}/{rhs.data_type}")


@pytest.mark.parametrize("seed", range(4))
def test_filter_matrix(impl, seed):
    chk = checker_for(impl)
    rng = np.random.default_rng(3000 + seed)
    sizes = [1, 2, 31, 32, 33, 255, 1024, 1025, 5000, 40000]
    for fn in [A.Equal, A.NotEqual, A.LessThan, A.GreaterThanOrEqual, A.And, A.Or]:
        for n in sizes:
            lhs = P.random_input(rng, n, allow_const=False)
            rhs = P.random_input(rng, n)
            # a previously filtered (sparse, ascending) index vector, as later filters see it
            rows = n + int(rng.integers(0, 50))
            for s in (lhs, rhs):
                if s.kind == "column" and s.mode in (1, 2):
                    s.values = P.random_values(rng, s.data_type, rows)
                    s.valid = rng.integers(0, 4, rows) != 0
            index = np.sort(rng.choice(rows, size=n, replace=False)).astype(np.uint32)
            got = P.run_filter(impl, [lhs, rhs], fn, n, index=index)
            check(chk, got, lambda be: P.run_filter(be, [lhs, rhs], fn, n, index=index), f"filter fn={fn} n={n}")
    for fn in [A.Noop, A.Not, A.IsNull, A.IsNotNull, A.Negate]:
        for n in sizes[:8]:
            spec = P.random_input(rng, n, allow_const=False)
            got = P.run_filter(impl, [spec], fn, n)
            check(chk, got, lambda be: P.run_filter(be, [spec], fn, n), f"unary filter fn={fn} n={n}")


SORT_AGGS = [(A.AGGR_SUM_UNSIGNED, 4), (A.AGGR_SUM_UNSIGNED, 8), (A.AGGR_SUM_SIGNED, 4), (A.AGGR_SUM_SIGNED, 8),
             (A.AGGR_SUM_FLOAT, 4), (A.AGGR_SUM_FLOAT, 8), (A.AGGR_MIN_UNSIGNED, 4), (A.AGGR_MIN_SIGNED, 4),
             (A.AGGR_MIN_FLOAT, 4), (A.AGGR_MAX_UNSIGNED, 4), (A.AGGR_MAX_SIGNED, 4), (A.AGGR_MAX_FLOAT, 4)]


@pytest.mark.parametrize("seed", range(4))
def test_sort_reduce(impl, seed):
    """Sort + Reduce: hashes, the stable order, first-row-of-run dims and measures, bit-exact
    (float measures are multiples of 1/64, so sums are exact in every association order)."""
    chk = checker_for(impl)
    rng = np.random.default_rng(4000 + seed)
    for nd in P.DIM_CONFIGS:
        for n in (1, 7, 64, 1000, 20000):
            agg, vb = SORT_AGGS[rng.integers(0, len(SORT_AGGS))]
            capacity = n + int(rng.integers(0, 9))
            block = P.random_dim_block(rng, nd, capacity, n, cardinality=int(rng.integers(2, 6)))
            meas = P.random_measures(rng, agg, vb, capacity)
            index = rng.permutation(n).astype(np.uint32) if rng.integers(0, 2) else None
            got = P.run_sort_reduce(impl, block, nd, capacity, n, meas, vb, agg, index=index)
            check(chk, got, lambda be: P.run_sort_reduce(be, block, nd, capacity, n, meas, vb, agg, index=index), f"sort_reduce nd={nd} n={n} agg={agg}/{vb}")


@pytest.mark.parametrize("seed", range(3))
def test_hash_reduce(impl, seed):
    """HashReduce: compared as a map dim-row -> measure (output order is unspecified)."""
    chk = checker_for(impl)
    rng = np.random.default_rng(5000 + seed)
    for nd in P.DIM_CONFIGS:
        for n in (1, 9, 500, 6000):
            agg, vb = [(A.AGGR_SUM_SIGNED, 4), (A.AGGR_SUM_SIGNED, 8), (A.AGGR_SUM_FLOAT, 4), (A.AGGR_SUM_FLOAT, 8),
                       (A.AGGR_SUM_UNSIGNED, 4), (A.AGGR_SUM_UNSIGNED, 8)][rng.integers(0, 6)]
            capacity = n + int(rng.integers(0, 5))
            block = P.random_dim_block(rng, nd, capacity, n, cardinality=int(rng.integers(2, 5)))
            meas = P.random_measures(rng, agg, vb, capacity)
            got = P.run_hash_reduce(impl, block, nd, capacity, n, meas, vb, agg)
            check(chk, got, lambda be: P.run_hash_reduce(be, block, nd, capacity, n, meas, vb, agg),
                  f"hash_reduce nd={nd} n={n} agg={agg}/{vb}")
