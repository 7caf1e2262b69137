"""Prefilter slicing of sorted archive batches (aresdb_b200/archive.py; reference qc.prefilterSlice,
query/aql_processor.go:925-982, cVectorParty.SliceByValue / SliceIndex, memstore/vector_party.go:371-432).

Property: running a query WITHOUT its prefilters on the sliced batch gives what the query WITH the prefilters as
ordinary filters gives on the whole batch — checked through the reference's per-node call sequence on the C
restatement and on the reference's own HOST build."""
import numpy as np
import pytest

import harness as H
import test_pipeline_parity as T
from aresdb_b200 import archive as AR
from reference_golden import reference_results  # noqa: F401  (autouse fixture)
from aresdb_b200 import cabi as A
from aresdb_b200 import expr as E, synth
from aresdb_b200.executor import LegacyBatchExecutor
from aresdb_b200.query import AggQuery, Measure

TS, CITY, STATUS, FARE = T.TS, T.CITY, T.STATUS, T.FARE
SCAN = [synth.COL_CITY_ID, synth.COL_STATUS, synth.COL_REQUEST_AT, synth.COL_FARE]   # sort columns first, in sort order
N = 12000


@pytest.fixture(scope="module")
def archive():
    rng = np.random.default_rng(1)
    city = rng.integers(1, 12, N).astype(np.uint16)
    status = rng.integers(0, 4, N).astype(np.uint8)
    order = np.lexsort((status, city))                       # sorted by (city, status), as archiving does
    city, status = city[order], status[order]
    ts = (synth.BASE_TS + rng.integers(0, 86400, N)).astype(np.uint32)
    fare = (rng.integers(0, 6400, N) / 64).astype(np.float32)
    return {synth.COL_CITY_ID: AR.compress(A.Uint16, city), synth.COL_STATUS: AR.compress(A.Uint8, status),
            synth.COL_REQUEST_AT: AR.ArchiveColumn(A.Uint32, ts, (rng.random(N) > 0.02).astype(np.uint8)),
            synth.COL_FARE: AR.ArchiveColumn(A.Float32, fare, (rng.random(N) > 0.02).astype(np.uint8))}


def run(be, q, cols, sl, scan=SCAN):
    ex = LegacyBatchExecutor(be.lib, be.space, q)
    ex.process_batch(AR.to_batch(be.space, {c: cols[c] for c in scan}, 4, sl))
    return ex.result()


def test_slice_by_value_and_index_match_a_linear_scan(archive):
    city = archive[synth.COL_CITY_ID]
    rows = np.repeat(city.values, np.diff(city.counts))
    for v in (0, 1, 5, 11, 12):
        s, e, si, ei = AR.slice_by_value(city, 0, N, v)
        hit = np.flatnonzero(rows == v)
        assert (s, e) == ((int(hit[0]), int(hit[-1]) + 1) if hit.size else (s, s))
        assert city.counts[si] == s and city.counts[ei] == e
    status = archive[synth.COL_STATUS]
    s, e, _, _ = AR.slice_by_value(city, 0, N, 5)
    si, ei = AR.slice_index(status, s, e)
    assert status.counts[si] == s and status.counts[ei] == e          # runs of the finer column nest in the coarser run
    ts = archive[synth.COL_REQUEST_AT]
    assert AR.slice_index(ts, s, e) == (s, e)


@pytest.mark.parametrize("backend_name", ["oracle", "ref"])
@pytest.mark.parametrize("eq, rng_pre, filters", [
    ([7], None, lambda: [E.eq(CITY, E.Lit(7))]),
    ([7], (1, AR.INCLUSIVE, 3, AR.EXCLUSIVE), lambda: [E.eq(CITY, E.Lit(7)), E.ge(STATUS, E.Lit(1)), E.lt(STATUS, E.Lit(3))]),
    ([3, 2], None, lambda: [E.eq(CITY, E.Lit(3)), E.eq(STATUS, E.Lit(2))]),
    ([], (4, AR.EXCLUSIVE, 9, AR.INCLUSIVE), lambda: [E.gt(CITY, E.Lit(4)), E.le(CITY, E.Lit(9))]),
    ([], (6, AR.INCLUSIVE, 0, AR.NO_BOUNDARY), lambda: [E.ge(CITY, E.Lit(6))]),
    ([], None, lambda: []),
])
def test_sliced_batch_equals_filtered_batch(archive, backend_name, eq, rng_pre, filters):
    be = H.get_backend(backend_name)
    dims = [E.floor(TS, E.Lit(3600)), STATUS]
    for measure in (Measure("sum", FARE), Measure("count")):
        whole = AR.prefilter_slice(archive, SCAN, N)
        exp = run(be, AggQuery(filters(), dims, measure), archive, whole)
        sl = AR.prefilter_slice(archive, SCAN, N, equality_values=eq, range_prefilter=rng_pre)
        assert 0 <= sl.start_row <= sl.end_row <= N
        got = run(be, AggQuery([], dims, measure), archive, sl)
        assert exp.groups > 0
        T.assert_same_result(got, exp, ctx=f"prefilter {eq} {rng_pre} {measure.kind}")


def test_absent_values_give_an_empty_slice(archive):
    sl = AR.prefilter_slice(archive, SCAN, N, equality_values=[99])
    assert sl.start_row == sl.end_row
    sl = AR.prefilter_slice(archive, SCAN, N, equality_values=[7], range_prefilter=(9, AR.INCLUSIVE, 20, AR.INCLUSIVE))
    assert sl.start_row == sl.end_row


def test_only_sort_columns_requested_index_space_is_runs(archive):
    """When the finest requested column is itself run-length encoded its runs are the index space (base counts): a
    count(*) then multiplies by the run lengths (query/iterator.hpp:626-645)."""
    orc = H.get_backend("oracle")
    scan = [synth.COL_CITY_ID, synth.COL_STATUS]
    q = AggQuery([], [STATUS], Measure("count"))
    sl = AR.prefilter_slice(archive, scan, N, equality_values=[5])
    got = run(orc, q, archive, sl, scan)
    city = np.repeat(archive[synth.COL_CITY_ID].values, np.diff(archive[synth.COL_CITY_ID].counts))
    status = np.repeat(archive[synth.COL_STATUS].values, np.diff(archive[synth.COL_STATUS].counts))
    want = {int(s): int(((city == 5) & (status == s)).sum()) for s in np.unique(status[city == 5])}
    have = {int(d): int(m) for d, m in zip(got.decoded_dims()[0], got.measures)}
    assert have == want and sl.first_column == synth.COL_STATUS


@pytest.mark.gpu
def test_fused_path_on_sliced_archive_batches():
    """The sliced batch (absolute row numbers in the count vectors, start row for uncompressed columns) through
    ExecuteBatchPlan: RLE columns are expanded once, then the staged fast path runs — same bits as the reference
    sequence on the whole batch with the prefilters as ordinary filters."""
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    from aresdb_b200.executor import FusedBatchExecutor
    rng = np.random.default_rng(2)
    n = 150000
    city = rng.integers(1, 12, n).astype(np.uint16)
    status = rng.integers(0, 4, n).astype(np.uint8)
    order = np.lexsort((status, city))
    city, status = city[order], status[order]
    ts = (synth.BASE_TS + rng.integers(0, 86400, n)).astype(np.uint32)
    fare = (rng.integers(0, 6400, n) / 64).astype(np.float32)
    cols = {synth.COL_CITY_ID: AR.compress(A.Uint16, city), synth.COL_STATUS: AR.compress(A.Uint8, status),
            synth.COL_REQUEST_AT: AR.ArchiveColumn(A.Uint32, ts, (rng.random(n) > 0.02).astype(np.uint8)),
            synth.COL_FARE: AR.ArchiveColumn(A.Float32, fare, (rng.random(n) > 0.02).astype(np.uint8))}
    dims = [E.floor(TS, E.Lit(3600)), STATUS]
    for eq, rng_pre, filters in (([7], None, [E.eq(CITY, E.Lit(7))]),
                                 ([4], (1, AR.INCLUSIVE, 3, AR.EXCLUSIVE), [E.eq(CITY, E.Lit(4)), E.ge(STATUS, E.Lit(1)), E.lt(STATUS, E.Lit(3))])):
        for measure in (Measure("sum", FARE), Measure("count")):
            exp = run(orc, AggQuery(filters, dims, measure), cols, AR.prefilter_slice(cols, SCAN, n))
            sl = AR.prefilter_slice(cols, SCAN, n, equality_values=eq, range_prefilter=rng_pre)
            ex = FusedBatchExecutor(eng.lib, eng.space, AggQuery([], dims, measure))
            b = AR.to_batch(eng.space, cols, 4, sl)
            ex.process_batch(b)
            got = ex.result()
            ex.close()
            T.assert_same_result(got, exp, ctx=f"fused sliced {eq} {rng_pre} {measure.kind}")


def test_match_prefilters_follows_the_sort_column_order():
    """AQLQueryContext.matchPrefilters (query/aql_compiler.go:658-765): equality filters pin leading sort columns, the
    first column with only range filters ends the match, a sort column without a filter ends it too."""
    sort_cols = [synth.COL_CITY_ID, synth.COL_STATUS]
    f = [E.gt(FARE, E.Lit(5.0)), E.eq(CITY, E.Lit(7)), E.lt(STATUS, E.Lit(3)), E.ge(STATUS, E.Lit(1)), E.ge(TS, E.Lit(100))]
    pf = AR.match_prefilters(f, sort_cols)
    assert pf.equality_values == [7] and pf.range_prefilter == (1, AR.INCLUSIVE, 3, AR.EXCLUSIVE)
    assert pf.prefilter_ids == [1, 2, 3] and pf.columns == sort_cols
    pf = AR.match_prefilters([E.eq(STATUS, E.Lit(2))], sort_cols)                  # leading sort column has no filter
    assert pf.equality_values == [] and pf.range_prefilter is None and pf.prefilter_ids == []
    pf = AR.match_prefilters([E.gt(CITY, E.Lit(4)), E.eq(STATUS, E.Lit(2))], sort_cols)   # a range filter ends the match
    assert pf.equality_values == [] and pf.range_prefilter == (4, AR.EXCLUSIVE, 0, AR.NO_BOUNDARY) and pf.prefilter_ids == [0]
    pf = AR.match_prefilters([E.eq(CITY, E.Lit(3)), E.eq(STATUS, E.Lit(2))], sort_cols)
    assert pf.equality_values == [3, 2] and pf.range_prefilter is None
    pf = AR.match_prefilters([E.eq(E.Lit(3), CITY)], sort_cols)                    # literal on the left: not matched
    assert pf.prefilter_ids == []


@pytest.mark.parametrize("seed", range(6))
def test_random_queries_match_slice_run(archive, seed):
    """End to end on the C restatement: match_prefilters -> prefilter_slice -> the query minus its prefilters on the
    slice == the whole query on the whole batch."""
    orc = H.get_backend("oracle")
    rng = np.random.default_rng(100 + seed)
    pool = [E.eq(CITY, E.Lit(int(rng.integers(1, 12)))), E.ge(CITY, E.Lit(int(rng.integers(1, 6)))), E.lt(CITY, E.Lit(int(rng.integers(6, 13)))),
            E.eq(STATUS, E.Lit(int(rng.integers(0, 4)))), E.gt(STATUS, E.Lit(0)), E.le(STATUS, E.Lit(2)), E.gt(FARE, E.Lit(20.0))]
    filters = [pool[i] for i in sorted(rng.choice(len(pool), size=int(rng.integers(1, 5)), replace=False))]
    if any(f.op == A.Equal and f.lhs is CITY for f in filters):
        filters = [f for f in filters if f.lhs is not CITY or f.op == A.Equal]     # one kind of filter per column
    dims = [STATUS, E.floor(TS, E.Lit(7200))]
    exp = run(orc, AggQuery(filters, dims, Measure("count")), archive, AR.prefilter_slice(archive, SCAN, N))
    pf = AR.match_prefilters(filters, [synth.COL_CITY_ID, synth.COL_STATUS])
    rest = [f for i, f in enumerate(filters) if i not in pf.prefilter_ids]
    sl = AR.prefilter_slice(archive, SCAN, N, pf.equality_values, pf.range_prefilter)
    got = run(orc, AggQuery(rest, dims, Measure("count")), archive, sl)
    T.assert_same_result(got, exp, ctx=f"seed {seed}: {len(pf.prefilter_ids)} prefilters of {len(filters)} filters")


def test_archive_scan_evaluates_the_time_filter_on_the_first_and_last_day_only():
    """processShard's archive loop (query/aql_processor.go:222-248, 627-638): the days the time filter touches are scanned,
    the filter itself runs for the first and the last of them; results equal the scan that filters every batch — on the
    reference's HOST build and the oracle — and the plan of a middle batch has two filter instructions less."""
    import harness as H
    import test_pipeline_parity as T
    from aresdb_b200 import aql, archive, cabi as A, synth
    from aresdb_b200.executor import LegacyBatchExecutor
    table = aql.Table("trips", [aql.Column(n, t) for n, t in zip(synth.COLUMN_NAMES, synth.COLUMN_TYPES)])
    day0 = synth.BASE_TS // 86400
    assert synth.BASE_TS % 86400 == 0
    frm, to = synth.BASE_TS + 86400 + 7 * 3600, synth.BASE_TS + 4 * 86400 + 5 * 3600      # day 1 07:00 .. day 4 05:00
    text = {"table": "trips", "measures": [{"sqlExpression": "sum(fare)", "rowFilters": ["status = 1"]}],
            "timeFilter": {"column": "request_at", "from": str(frm), "to": str(to - 1)},
            "dimensions": [{"sqlExpression": "request_at", "timeBucketizer": "hour"}, {"sqlExpression": "city_id"}]}
    q = aql.compile_query(text, table, synth.BASE_TS + 10 * 86400)
    lo, hi = q.time_filter_range
    assert hi - lo == 2 and q.time_range[0] == frm
    assert len(q.plan_instructions()) - len(q.plan_instructions(time_filters=False)) == 2
    assert list(archive.archive_batch_ids(q.time_range, 0)) == [day0 + 1, day0 + 2, day0 + 3, day0 + 4]
    assert list(archive.archive_batch_ids((None, frm), 0)) == list(range(0, day0 + 2))
    assert archive.archive_batch_ids((frm, None), synth.BASE_TS + 2 * 86400 + 5).stop == day0 + 3
    # (an archive batch's time column is never NULL and lies inside its day: that is what makes the rule exact)
    hbs = {day0 + d: synth.generate_batch(d, 3000 + 500 * d, num_cities=6, null_rate=0.0) for d in range(6)}
    def scans(be):
        results = {}
        for rule in (True, False):
            ex = LegacyBatchExecutor(be.lib, be.space, q)
            keep = {day: T.upload(be, hb) for day, hb in hbs.items()}
            if rule:
                results["done"] = [list(d) for d in archive.scan_archive_batches(ex, keep, q.time_range, 0)]
            else:
                for day in archive.archive_batch_ids(q.time_range, 0):
                    ex.process_batch(keep[day])
            results["rule" if rule else "every batch"] = ex.result()
        return results
    import reference_golden as R
    want_done = [[day0 + 1, True], [day0 + 2, False], [day0 + 3, False], [day0 + 4, True]]
    got = scans(H.get_backend("oracle"))
    assert got["done"] == want_done and got["rule"].groups > 60
    T.assert_same_result(got["rule"], got["every batch"], ctx="oracle")
    exp = R.expected(scans)                                # the reference's HOST build
    assert exp["done"] == want_done and exp["rule"]["groups"] > 60
    R.assert_same_result(got["every batch"], exp["every batch"], ctx="reference, every batch")
    R.assert_same_result(got["every batch"], exp["rule"], ctx="reference, first / last day rule")


@pytest.mark.gpu
def test_archive_scan_on_the_fused_path():
    """The same scan through ExecuteBatchPlan: first / last day with the full plan, the days in between with the plan
    that has no time-filter instructions (its own specialised kernel), zone maps on — equal to the oracle's call sequence
    that filters every batch."""
    import harness as H
    import test_pipeline_parity as T
    from aresdb_b200 import aql, archive, synth
    from aresdb_b200.executor import FusedBatchExecutor
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    table = aql.Table("trips", [aql.Column(n, t) for n, t in zip(synth.COLUMN_NAMES, synth.COLUMN_TYPES)])
    day0 = synth.BASE_TS // 86400
    frm, to = synth.BASE_TS + 86400 + 7 * 3600, synth.BASE_TS + 4 * 86400 + 5 * 3600
    for measure in ("sum(fare)", "count(*)"):
        text = {"table": "trips", "measures": [{"sqlExpression": measure, "rowFilters": ["status = 1", "fare > 5.0"]}],
                "timeFilter": {"column": "request_at", "from": str(frm), "to": str(to - 1)},
                "dimensions": [{"sqlExpression": "request_at", "timeBucketizer": "hour"}, {"sqlExpression": "city_id"}]}
        q = aql.compile_query(text, table, synth.BASE_TS + 10 * 86400)
        hbs = {day0 + d: synth.generate_batch(d, 30000 + 5000 * d, num_cities=20, null_rate=0.0) for d in range(6)}
        exp = T.run_legacy(orc, q, [hbs[d] for d in archive.archive_batch_ids(q.time_range, 0)])
        for zone_maps in (False, True):
            ex = FusedBatchExecutor(eng.lib, eng.space, q)
            keep = {day: T.upload(eng, hb, 0, synth.zone_map(hb) if zone_maps else None) for day, hb in hbs.items()}
            done = archive.scan_archive_batches(ex, keep, q.time_range, 0)
            assert [d for d, _ in done] == list(range(day0 + 1, day0 + 5)) and [f for _, f in done] == [True, False, False, True]
            got = ex.result()
            ex.close()
            T.assert_same_result(got, exp, ctx=f"{measure} zone_maps={zone_maps}")


def test_shard_scan_live_batches_with_the_cutoff_filter_then_archive_days():
    """processShard (query/aql_processor.go:166-248): live batches carry rows on both sides of the archiving cutoff — those
    below it are the archive's and are cut by `time >= cutoff` —, archive days are scanned when the range starts below the
    cutoff.  count(*) by hour against numpy, on the reference's HOST build and the oracle; ranges that end before the cutoff
    or start after it touch one store only."""
    import harness as H
    import test_pipeline_parity as T
    from aresdb_b200 import aql, archive, synth
    from aresdb_b200.executor import LegacyBatchExecutor
    table = aql.Table("trips", [aql.Column(n, t) for n, t in zip(synth.COLUMN_NAMES, synth.COLUMN_TYPES)])
    day0 = synth.BASE_TS // 86400
    cutoff = synth.BASE_TS + 3 * 86400
    arch = {day0 + d: synth.generate_batch(d, 2500, num_cities=4, null_rate=0.0) for d in range(3)}          # days 0..2
    rng = np.random.default_rng(11)
    live = []
    for i in range(3):          # unsorted rows of days 1..5: part of them already archived
        hb = synth.generate_batch(7 + i, 3000, num_cities=4, null_rate=0.0)
        hb.values[0] = (synth.BASE_TS + rng.integers(1 * 86400, 6 * 86400, hb.num_rows)).astype(np.uint32)
        live.append(hb)

    def expected(frm, to):
        out = {}
        days = archive.archive_batch_ids((frm, to), 0)
        ts = [arch[d].values[0] for d in days if d in arch and cutoff > frm] + ([hb.values[0][hb.values[0] >= cutoff] for hb in live] if cutoff < to else [])
        for t in np.concatenate(ts).astype(np.int64) if ts else []:
            if frm <= t < to:
                out[int(t) // 3600 * 3600] = out.get(int(t) // 3600 * 3600, 0) + 1
        return out

    ranges = {"both": (synth.BASE_TS + 86400 + 1800, synth.BASE_TS + 5 * 86400 - 1800),
              "archive only": (synth.BASE_TS + 3600, synth.BASE_TS + 2 * 86400),
              "live only": (cutoff + 7200, cutoff + 2 * 86400)}
    import reference_golden as R
    for name, (frm, to) in ranges.items():
        text = {"table": "trips", "measures": [{"sqlExpression": "count(*)"}],
                "timeFilter": {"column": "request_at", "from": str(frm), "to": str(to - 1)},
                "dimensions": [{"sqlExpression": "request_at", "timeBucketizer": "hour"}]}
        q = aql.compile_query(text, table, synth.BASE_TS + 30 * 86400)
        frm, to = q.time_range

        def scan(be):
            ex = LegacyBatchExecutor(be.lib, be.space, q)
            done = archive.scan_shard(ex, [T.upload(be, hb) for hb in live], {d: T.upload(be, hb) for d, hb in arch.items()},
                                      cutoff, q.time_range, 0)
            res = ex.result()
            return {"live": done["live"] > 0, "archive": len(done["archive"]) > 0,
                    "hours": dict(zip(np.array(res.decoded_dims()[0], np.int64).tolist(), res.measures.tolist()))}
        want = {"live": name != "archive only", "archive": name != "live only", "hours": expected(frm, to)}
        assert scan(H.get_backend("oracle")) == want and len(want["hours"]) > 10, name
        R.assert_same(want, R.expected(scan), f"{name}: reference HOST build")
    # the cutoff filter is one more filter instruction, ahead of the time filters
    assert len(q.plan_instructions(cutoff=cutoff)) == len(q.plan_instructions()) + 1


@pytest.mark.gpu
def test_shard_scan_on_the_fused_path():
    """Live batches with the cutoff filter (a plan with one more filter instruction, the cutoff a literal), archive days
    with / without the time filters: ExecuteBatchPlan against the oracle's call sequence over the same scan."""
    import harness as H
    import test_pipeline_parity as T
    from aresdb_b200 import aql, archive, synth
    from aresdb_b200.executor import FusedBatchExecutor, LegacyBatchExecutor
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    table = aql.Table("trips", [aql.Column(n, t) for n, t in zip(synth.COLUMN_NAMES, synth.COLUMN_TYPES)])
    day0 = synth.BASE_TS // 86400
    cutoff = synth.BASE_TS + 3 * 86400
    arch = {day0 + d: synth.generate_batch(d, 20000, num_cities=12, null_rate=0.0) for d in range(3)}
    rng = np.random.default_rng(11)
    live = []
    for i in range(3):
        hb = synth.generate_batch(7 + i, 25000, num_cities=12, null_rate=0.0)
        hb.values[0] = (synth.BASE_TS + rng.integers(1 * 86400, 6 * 86400, hb.num_rows)).astype(np.uint32)
        live.append(hb)
    frm, to = synth.BASE_TS + 86400 + 1800, synth.BASE_TS + 5 * 86400 - 1800
    text = {"table": "trips", "measures": [{"sqlExpression": "sum(fare)", "rowFilters": ["status = 1"]}],
            "timeFilter": {"column": "request_at", "from": str(frm), "to": str(to)},
            "dimensions": [{"sqlExpression": "request_at", "timeBucketizer": "hour"}, {"sqlExpression": "city_id"}]}
    q = aql.compile_query(text, table, synth.BASE_TS + 30 * 86400)
    results = []
    for be, cls in ((orc, LegacyBatchExecutor), (eng, FusedBatchExecutor)):
        ex = cls(be.lib, be.space, q)
        keep_live = [T.upload(be, hb, 0, synth.zone_map(hb) if be is eng else None) for hb in live]
        keep_arch = {d: T.upload(be, hb, 0, synth.zone_map(hb) if be is eng else None) for d, hb in arch.items()}
        done = archive.scan_shard(ex, keep_live, keep_arch, cutoff, q.time_range, 0)
        # days 1 .. 4 are scanned; the archive holds 1 and 2: the first scanned day with the time filter, day 2 without
        assert done["live"] == 3 and done["archive"] == [(day0 + 1, True), (day0 + 2, False)]
        results.append(ex.result())
    assert results[0].groups > 500
    T.assert_same_result(results[1], results[0], ctx="shard scan")
