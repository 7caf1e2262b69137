"""The AQL front-end subset (aresdb_b200/aql.py) and BASELINE config 1: the reference's
examples/1k_trips data set and its two example queries (count(*) / sum(fare) of completed trips
by hour over the last 24 hours).  The expectation in tests/golden/trips_1k.npz was produced by the
reference's HOST build (tests/golden/make_trips_fixture.py); a numpy restatement of the query
cross-checks the fixture itself."""
import datetime as dt
from pathlib import Path

import numpy as np
import pytest

import harness as H
import reference_golden as R
from reference_golden import reference_results  # noqa: F401  (autouse fixture)
from aresdb_b200 import aql, cabi as A, columns, expr as E
from aresdb_b200.executor import Batch, FusedBatchExecutor, LegacyBatchExecutor

GOLDEN = Path(__file__).resolve().parent / "golden" / "trips_1k.npz"


def _queries():
    def q(measure):
        return {"table": "trips",
                "measures": [{"alias": "value", "sqlExpression": measure, "rowFilters": ["status='completed'"]}],
                "timeFilter": {"column": "request_at", "from": "24 hours ago", "to": "this quarter-hour"},
                "dimensions": [{"alias": "ts", "sqlExpression": "request_at", "timeBucketizer": "hour"}],
                "joins": []}
    return {"total_trips": q("count(*)"), "total_fare": q("sum(fare)")}


@pytest.fixture(scope="module")
def trips():
    z = np.load(GOLDEN)
    names = [str(s) for s in z["status_names"]]
    table = aql.Table("trips", [aql.Column("request_at", A.Uint32), aql.Column("city_id", A.Uint16),
                                aql.Column("status", A.Uint8, enum={n: i for i, n in enumerate(names)}),
                                aql.Column("fare", A.Float32)])
    return z, table, int(z["now"])


def _upload(be, z, table):
    vps, keep = [], []
    for c in table.columns:
        buf, vp = columns.make_column(be.space, c.data_type, z[c.name])
        vps.append(vp)
        keep.append(buf)
    return Batch(vps, len(z["fare"]), keep=keep)


def _check(res, z, name):
    hours = np.array(res.decoded_dims()[0], np.uint32)
    got = dict(zip(hours.tolist(), res.measures.tolist()))
    exp = dict(zip(z[f"{name}_hours"].tolist(), z[f"{name}_values"].tolist()))
    assert got == exp


def test_fixture_agrees_with_numpy(trips):
    """The stored reference results equal an independent numpy evaluation of the two queries."""
    z, table, now = trips
    frm, to = aql.parse_time_filter({"from": "24 hours ago", "to": "this quarter-hour"}, now)
    ts, fare = z["request_at"].astype(np.int64), z["fare"].astype(np.float64)
    keep = (z["status"] == table.columns[2].enum["completed"]) & (ts >= frm) & (ts < to)
    hours = ts[keep] - ts[keep] % 3600
    for name, weights in (("total_trips", None), ("total_fare", fare[keep])):
        uniq = np.unique(hours)
        vals = [(weights[hours == h].sum() if weights is not None else int((hours == h).sum())) for h in uniq]
        exp = dict(zip(z[f"{name}_hours"].tolist(), z[f"{name}_values"].tolist()))
        assert exp == dict(zip(uniq.tolist(), vals))


@pytest.mark.parametrize("name", ["total_trips", "total_fare"])
def test_example_queries_on_cpu_checkers(name, trips, impl):
    if impl.is_gpu:
        pytest.skip("covered by the gpu tests below")
    z, table, now = trips
    ex = LegacyBatchExecutor(impl.lib, impl.space, aql.compile_query(_queries()[name], table, now))
    ex.process_batch(_upload(impl, z, table))
    _check(ex.result(), z, name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["total_trips", "total_fare"])
def test_example_queries_on_b200(name, trips):
    """config 1 through both forms of the engine: per-node entry points and the fused plan."""
    z, table, now = trips
    eng = H.get_backend("b200")
    q = aql.compile_query(_queries()[name], table, now)
    batch = _upload(eng, z, table)
    legacy = LegacyBatchExecutor(eng.lib, eng.space, q)
    legacy.process_batch(batch)
    _check(legacy.result(), z, name)
    fused = FusedBatchExecutor(eng.lib, eng.space, q)
    fused.process_batch(batch)
    _check(fused.result(), z, name)
    fused.close()


# ---- front-end unit tests (reference behaviour cited per case) -------------------------------------------
NOW = int(dt.datetime(2023, 11, 15, 1, 39, 5, tzinfo=dt.timezone.utc).timestamp())   # a Wednesday


def _ts(*a):
    return int(dt.datetime(*a, tzinfo=dt.timezone.utc).timestamp())


@pytest.mark.parametrize("frm,to,exp", [
    ("24 hours ago", "this quarter-hour", (_ts(2023, 11, 14, 1), _ts(2023, 11, 15, 1, 45))),
    ("today", "", (_ts(2023, 11, 15), NOW)),                       # `to` defaults to now (time_filter.go:357-360)
    ("yesterday", "yesterday", (_ts(2023, 11, 14), _ts(2023, 11, 15))),
    ("last week", "this week", (_ts(2023, 11, 6), _ts(2023, 11, 20))),   # weeks start on Monday
    ("this month", "this month", (_ts(2023, 11, 1), _ts(2023, 12, 1))),
    ("this quarter", "this quarter", (_ts(2023, 10, 1), _ts(2024, 1, 1))),
    ("2 years ago", "last year", (_ts(2021, 1, 1), _ts(2023, 1, 1))),
    ("-3d", "-1d", (_ts(2023, 11, 12), _ts(2023, 11, 15))),
    ("2023-Q2", "2023-Q2", (_ts(2023, 4, 1), _ts(2023, 7, 1))),
    ("2023-02", "2023-02-28 13:30", (_ts(2023, 2, 1), _ts(2023, 2, 28, 13, 45))),  # :30 aligns to the quarter-hour
    ("2023-02-28 13:31", "2023-02-28 13", (_ts(2023, 2, 28, 13, 31), _ts(2023, 2, 28, 14))),
    ("1700000000", "1700000060000", (1700000000, 1700000060)),   # epoch seconds / milliseconds
])
def test_time_filter_expressions(frm, to, exp):
    assert aql.parse_time_filter({"from": frm, "to": to}, NOW) == exp


def test_time_bucketizers():
    t = aql.Table("t", [aql.Column("ts", A.Uint32)])
    col = t.ref("ts")

    def floor(e, n):
        return isinstance(e, E.Binary) and e.op == A.Floor and e.rhs.value == n

    for s, n in (("hour", 3600), ("day", 86400), ("minute", 60), ("3m", 180), ("4 hours", 14400), ("quarter-hour", 900),
                 ("30 minutes", 1800), ("12h", 43200)):
        assert floor(aql.time_dimension_expr(s, col), n), s
    for bad in ("7m", "5h", "2d", "fortnight", "61 minutes"):
        with pytest.raises(aql.AQLError):
            aql.time_dimension_expr(bad, col)
    e = aql.time_dimension_expr("hour of day", col)            # floor(ts % 86400, 3600)
    assert floor(e, 3600) and e.lhs.op == A.Mod and e.lhs.rhs.value == 86400
    e = aql.time_dimension_expr("day of week", col)            # floor((ts - 4d) % 7d, 1d) / 86400.0
    assert e.op == A.Divide and e.rhs.value == 86400.0 and e.lhs.lhs.lhs.op == A.Minus and e.lhs.lhs.lhs.rhs.value == 345600
    assert aql.time_dimension_expr("time of day", col).op == A.Mod
    assert aql.time_dimension_expr("week", col).op == A.GetWeekStart
    assert aql.time_dimension_expr("quarter of year", col).op == A.GetQuarterOfYear
    assert floor(aql.time_dimension_expr("10 minutes of day", col), 600)
    with pytest.raises(aql.AQLError):
        aql.time_dimension_expr("7 minutes of day", col)


def test_expression_parser_and_measures():
    t = aql.Table("trips", [aql.Column("request_at", A.Uint32), aql.Column("city_id", A.Uint16),
                            aql.Column("status", A.Uint8, enum={"completed": 0, "canceled": 1}),
                            aql.Column("fare", A.Float32), aql.Column("driver_hll", A.Uint32, hll=True)])
    e = aql.parse_expression("fare > 5.5 and (trips.city_id != 0 or not status = 'canceled')", t)
    assert e.op == A.And and e.lhs.op == A.GreaterThan and e.rhs.op == A.Or and e.rhs.rhs.op == A.Not
    assert e.rhs.rhs.expr.rhs.value == 1                       # enum literal -> dictionary id
    assert aql.parse_expression("status = 'never seen'", t).rhs.value == -1
    assert aql.parse_expression("1 + 2 * 3", t).op == A.Plus   # precedence
    with pytest.raises(aql.AQLError):
        aql.parse_expression("fare = 'completed'", t)

    def q(measure, **kw):
        return aql.compile_query(dict({"table": "trips", "measures": [{"sqlExpression": measure}]}, **kw), t, NOW)

    assert q("count(*)").agg_func == A.AGGR_SUM_UNSIGNED and q("count(*)").measure_bytes == 4
    assert q("sum(fare)").agg_func == A.AGGR_SUM_FLOAT and q("sum(fare)").measure_bytes == 8
    assert q("sum(city_id + 1)").agg_func == A.AGGR_SUM_UNSIGNED
    assert q("min(fare)").agg_func == A.AGGR_MIN_FLOAT and q("max(city_id)").agg_func == A.AGGR_MAX_UNSIGNED
    h = q("countdistincthll(city_id)")
    assert h.is_hll and isinstance(h.measure, E.Unary) and h.measure.op == A.GetHLLValue
    assert isinstance(q("countdistincthll(driver_hll)").measure, E.Col)    # already an hll column: no functor
    assert isinstance(q("hll(driver_hll)").measure, E.Col)
    for bad in ("fare", "sum(fare, 1)", "median(fare)", "hll(city_id)"):
        with pytest.raises(ValueError):
            q(bad)
    with pytest.raises(aql.AQLError):
        q("count(*)", joins=[{"table": "cities"}])
    two_dims = q("count(*)", dimensions=[{"sqlExpression": "request_at", "timeBucketizer": "day"}, {"sqlExpression": "city_id"}])
    assert two_dims.num_dims_per_width == [0, 0, 1, 1, 0]


# ---- time zones with a fixed offset over the query's range -------------------------------------------------------
def _tz_table():
    from aresdb_b200 import aql
    return aql.Table("trips", [aql.Column("request_at", A.Uint32), aql.Column("city_id", A.Uint16),
                               aql.Column("fare", A.Float32)])


def test_parse_timezone_forms():
    import datetime as dt
    from aresdb_b200 import aql
    assert aql.parse_timezone(None) is dt.timezone.utc and aql.parse_timezone("UTC") is dt.timezone.utc
    assert aql.parse_timezone("-8").utcoffset(None) == dt.timedelta(hours=-8)
    assert aql.parse_timezone("5:30").utcoffset(None) == dt.timedelta(hours=5, minutes=30)
    assert aql.parse_timezone("-3:30").utcoffset(None) == -dt.timedelta(hours=3, minutes=30)
    with pytest.raises(aql.AQLError):
        aql.parse_timezone("Not/AZone")


def test_fixed_offset_zone_shifts_time_filter_and_bucketizer():
    """timezone "-8": `today` is the local calendar day (08:00 UTC to 08:00 UTC), and the hour bucketizer floors the
    local clock: FLOOR(request_at + (-28800), 3600) — query/time_bucketizer.go:72-146."""
    from aresdb_b200 import aql, expr as E
    now = 1_727_000_000                                       # 2024-09-22 10:13:20 UTC = 02:13 local
    q = {"table": "trips", "timezone": "-8", "measures": [{"sqlExpression": "count(*)"}],
         "timeFilter": {"column": "request_at", "from": "today"},
         "dimensions": [{"sqlExpression": "request_at", "timeBucketizer": "hour"}]}
    agg = aql.compile_query(q, _tz_table(), now)
    day_start_utc = 1_726_963_200 + 8 * 3600                  # local midnight of 2024-09-22 in UTC-8
    lits = sorted(int(f.rhs.value) for f in agg.filters)
    assert lits == [day_start_utc, now] and agg.tz_offset == -28800
    d = agg.dimensions[0]
    assert d.op == A.Floor and d.lhs.op == A.Plus and int(d.lhs.rhs.value) == -28800 and int(d.rhs.value) == 3600
    utc = aql.compile_query(dict(q, timezone="UTC"), _tz_table(), now)
    assert sorted(int(f.rhs.value) for f in utc.filters) == [1_726_963_200, now] and utc.tz_offset == 0
    assert utc.dimensions[0].lhs.__class__ is E.Col


def test_named_zone_without_a_switch_in_range_and_with_one():
    from aresdb_b200 import aql
    q = {"table": "trips", "timezone": "America/Los_Angeles", "measures": [{"sqlExpression": "count(*)"}],
         "timeFilter": {"column": "request_at", "from": "2024-09-20", "to": "2024-09-21"},
         "dimensions": [{"sqlExpression": "request_at", "timeBucketizer": "day"}]}
    try:
        agg = aql.compile_query(q, _tz_table(), 1_727_000_000)
    except aql.AQLError:
        pytest.skip("no tz database on this box")
    assert agg.tz_offset == -7 * 3600                          # PDT
    assert sorted(int(f.rhs.value) for f in agg.filters) == [1_726_815_600, 1_726_988_400]   # local midnights 09-20 .. 09-22
    q["timeFilter"] = {"column": "request_at", "from": "2024-11-01", "to": "2024-11-05"}      # DST ends 2024-11-03 09:00 UTC
    one = aql.compile_query(q, _tz_table(), 1_731_000_000)
    assert (one.tz_offset, one.tz_to_offset, one.dst_switch) == (-25200, -28800, 1_730_624_400)
    q["timeFilter"] = {"column": "request_at", "from": "2024-01-01", "to": "2025-01-01"}      # two switches, same offset at both ends
    with pytest.raises(aql.AQLError, match="more than one daylight-saving switch"):
        aql.compile_query(q, _tz_table(), 1_731_000_000)


def test_one_switch_in_range_builds_the_references_expression_and_evaluates_to_it():
    """The reference's own case (query/time_bucketizer_test.go:256-330): Los Angeles, 1509772380 .. 1509882360 ->
    requested_at + (-25200 + 3600 * (requested_at >= 1509872400)), FLOOR 3600 — structure and constants; then the same query
    through the reference call sequence on the HOST build and the C restatement against numpy."""
    import harness as H
    import test_pipeline_parity as T
    from aresdb_b200 import aql, synth
    from aresdb_b200.postprocess import DimensionMeta, format_time_dimension
    table = aql.Table("trips", [aql.Column(n, t) for n, t in zip(synth.COLUMN_NAMES, synth.COLUMN_TYPES)])
    q = {"table": "trips", "timezone": "America/Los_Angeles", "measures": [{"sqlExpression": "count(*)"}],
         "timeFilter": {"column": "request_at", "from": "1509772380", "to": "1509882360"},
         "dimensions": [{"sqlExpression": "request_at", "timeBucketizer": "hour"}]}
    try:
        agg = aql.compile_query(q, table, 1_509_900_000)
    except aql.AQLError as e:
        if "parse" in str(e):
            pytest.skip("no tz database on this box")
        raise
    d = agg.dimensions[0]
    assert d.op == A.Floor and int(d.rhs.value) == 3600 and d.lhs.op == A.Plus and isinstance(d.lhs.lhs, E.Col)
    shift = d.lhs.rhs
    assert shift.op == A.Plus and int(shift.lhs.value) == -25200 and shift.lhs.type == E.Type.Signed
    assert shift.rhs.op == A.Multiply and int(shift.rhs.lhs.value) == 3600 and shift.rhs.lhs.type == E.Type.Signed
    assert shift.rhs.rhs.op == A.GreaterThanOrEqual and int(shift.rhs.rhs.rhs.value) == 1_509_872_400
    assert (agg.tz_offset, agg.tz_to_offset, agg.dst_switch) == (-25200, -28800, 1_509_872_400)
    # rows on both sides of the switch
    rng = np.random.default_rng(5)
    n = 5000
    ts = rng.integers(1_509_772_380 - 3000, 1_509_882_360 + 3000, n).astype(np.uint32)
    ones = np.ones(n, np.uint8)
    hb = synth.HostBatch([ts, np.full(n, 3, np.uint16), ones.copy(), np.ones(n, np.float32)], [ones, ones.copy(), ones.copy(), ones.copy()], n, 0)
    keep = (ts >= 1_509_772_380) & (ts < aql.parse_time_filter(q["timeFilter"], 0, aql.parse_timezone("America/Los_Angeles"))[1])
    t64 = ts.astype(np.int64)
    local = t64 + (-25200 + 3600 * (t64 >= 1_509_872_400))
    exp = {}
    for b in (local[keep] // 3600 * 3600).tolist():
        exp[b] = exp.get(b, 0) + 1
    def hours(be):
        res = T.run_legacy(be, agg, [hb])
        return dict(zip(np.array(res.decoded_dims()[0], np.int64).tolist(), res.measures.tolist()))
    got = hours(H.get_backend("oracle"))
    assert got == exp and len(got) > 20
    R.assert_same(exp, R.expected(hours), "reference HOST build")
    # numeric output back to instants (utils.AdjustOffset): buckets before the switch by the from-offset, later ones by the to-offset
    meta = DimensionMeta(time_bucketizer="hour", time_unit="second", from_offset=-25200, to_offset=-28800, dst_switch=1_509_872_400)
    assert format_time_dimension(1_509_872_400 - 28800 - 3600, meta) == str(1_509_872_400 - 28800 - 3600 + 25200)
    assert format_time_dimension(1_509_872_400 - 28800, meta) == str(1_509_872_400)


def test_numeric_time_dimension_output_is_an_instant_again():
    from aresdb_b200.postprocess import DimensionMeta, format_time_dimension
    local_bucket = 1_726_963_200 + 3 * 3600                   # 03:00 on the local clock, produced with offset -8h
    meta = DimensionMeta(time_bucketizer="hour", time_unit="second", from_offset=-28800)
    assert format_time_dimension(local_bucket, meta) == str(local_bucket + 28800)
    assert format_time_dimension(local_bucket, DimensionMeta(time_bucketizer="hour")) == "2024-09-22 03:00"


def test_fixed_offset_query_end_to_end_on_the_checker():
    """The compiled query (shifted time column, local-day time filter) through the reference call sequence on the C
    restatement against a numpy restatement of what it means."""
    import harness as H
    import test_pipeline_parity as T
    from aresdb_b200 import aql, synth
    orc = H.get_backend("oracle")
    table = aql.Table("trips", [aql.Column(n, t) for n, t in zip(synth.COLUMN_NAMES, synth.COLUMN_TYPES)])
    hb = synth.generate_batch(0, 6000, num_cities=5, null_rate=0.0)
    now = synth.BASE_TS + 86400 + 7 * 3600                     # 07:00 UTC of the next day = 23:00 local (UTC-8) of day 0
    q = {"table": "trips", "timezone": "-8", "measures": [{"sqlExpression": "count(*)"}],
         "timeFilter": {"column": "request_at", "from": "today"},
         "dimensions": [{"sqlExpression": "request_at", "timeBucketizer": "hour"}]}
    agg = aql.compile_query(q, table, now)
    got = T.run_legacy(orc, agg, [hb])
    ts = hb.values[synth.COL_REQUEST_AT].astype(np.int64)
    lo = synth.BASE_TS + 8 * 3600                               # local midnight of day 0
    sel = ts[(ts >= lo) & (ts < now)]
    want = {}
    for b in ((sel - 28800) // 3600 * 3600):
        want[int(b)] = want.get(int(b), 0) + 1
    have = {int(d): int(m) for d, m in zip(got.decoded_dims()[0], got.measures)}
    assert have == want and len(have) == 16                     # local hours 00 .. 15 of the data's day


def test_in_lists_null_tests_and_bitwise_operators_end_to_end():
    """`IN` / `NOT IN` (expanded into OR chains of equalities, enum literals through the dictionary), `IS [NOT] NULL`, `& | ^ ~`
    with the reference parser's precedence (query/expr/token.go:302-331) — parsed here, evaluated by the reference call
    sequence on the HOST build and the C restatement, against numpy with three-valued logic (a NULL operand never passes)."""
    import harness as H
    import test_pipeline_parity as T
    from aresdb_b200 import aql, synth
    enum = {"none": 0, "completed": 1, "cancelled": 2, "other": 3}
    table = aql.Table("trips", [aql.Column("request_at", A.Uint32), aql.Column("city_id", A.Uint16),
                                aql.Column("status", A.Uint8, enum=enum), aql.Column("fare", A.Float32)])
    hb = synth.generate_batch(0, 8000, num_cities=9, null_rate=0.08)
    ts, city, status, fare = hb.values
    vt, vc, vs, vf = [v != 0 for v in hb.valid]
    cases = {
        "city_id in (1, 3, 5)": vc & np.isin(city, [1, 3, 5]),
        "city_id not in (1, 3)": vc & ~np.isin(city, [1, 3]),
        "status in ('completed', 'other', 'never heard of')": vs & np.isin(status, [1, 3]),
        "fare is not null": vf,
        "fare is null or city_id in (2)": ~vf | (vc & (city == 2)),
        "city_id & 1 = 1": vc & ((city & 1) == 1),
        "city_id | 4 = 5 and status is not null": vc & ((city | 4) == 5) & vs,
        "city_id ^ 1 * 2 = 4": vc & (((city ^ 1) * 2) == 4),      # XOR binds tighter than * in this grammar
        "~city_id & 7 = 6": vc & (((~city.astype(np.int64)) & 7) == 6),
        "city_id in ()": np.zeros(len(city), bool),
    }
    for text, keep in cases.items():
        q = {"table": "trips", "measures": [{"sqlExpression": "count(*)"}], "rowFilters": [text],
             "dimensions": [{"sqlExpression": "status"}]}
        agg = aql.compile_query(q, table, 0)
        exp = {}
        for s_, ok in zip(status[keep].tolist(), vs[keep].tolist()):
            k = s_ if ok else None
            exp[k] = exp.get(k, 0) + 1
        def groups(be):
            res = T.run_legacy(be, agg, [hb])
            return dict(zip(res.decoded_dims()[0], res.measures.tolist()))
        assert groups(H.get_backend("oracle")) == exp, text
        R.assert_same(exp, R.expected(groups), f"{text}: reference HOST build")
    for bad in ("fare + 1 in (2)", "city_id not 3", "fare is 3", "city_id in 1"):
        with pytest.raises(aql.AQLError):
            aql.parse_expression(bad, table)


def test_a_whole_aql_file_compiles_verbatim(trips):
    """The text of the reference's example files (examples/1k_trips/queries/*.aql, restated here: one element each) through
    compile_request: the same plans as the per-query entry point."""
    import json
    z, table, now = trips
    for name, q in _queries().items():
        text = json.dumps({"queries": [q]}, indent=2)
        got = aql.compile_request(text, table, now)
        one = aql.compile_query(q, table, now)
        assert len(got) == 1 and [repr(f) for f in got[0].filters] == [repr(f) for f in one.filters]
        assert repr(got[0].dimensions) == repr(one.dimensions) and got[0].agg_func == one.agg_func
    assert len(aql.compile_request({"queries": list(_queries().values())}, table, now)) == 2
    with pytest.raises(aql.AQLError):
        aql.compile_request("{}", table, now)
