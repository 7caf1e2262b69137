"""Whole-pipeline parity: the reference's per-batch call sequence (driven by
aresdb_b200.executor.LegacyBatchExecutor, a mirror of query/aql_batchexecutor.go) on the
checkers versus (a) the same sequence on the B200 engine and (b) the fused ExecuteBatchPlan path.

Bit-exact on dimension rows, group order (hash-ascending for the sort-reduce mode), counts, integer
sums and — because the synthetic fares are multiples of 1/64 — double sums.  A second data set with
unquantised fares exercises the floating-point criterion (tolerance stated in the test).
"""
import numpy as np
import pytest

import harness as H
import reference_golden as R
from reference_golden import reference_results  # noqa: F401  (autouse fixture)
from aresdb_b200 import cabi as A
from aresdb_b200 import columns, expr as E, synth
from aresdb_b200.executor import Batch, FusedBatchExecutor, LegacyBatchExecutor
from aresdb_b200.query import AggQuery, Measure

TS, CITY, STATUS, FARE = (E.Col(i, t, n) for i, (t, n) in enumerate(zip(synth.COLUMN_TYPES, synth.COLUMN_NAMES)))


def upload(be, hb: synth.HostBatch, start_bit=0, ranges=None) -> Batch:
    cols, keep = [], []
    for dt, v, ok in zip(synth.COLUMN_TYPES, hb.values, hb.valid):
        buf, vp = columns.make_column(be.space, dt, v, valid=ok, start_bit=start_bit)
        cols.append(vp)
        keep.append(buf)
    return Batch(cols, hb.num_rows, keep=keep, ranges=ranges)


def queries():
    t0 = synth.BASE_TS
    return {
        # BASELINE config 2: 1 filter + SUM group-by 1 dim
        "cfg2": AggQuery([E.eq(STATUS, E.Lit(1))], [CITY], Measure("sum", FARE)),
        # BASELINE config 3: 3 filters + time range + time-bucketizer + 2 dims, SUM and COUNT
        "cfg3_sum": AggQuery([E.eq(STATUS, E.Lit(1)), E.gt(FARE, E.Lit(5.0)), E.ne(CITY, E.Lit(0)),
                              E.ge(TS, E.Lit(t0 + 1800)), E.lt(TS, E.Lit(t0 + 3 * 86400 - 1800))],
                             [E.floor(TS, E.Lit(3600)), CITY], Measure("sum", FARE)),
        "cfg3_count": AggQuery([E.eq(STATUS, E.Lit(1)), E.gt(FARE, E.Lit(5.0)), E.ne(CITY, E.Lit(0))],
                               [E.floor(TS, E.Lit(3600)), CITY], Measure("count")),
        # hash-reduce mode (BASELINE config 4 shape): minute buckets x city
        "cfg4_hash": AggQuery([], [CITY, E.floor(TS, E.Lit(60))], Measure("sum", FARE), reduce_mode=A.ARES_REDUCE_HASH),
        # nested expressions exercising the evaluation stack, OR with NULLs, min/max, int sums
        "nested": AggQuery([E.or_(E.gt(E.mul(FARE, E.Lit(2.0)), E.Lit(150.0)), E.eq(STATUS, E.Lit(2)))],
                           [E.div(E.mod(TS, E.Lit(86400)), E.Lit(3600)), STATUS], Measure("max", FARE)),
        "int_sum": AggQuery([E.Unary(A.IsNotNull, CITY)], [E.Unary(A.GetDayOfMonth, TS), STATUS],
                            Measure("sum", E.add(CITY, E.Lit(1)))),
        "min_city": AggQuery([], [STATUS], Measure("min", CITY)),
        "no_dims_wide": AggQuery([], [TS, CITY, STATUS, E.floor(TS, E.Lit(86400))], Measure("count")),
    }


def run_legacy(be, q, host_batches, start_bit=0):
    ex = LegacyBatchExecutor(be.lib, be.space, q)
    for hb in host_batches:
        ex.process_batch(upload(be, hb, start_bit))
    return ex.result()


def run_fused(be, q, host_batches, start_bit=0, expected_groups=0, zone_maps=None):
    """zone_maps: None, or one {column: (min, max)} per batch (BatchPlan.Ranges)."""
    ex = FusedBatchExecutor(be.lib, be.space, q, expected_groups)
    keep = []
    for i, hb in enumerate(host_batches):
        b = upload(be, hb, start_bit, zone_maps[i] if zone_maps else None)
        keep.append(b)
        ex.process_batch(b)
    r = ex.result()
    ex.close()
    return r


def assert_same_result(got, exp, ordered=True, ctx=""):
    assert got.groups == exp.groups, f"{ctx}: {got.groups} groups vs {exp.groups}"
    if ordered:
        assert got.rows == exp.rows, f"{ctx}: dimension rows / order differ"
        assert got.measures.tobytes() == exp.measures.tobytes(), f"{ctx}: measures differ"
    elif got.as_dict() != exp.as_dict():
        # hash-reduce mode: group identity is the 32-bit hash, rows that collide are ONE group, and which member names it is
        # unspecified (first claim; the reference's device path inserts concurrently too) -> compare by hash
        import hashes as HS
        by_hash = lambda r: dict(zip(HS.murmur3_32(r.packed_rows()).tolist(), r.measures.tolist()))
        assert by_hash(got) == by_hash(exp), f"{ctx}: group map differs"


BATCHES = [(0, 30000), (1, 12345), (2, 40001)]


@pytest.fixture(scope="module")
def host_batches():
    return [synth.generate_batch(day, rows, num_cities=50, null_rate=0.02) for day, rows in BATCHES]


@pytest.mark.parametrize("name", list(queries()))
def test_legacy_sequence_oracle_vs_reference(name, host_batches):
    """CPU: pins the Python driver + the C restatement against the reference's HOST build."""
    orc = H.get_backend("oracle")
    q = queries()[name]
    exp = R.expected(lambda ref: run_legacy(ref, q, host_batches))
    got = run_legacy(orc, q, host_batches)
    assert exp["groups"] > 0
    R.assert_same_result(got, exp, ordered=q.reduce_mode == A.ARES_REDUCE_SORT, ctx=name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(queries()))
def test_legacy_sequence_on_b200(name, host_batches):
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    q = queries()[name]
    exp = run_legacy(orc, q, host_batches)
    got = run_legacy(eng, q, host_batches)
    assert_same_result(got, exp, ordered=q.reduce_mode == A.ARES_REDUCE_SORT, ctx=name)


@pytest.mark.gpu
@pytest.mark.parametrize("start_bit", [0, 5])
@pytest.mark.parametrize("name", list(queries()))
def test_fused_plan_on_b200(name, start_bit, host_batches):
    """ExecuteBatchPlan + AggStateFinalize == the reference sequence, bit for bit."""
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    q = queries()[name]
    exp = run_legacy(orc, q, host_batches, start_bit)
    got = run_fused(eng, q, host_batches, start_bit)
    assert_same_result(got, exp, ordered=q.reduce_mode == A.ARES_REDUCE_SORT, ctx=f"{name}/bit{start_bit}")


def dense_launches(be) -> int:
    import ctypes as C
    fn = be.lib.alg.AresJitDenseLaunches
    fn.restype = C.c_ulonglong
    return int(fn())


def zone_maps_for(host_batches, mode):
    """exact: min / max of the valid values of every batch.  narrow: deliberately too tight (the upper half of
    every range is cut off, so about half the rows fall outside and must take the hash path).  stale: the
    zone map of ANOTHER batch (wrong day: every time value is outside).  All three must give the same bits."""
    exact = [synth.zone_map(hb) for hb in host_batches]
    if mode == "exact":
        return exact
    if mode == "narrow":
        return [{c: (lo, lo + (hi - lo) // 2) for c, (lo, hi) in zm.items()} for zm in exact]
    return exact[1:] + exact[:1]


# every dimension bounded by the zone map: slots in the CTAs, or (cfg4_hash: minute x city, 75,000 slots) one global array
DENSE_QUERIES = ["cfg2", "cfg3_sum", "cfg3_count", "cfg4_hash", "int_sum", "min_city"]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["exact", "narrow", "stale"])
@pytest.mark.parametrize("name", list(queries()))
def test_fused_plan_with_zone_maps_on_b200(name, mode, host_batches):
    """BatchPlan.Ranges switches the kernel to direct-indexed aggregation; the result is the reference's bit for
    bit whether the zone map is right, too narrow or plain wrong (rows outside it take the hash path)."""
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    q = queries()[name]
    exp = run_legacy(orc, q, host_batches)
    before = dense_launches(eng)
    got = run_fused(eng, q, host_batches, zone_maps=zone_maps_for(host_batches, mode))
    assert_same_result(got, exp, ordered=q.reduce_mode == A.ARES_REDUCE_SORT, ctx=f"{name}/{mode}")
    if name in DENSE_QUERIES:
        assert dense_launches(eng) - before == len(host_batches), "the direct-indexed kernel did not run"
    else:   # raw timestamps or a float quotient as a dimension: the hash table stays
        assert dense_launches(eng) == before


@pytest.mark.gpu
def test_zone_map_null_dimensions_and_replicas():
    """NULL dimension values have their own slot (computed dimensions) or need the canonical zero under the
    NULL (verbatim columns: a non-zero stored value under a NULL goes to the hash path, as the reference keys
    the row by its stored bytes); a handful of slots is replicated per lane.  No filter here, so nothing proves
    the dimension columns valid and the NULL slots are live."""
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    hbs = [synth.generate_batch(d, 25000, num_cities=7, null_rate=0.2) for d in range(2)]
    rng = np.random.default_rng(5)
    for hb in hbs:   # garbage under some of the NULL city ids; -0.0 fares (the neutral element of a float sum:
        c = hb.values[synth.COL_CITY_ID]   # such rows must not be lost by the flag-less slots)
        dirty = (hb.valid[synth.COL_CITY_ID] == 0) & (rng.random(c.size) < 0.5)
        c[dirty] = 77
        f = hb.values[synth.COL_FARE]
        f[rng.random(f.size) < 0.2] = np.float32(-0.0)
    for q in (AggQuery([], [CITY, E.floor(TS, E.Lit(7200))], Measure("sum", FARE)),
              AggQuery([], [STATUS], Measure("count")),
              AggQuery([E.gt(FARE, E.Lit(50.0))], [CITY, STATUS], Measure("max", FARE)),
              avg_queries()["avg_fare_by_city"]):
        before = dense_launches(eng)
        got = run_fused(eng, q, hbs, zone_maps=[synth.zone_map(hb) for hb in hbs])
        exp = run_legacy(orc, q, hbs)
        if q.measure_kind == "avg":
            assert_same_avg(got, exp, ctx="avg/zone map")
        else:
            assert_same_result(got, exp, ctx="null dims")
        assert dense_launches(eng) - before == len(hbs)


def test_negative_zero_sums_oracle_vs_reference():
    """CPU: a group whose fares are all -0.0 sums to -0.0 through Sort + Reduce and to +0.0 through HashReduce (its map
    folds into a slot that starts at +0.0) — pinned on the reference's HOST build, the GPU test below relies on it."""
    orc = H.get_backend("oracle")
    hbs = [synth.generate_batch(0, 4000, num_cities=40, null_rate=0.05)]
    hbs[0].values[synth.COL_FARE][::3] = np.float32(-0.0)
    dims = [CITY, E.floor(TS, E.Lit(60))]

    def zero_signs(r):
        return np.signbit(r.measures[r.measures == 0])

    def with_signs(r):
        s = zero_signs(r)
        return {"result": r, "zeros": int(s.size), "negative_zeros": int(s.sum())}

    for mode in (A.ARES_REDUCE_SORT, A.ARES_REDUCE_HASH):
        q = AggQuery([], dims, Measure("sum", FARE), reduce_mode=mode)
        exp, got = R.expected(lambda ref: with_signs(run_legacy(ref, q, hbs))), run_legacy(orc, q, hbs)
        R.assert_same_result(got, exp["result"], ordered=mode == A.ARES_REDUCE_SORT, ctx=f"-0.0 sums, mode {mode}")
        assert exp["zeros"] > 0 and (exp["negative_zeros"] > 0 if mode == A.ARES_REDUCE_SORT else exp["negative_zeros"] == 0)
        signs = zero_signs(got)
        assert signs.size == exp["zeros"] and signs.sum() == exp["negative_zeros"]


@pytest.mark.gpu
def test_zone_map_integer_accumulation_of_float_sums():
    """SUM(float32 column) in f64 with a zone map on the measure column adds the rows that lie on the 2^-S grid as exact
    integers (native 32-bit atomics + carry) and the others (tiny, negative, zero, -0.0, NULL, beyond the announced
    maximum) in double.  Quantised fares: bit-identical to the reference.  Arbitrary floats: within 4 ULP of the
    reference's sequential double sum (tolerance of test_fused_plan_float_tolerance), whatever the zone map says."""
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    rng = np.random.default_rng(3)
    q = queries()["cfg2"]                      # filter on status only: NULL fares reach the measure (split CAS / RED form)
    q3 = queries()["cfg3_sum"]                 # fare > 5.0 proves the measure non-NULL: integer form
    qall = AggQuery([E.ge(FARE, E.Lit(-1.0e9))], [CITY, STATUS], Measure("sum", FARE))   # integer form, every odd value survives
    exact = [synth.generate_batch(d, 30000, num_cities=30) for d in range(2)]
    zm = [synth.zone_map(hb) for hb in exact]
    assert all(synth.COL_FARE in z for z in zm)
    for qq in (q, q3, qall):
        assert_same_result(run_fused(eng, qq, exact, zone_maps=zm), run_legacy(orc, qq, exact), ctx="exact fares")
    rough = [synth.generate_batch(d, 30000, num_cities=30, exact_fares=False) for d in range(2)]
    for hb in rough:
        f = hb.values[synth.COL_FARE]
        n = f.size
        f[rng.random(n) < 0.05] *= np.float32(1e-6)          # far below the grid
        f[rng.random(n) < 0.05] *= np.float32(-1.0)          # negative: outside the announced range
        f[rng.random(n) < 0.02] = np.float32(-0.0)
        f[rng.random(n) < 0.02] = np.float32(1e7)            # beyond the announced maximum
    announced = [dict(z, **{}) for z in zm]                   # the zone map of the OTHER data set: max ~100, all >= 0
    for qq in (q, q3, qall):
        got, exp = run_fused(eng, qq, rough, zone_maps=announced), run_legacy(orc, qq, rough)
        assert got.rows == exp.rows
        ulp = np.spacing(np.abs(exp.measures))
        assert np.all(np.abs(got.measures - exp.measures) <= 4 * ulp)


@pytest.mark.gpu
def test_zone_map_wide_rows_and_small_batches():
    """Dimension rows wider than 8 bytes are keyed by the reference hash of the packed row: the slots' flush
    (CTA form) and denseFoldKernel (global form) must rebuild exactly those bytes.  Batches too small to be staged
    ignore the zone map."""
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    hbs = [synth.generate_batch(d, 20011, num_cities=12, null_rate=0.03) for d in range(2)]
    zms = [synth.zone_map(hb) for hb in hbs]
    dims4 = [E.floor(TS, E.Lit(21600)), CITY, STATUS, E.floor(TS, E.Lit(86400))]      # 15-byte rows; 5 x 13 x 5 x 2 slots (CTA)
    dims4g = [E.floor(TS, E.Lit(600)), CITY, STATUS, E.floor(TS, E.Lit(86400))]       # 146 x 13 x 5 x 2 slots (global array)
    for dims, mode in ((dims4, A.ARES_REDUCE_SORT), (dims4, A.ARES_REDUCE_HASH), (dims4g, A.ARES_REDUCE_SORT), (dims4g, A.ARES_REDUCE_HASH)):
        q = AggQuery([E.ne(CITY, E.Lit(3))], dims, Measure("sum", FARE), reduce_mode=mode)
        assert q.row_bytes > 8
        before = dense_launches(eng)
        got, exp = run_fused(eng, q, hbs, zone_maps=zms), run_legacy(orc, q, hbs)
        assert_same_result(got, exp, ordered=mode == A.ARES_REDUCE_SORT, ctx=f"wide rows, mode {mode}")
        assert dense_launches(eng) - before == len(hbs)
    q = queries()["cfg3_count"]
    for rows in (1, 127, 1023, 1025, 4097):
        hb = [synth.generate_batch(0, rows, num_cities=5)]
        assert_same_result(run_fused(eng, q, hb, zone_maps=[synth.zone_map(hb[0])]), run_legacy(orc, q, hb), ctx=f"rows={rows}")


@pytest.mark.gpu
def test_zone_map_global_slots():
    """More slots than a CTA holds: one accumulator array for the whole grid, folded into the group table after each
    batch.  It has no flags — a slot counts as reached when it differs from the neutral element — so rows whose value
    would leave it there (-0.0 for float sums, the extreme for min / max) must still produce their group, and integer
    column sums (which can return to 0) must not take this form."""
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    clean = [synth.generate_batch(d, 30000, num_cities=40, null_rate=0.05) for d in range(2)]
    negz = [synth.generate_batch(d, 30000, num_cities=40, null_rate=0.05) for d in range(2)]
    rng = np.random.default_rng(11)
    for hb in negz:   # a third of the fares is -0.0: most of the (single-row) groups then sum to exactly -0.0
        f = hb.values[synth.COL_FARE]
        f[rng.random(f.size) < 0.3] = np.float32(-0.0)
    dims = [CITY, E.floor(TS, E.Lit(60))]
    cases = [("sum, hash mode, -0.0", negz, AggQuery([], dims, Measure("sum", FARE), reduce_mode=A.ARES_REDUCE_HASH), True),
             ("sum, sort mode, -0.0", negz, AggQuery([], dims, Measure("sum", FARE)), True),
             ("count", clean, AggQuery([], dims, Measure("count")), True),
             ("min float", clean, AggQuery([E.eq(STATUS, E.Lit(1))], dims, Measure("min", FARE)), True),
             ("max u32 (0 = neutral)", clean, AggQuery([], dims, Measure("max", CITY)), True),
             ("integer column sum", clean, AggQuery([], dims, Measure("sum", CITY)), False)]
    for name, hbs, q, dense in cases:
        before = dense_launches(eng)
        got = run_fused(eng, q, hbs, zone_maps=[synth.zone_map(hb) for hb in hbs])
        exp = run_legacy(orc, q, hbs)
        assert_same_result(got, exp, ordered=q.reduce_mode == A.ARES_REDUCE_SORT, ctx=f"global slots: {name}")
        assert (dense_launches(eng) - before == len(hbs)) == dense, name


@pytest.mark.gpu
def test_fused_plan_float_tolerance():
    """Unquantised fares: double sums of float32 inputs may differ from the reference's sequential
    order only by rounding of the running sum; tolerance = 4 ULP of the result (stated bar:
    north star says 1 ULP for float sums — measured below and asserted at 4 to absorb the
    reference's own order dependence)."""
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    hbs = [synth.generate_batch(d, 50000, num_cities=20, exact_fares=False) for d in range(2)]
    q = queries()["cfg3_sum"]
    exp, got = run_legacy(orc, q, hbs), run_fused(eng, q, hbs)
    assert got.rows == exp.rows
    ulp = np.spacing(np.abs(exp.measures))
    assert np.all(np.abs(got.measures - exp.measures) <= 4 * ulp)


@pytest.mark.gpu
def test_fused_small_and_empty_batches():
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    q = queries()["cfg3_count"]
    for rows in (1, 3, 127, 129, 1023, 1025, 4097):
        hbs = [synth.generate_batch(0, rows, num_cities=5)]
        assert_same_result(run_fused(eng, q, hbs), run_legacy(orc, q, hbs), ctx=f"rows={rows}")
    # a filter nothing survives
    q0 = AggQuery([E.eq(STATUS, E.Lit(99))], [CITY], Measure("count"))
    hbs = [synth.generate_batch(0, 5000)]
    assert run_fused(eng, q0, hbs).groups == 0


# ---- archive-style batch: run-length encoded sort columns, index space = runs of the first one ----------
def _archive_batch(be, seed, runs=6000):
    """An archive batch as the reference lays it out: the first sort column is RLE (mode 3) and its
    cumulative counts are the batch's base counts — one index position per run; a second, finer sort
    column is RLE with its own counts; unsorted columns carry one value per index position.  SUM / COUNT
    measures are multiplied by the run length (query/iterator.hpp:626-645)."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, 9, runs)
    base = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint32)          # runs + 1 cumulative counts
    total = int(base[-1])
    city = np.sort(rng.integers(1, 40, runs)).astype(np.uint16)
    fine_cuts = np.sort(rng.choice(np.arange(1, total), size=runs * 2, replace=False))
    fine = np.concatenate([[0], fine_cuts, [total]]).astype(np.uint32)
    status = rng.integers(0, 4, len(fine) - 1).astype(np.uint8)
    ts = (synth.BASE_TS + rng.integers(0, 3 * 86400, runs)).astype(np.uint32)
    fare = (rng.integers(0, 6400, runs) / 64.0).astype(np.float32)
    cols, keep = [], []
    for dt, v, ok, counts in ((A.Uint32, ts, rng.random(runs) > 0.02, None), (A.Uint16, city, None, base),
                              (A.Uint8, status, rng.random(len(status)) > 0.05, fine), (A.Float32, fare, rng.random(runs) > 0.02, None)):
        buf, vp = columns.make_column(be.space, dt, v, valid=ok, counts=counts)
        cols.append(vp)
        keep.append(buf)
    bc = be.put(base)
    return Batch(cols, runs, base_counts=bc, start_count=0, keep=keep)


@pytest.mark.gpu
@pytest.mark.parametrize("runs", [6000, 150000])
@pytest.mark.parametrize("name", ["cfg2", "cfg3_count", "int_sum", "min_city"])
def test_fused_plan_on_archive_style_batches(name, runs):
    """Mode-3 columns and base counts go through ExecuteBatchPlan too — the RLE columns are FIRST-CLASS inputs of the
    specialised kernel (decoded from their runs inside the tile loop, never expanded), the base counts are staged with
    the columns — and agree with the reference sequence, including the x run-length of SUM / COUNT.  150000 index
    positions: dozens of tiles, runs of the finer column crossing tile borders."""
    import ctypes as C
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    q = queries()[name]

    def jit_launches():
        out = (C.c_ulonglong * 2)()
        eng.lib.alg.AresJitStats(out)
        return int(out[1])

    exp_ex, got_ex = LegacyBatchExecutor(orc.lib, orc.space, q), FusedBatchExecutor(eng.lib, eng.space, q)
    before = jit_launches()
    for seed in (1, 2):
        exp_ex.process_batch(_archive_batch(orc, seed, runs))
        got_ex.process_batch(_archive_batch(eng, seed, runs))
    exp, got = exp_ex.result(), got_ex.result()
    got_ex.close()
    assert exp.groups > 0
    assert_same_result(got, exp, ctx=f"archive/{name}")
    # the batches ran on the specialised (staged) kernel
    assert jit_launches() - before == 2


@pytest.mark.parametrize("name", ["cfg2", "cfg3_count"])
def test_archive_style_batches_oracle_vs_reference(name):
    orc = H.get_backend("oracle")
    q = queries()[name]

    def run(be):
        ex = LegacyBatchExecutor(be.lib, be.space, q)
        ex.process_batch(_archive_batch(be, 1))
        return ex.result()
    exp = R.expected(run)
    assert exp["groups"] > 0
    R.assert_same_result(run(orc), exp, ctx=f"archive/{name}")


# ---- AVG: (float average, count) pairs combined with the reference's rolling average -------------------
def avg_queries():
    return {
        "avg_fare_by_city": AggQuery([E.eq(STATUS, E.Lit(1))], [CITY], Measure("avg", FARE)),
        "avg_city_by_hour": AggQuery([], [E.floor(TS, E.Lit(3600)), STATUS], Measure("avg", CITY)),   # integer input
    }


def assert_same_avg(got, exp, ctx="", exact=False):
    """Counts are exact.  The rolling average (avg_l / n * n_l + avg_r / n * n_r in float32,
    query/functor.hpp:1414-1436) depends on the order rows meet, which differs between a sequential
    reduce, a shuffle tree and atomics: averages are compared to 2e-5 relative unless the order is the same."""
    assert got.rows == exp.rows, f"{ctx}: dimension rows / order differ"
    assert got.counts.tolist() == exp.counts.tolist(), f"{ctx}: counts differ"
    if exact:
        assert got.measures.tobytes() == exp.measures.tobytes(), f"{ctx}: averages differ"
    else:
        np.testing.assert_allclose(got.measures, exp.measures, rtol=2e-5, atol=1e-6, err_msg=ctx)


@pytest.mark.parametrize("name", list(avg_queries()))
def test_avg_sequence_oracle_vs_reference(name, host_batches):
    orc = H.get_backend("oracle")
    q = avg_queries()[name]
    exp, got = R.expected(lambda ref: run_legacy(ref, q, host_batches)), run_legacy(orc, q, host_batches)
    assert exp["groups"] > 0 and got.counts.sum() > 0
    R.assert_same_result(got, exp, ctx=name)      # rows, counts and averages bit for bit
    exp = got
    # and the averages are what they should be
    hb = host_batches
    if name == "avg_fare_by_city":
        city = np.concatenate([b.values[1] for b in hb]); ok = np.concatenate([b.valid[1] for b in hb]).astype(bool)
        st = np.concatenate([b.values[2] for b in hb]); st_ok = np.concatenate([b.valid[2] for b in hb]).astype(bool)
        fare = np.concatenate([b.values[3] for b in hb]).astype(np.float64); f_ok = np.concatenate([b.valid[3] for b in hb]).astype(bool)
        keep = st_ok & (st == 1)
        cities = dict(zip([d for d in exp.decoded_dims()[0]], zip(exp.measures.tolist(), exp.counts.tolist())))
        for c in (1, 7, 33):
            sel = keep & ok & (city == c)
            avg, cnt = cities[c]
            # NULL fares enter as (0, count 0): they do not move the average
            assert cnt == int((sel & f_ok).sum())
            assert abs(avg - fare[sel & f_ok].mean()) < 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(avg_queries()))
def test_avg_on_b200(name, host_batches):
    """Per-node entry points and the fused plan (AVG accumulates through a 64-bit CAS around the same
    rolling-average combine)."""
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    q = avg_queries()[name]
    exp = run_legacy(orc, q, host_batches)
    assert_same_avg(run_legacy(eng, q, host_batches), exp, f"{name}/legacy")
    assert_same_avg(run_fused(eng, q, host_batches), exp, f"{name}/fused")


# ---- column modes 0 / 1, bool columns, 8- and 16-byte dimension columns ----------------------------------
def _mixed_batch(be, seed, rows=30011):
    """request_at: mode 1 (no null vector); city: mode 0 (constant default for the whole batch);
    flag: bit-packed bool with nulls and a StartingIndex; fare: mode 2; id64: Int64; uuid: UUID (16 bytes)."""
    rng = np.random.default_rng(seed)
    ts = (synth.BASE_TS + rng.integers(0, 86400, rows)).astype(np.uint32)
    flag = rng.integers(0, 2, rows).astype(np.uint8)
    fare = (rng.integers(0, 6400, rows) / 64.0).astype(np.float32)
    id64 = rng.integers(-5, 5, rows).astype(np.int64) * (1 << 40)
    uuid = np.zeros((rows, 2), np.uint64)
    uuid[:, 0] = rng.integers(0, 3, rows).astype(np.uint64) * np.uint64(0x0123456789ABCDEF)
    uuid[:, 1] = rng.integers(0, 2, rows).astype(np.uint64) * np.uint64(0xFEDCBA9876543210)
    keep, cols = [], []
    for dt, v, ok, sb in ((A.Uint32, ts, None, 0), (None, None, None, 0), (A.Bool, flag, rng.random(rows) > 0.1, 3),
                          (A.Float32, fare, rng.random(rows) > 0.05, 0), (A.Int64, id64, rng.random(rows) > 0.05, 0),
                          (A.UUID, uuid, rng.random(rows) > 0.05, 0)):
        if dt is None:
            cols.append(columns.constant_column(A.Uint16, 7, True))
            continue
        buf, vp = columns.make_column(be.space, dt, v, valid=ok, start_bit=sb)
        cols.append(vp)
        keep.append(buf)
    return Batch(cols, rows, keep=keep)


def mixed_queries():
    ts, city, flag, fare = E.Col(0, A.Uint32, "ts"), E.Col(1, A.Uint16, "city"), E.Col(2, A.Bool, "flag"), E.Col(3, A.Float32, "fare")
    id64, uuid = E.Col(4, A.Int64, "id64"), E.Col(5, A.UUID, "uuid")
    return {
        "const_and_bool": AggQuery([flag], [city, E.floor(ts, E.Lit(7200)), flag], Measure("sum", fare)),
        "not_bool_filter": AggQuery([E.Unary(A.Not, flag)], [E.floor(ts, E.Lit(21600))], Measure("count")),
        "int64_dim": AggQuery([E.gt(fare, E.Lit(50.0))], [id64, flag], Measure("max", fare)),
        "uuid_dim": AggQuery([], [uuid, city], Measure("count")),
        "uuid_and_int64": AggQuery([E.Unary(A.IsNotNull, fare)], [uuid, id64, E.floor(ts, E.Lit(43200))], Measure("sum", fare)),
    }


@pytest.mark.parametrize("name", list(mixed_queries()))
def test_mixed_column_modes_oracle_vs_reference(name):
    orc = H.get_backend("oracle")
    q = mixed_queries()[name]

    def run(be):
        ex = LegacyBatchExecutor(be.lib, be.space, q)
        for seed in (1, 2):
            ex.process_batch(_mixed_batch(be, seed))
        return ex.result()
    exp = R.expected(run)
    assert exp["groups"] > 1
    R.assert_same_result(run(orc), exp, ctx=name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(mixed_queries()))
def test_mixed_column_modes_on_b200(name):
    """Mode-0 / mode-1 columns, bit-packed bool columns with a bit offset, and 8- / 16-byte dimension columns
    (read straight from global memory by the fused kernel) through both forms of the engine."""
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    q = mixed_queries()[name]
    exp_ex = LegacyBatchExecutor(orc.lib, orc.space, q)
    leg_ex, fus_ex = LegacyBatchExecutor(eng.lib, eng.space, q), FusedBatchExecutor(eng.lib, eng.space, q)
    for seed in (1, 2):
        exp_ex.process_batch(_mixed_batch(orc, seed))
        b = _mixed_batch(eng, seed)
        leg_ex.process_batch(b)
        fus_ex.process_batch(b)
    exp = exp_ex.result()
    assert_same_result(leg_ex.result(), exp, ctx=f"{name}/legacy")
    assert_same_result(fus_ex.result(), exp, ctx=f"{name}/fused")
    fus_ex.close()
