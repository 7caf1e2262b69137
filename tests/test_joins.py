"""Dimension-table joins (SURVEY.md §8 f4): HashLookup + ForeignColumnInput reads + timezone lookup through the per-node
C ABI (the reference's HOST build, the C restatement, the B200 engine) and through the fused ExecuteBatchPlan path.
Golden vectors: HashLookupTest.CheckLookup / CheckUUID (reference query/algorithm_unittest.cu:731-880) — cuckoo indexes
built by the reference's Go memstore."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

import harness as H
import reference_golden as R
from reference_golden import reference_results  # noqa: F401  (autouse fixture)
import test_pipeline_parity as T
from aresdb_b200 import cabi as A, columns, expr as E, joins as J, synth
from aresdb_b200.query import AggQuery, Join, Measure

BACKENDS = [pytest.param("ref", id="ref"), pytest.param("oracle", id="oracle"), pytest.param("b200", marks=pytest.mark.gpu, id="b200")]

GOLDEN = np.load(Path(__file__).parent / "golden" / "hash_lookup.npz")   # made by tests/golden/make_hash_lookup_fixture.py


def _hash_index(be, raw, seeds, key_bytes, num_hashes, num_buckets):
    buf = be.put(np.asarray(raw, np.uint8))
    h = A.CuckooHashIndex()
    h.buckets = buf.ptr
    for i in range(4):
        h.seeds[i] = seeds[i]
    h.keyBytes, h.numHashes, h.numBuckets = key_bytes, num_hashes, num_buckets
    return h, buf


@pytest.mark.parametrize("backend", BACKENDS)
def test_hash_lookup_golden_check_lookup(backend):
    be = H.get_backend(backend)
    kb, nh, nb = GOLDEN["lookup_params"].tolist()
    assert GOLDEN["lookup_buckets"].size == 312
    h, keep = _hash_index(be, GOLDEN["lookup_buckets"], GOLDEN["lookup_seeds"].tolist(), kb, nh, nb)
    n = 18
    buf, vp = columns.make_column(be.space, A.Int32, np.arange(n, dtype=np.int32), valid=np.ones(n, np.uint8))
    idx = be.put(np.arange(n, dtype=np.uint32))
    out = be.zeros(8 * n)
    be.lib.HashLookup(A.vp_input(vp), out.ptr, idx.ptr, n, None, 0, h, be.space.stream, be.device)
    got = out.get(np.uint32, 2 * n).reshape(n, 2)
    assert got[:, 0].tolist() == [0] * n and got[:, 1].tolist() == list(range(n))   # RecordID {0, i}


@pytest.mark.parametrize("backend", BACKENDS)
def test_hash_lookup_golden_check_uuid(backend):
    """HashLookupTest.CheckUUID: 16-byte keys {0,0}, {1,0}, {2,0}."""
    be = H.get_backend(backend)
    kb, nh, nb = GOLDEN["uuid_params"].tolist()
    h, keep = _hash_index(be, GOLDEN["uuid_buckets"], GOLDEN["uuid_seeds"].tolist(), kb, nh, nb)
    n = 3
    vals = np.zeros((n, 2), np.uint64)
    vals[:, 0] = np.arange(n)
    buf, vp = columns.make_column(be.space, A.UUID, vals.reshape(-1), valid=np.ones(n, np.uint8))
    vp.Length = n
    idx = be.put(np.arange(n, dtype=np.uint32))
    out = be.zeros(8 * n)
    be.lib.HashLookup(A.vp_input(vp), out.ptr, idx.ptr, n, None, 0, h, be.space.stream, be.device)
    got = out.get(np.uint32, 2 * n).reshape(n, 2)
    assert got[:, 0].tolist() == [0] * n and got[:, 1].tolist() == list(range(n))


def _dimension_table(be, n_cities=60, rows_per_batch=25, seed=3):
    rng = np.random.default_rng(seed)
    city = rng.permutation(np.arange(1, n_cities + 1)).astype(np.uint16)        # primary key
    region = rng.integers(0, 7, n_cities).astype(np.uint8)
    tz_enum = rng.integers(0, 12, n_cities).astype(np.uint8)                     # enum -> timezone offset table
    surge = (rng.integers(0, 40, n_cities) / 8.0).astype(np.float32)
    valid = [None, (rng.random(n_cities) > 0.1).astype(np.uint8), (rng.random(n_cities) > 0.1).astype(np.uint8), None]
    types = [A.Uint16, A.Uint8, A.Uint8, A.Float32]
    table = J.DimensionTable.build(be.space, types, [city, region, tz_enum, surge], valid, pk_column=0, rows_per_batch=rows_per_batch)
    return table, dict(city=city, region=region, tz=tz_enum, surge=surge, valid=valid)


@pytest.mark.parametrize("backend", BACKENDS)
def test_hash_lookup_built_index_finds_every_key_and_rejects_the_rest(backend):
    be = H.get_backend(backend)
    table, data = _dimension_table(be)
    keys = np.concatenate([data["city"], np.array([0, 61, 999, 65535], np.uint16)]).astype(np.uint16)
    valid = np.ones(len(keys), np.uint8)
    valid[5] = 0
    buf, vp = columns.make_column(be.space, A.Uint16, keys, valid=valid)
    idx = be.put(np.arange(len(keys), dtype=np.uint32))
    out = be.zeros(8 * len(keys))
    be.lib.HashLookup(A.vp_input(vp), out.ptr, idx.ptr, len(keys), None, 0, table.hash_index(), be.space.stream, be.device)
    got = out.get(np.uint8, 8 * len(keys)).reshape(-1, 8)
    batch = got[:, :4].copy().view(np.int32).reshape(-1)
    row = got[:, 4:].copy().view(np.uint32).reshape(-1)
    for i in range(60):
        if i == 5:
            assert (batch[i], row[i]) == (0, 0)          # NULL key
        else:
            assert (batch[i], row[i]) == (J.BASE_BATCH_ID + i // 25, i % 25)
    assert batch[60:].tolist() == [0] * 4 and row[60:].tolist() == [0] * 4


def join_queries(table, tz_ptr, tz_size):
    TS, CITY, STATUS, FARE = T.TS, T.CITY, T.STATUS, T.FARE
    REGION = E.ForeignCol(0, 1, A.Uint8, "region")
    TZ = E.ForeignCol(0, 2, A.Uint8, "tz", timezone=True)
    SURGE = E.ForeignCol(0, 3, A.Float32, "surge")
    j = [Join(table, CITY, tz_ptr, tz_size)]
    return {
        # group by a dimension-table column, filter on another one
        "by_region": AggQuery([E.eq(STATUS, E.Lit(1)), E.gt(SURGE, E.Lit(1.0))], [REGION, E.floor(TS, E.Lit(3600))],
                              Measure("sum", FARE), joins=j),
        # time bucket in the city's local time: request_at + tz offset of the joined city (the timezone table)
        "local_hour": AggQuery([E.ne(CITY, E.Lit(0))], [E.floor(E.add(TS, TZ), E.Lit(3600))], Measure("count"), joins=j),
        # measure from the dimension table, unmatched rows (NULL surge) contribute the identity
        "sum_surge": AggQuery([], [STATUS], Measure("sum", SURGE), joins=j),
        "unmatched": AggQuery([E.Unary(A.IsNull, REGION)], [CITY], Measure("count"), joins=j),
    }


def _tz_table(be):
    tz = (np.arange(12, dtype=np.int16) - 5) * 1800      # half-hour steps, some negative
    buf = be.put(tz)
    return buf, len(tz)


@pytest.fixture(scope="module")
def host_batches():
    # cities 1..80: 61..80 are NOT in the dimension table (unmatched rows)
    return [synth.generate_batch(d, n, num_cities=80, null_rate=0.03) for d, n in ((0, 20000), (1, 7777))]


@pytest.mark.parametrize("name", ["by_region", "local_hour", "sum_surge", "unmatched"])
def test_join_sequence_oracle_vs_reference(name, host_batches):
    def run(be):
        table, _ = _dimension_table(be)
        tzb, tzn = _tz_table(be)
        return T.run_legacy(be, join_queries(table, tzb.ptr, tzn)[name], host_batches)
    exp = R.expected(run)
    assert exp["groups"] > 0
    R.assert_same_result(run(H.get_backend("oracle")), exp, ctx=name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["by_region", "local_hour", "sum_surge", "unmatched"])
def test_join_sequence_on_b200(name, host_batches):
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    res = []
    for be in (orc, eng):
        table, _ = _dimension_table(be)
        tzb, tzn = _tz_table(be)
        res.append(T.run_legacy(be, join_queries(table, tzb.ptr, tzn)[name], host_batches))
    T.assert_same_result(res[1], res[0], ctx=name)


@pytest.mark.gpu
@pytest.mark.parametrize("jit", ["1", "0"])
@pytest.mark.parametrize("name", ["by_region", "local_hour", "sum_surge", "unmatched"])
def test_fused_join_on_b200(name, jit, host_batches, monkeypatch):
    """ExecuteBatchPlan with joined tables (the lookup is a gather stage of the fused kernel; jit=0: the interpreter
    kernel — the switch is read once per process, so that variant runs in a child) == the reference call sequence."""
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    if jit == "0":
        import os
        import subprocess
        import sys
        code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
                "import test_joins as TJ, harness as H, test_pipeline_parity as T\n"
                "from aresdb_b200 import synth\n"
                "hbs = [synth.generate_batch(d, n, num_cities=80, null_rate=0.03) for d, n in ((0, 20000), (1, 7777))]\n"
                "TJ._fused_vs_oracle(%r, hbs)\nprint('ok')\n") % (str(Path(__file__).parent), str(Path(__file__).parent.parent), name)
        r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, ARESDB_B200_JIT="0"), capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout[-1500:] + r.stderr[-3000:]
        return
    _fused_vs_oracle(name, host_batches)


def _fused_vs_oracle(name, host_batches):
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    otable, _ = _dimension_table(orc)
    otz, tzn = _tz_table(orc)
    exp = T.run_legacy(orc, join_queries(otable, otz.ptr, tzn)[name], host_batches)
    etable, _ = _dimension_table(eng)
    etz, _ = _tz_table(eng)
    got = T.run_fused(eng, join_queries(etable, etz.ptr, tzn)[name], host_batches)
    T.assert_same_result(got, exp, ctx=name)
