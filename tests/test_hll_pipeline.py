"""HyperLogLog queries through the whole per-batch call sequence (reference
query/aql_batchexecutor.go:219-233 -> query/hll.cu:262-290): several batches with carried
(key, value) rows, register vectors built on the last batch.

Byte-exact: the dimension rows in output order, the per-group register counts and the sparse /
dense register vector.  The reference's HOST build is the expectation on the CPU; on the GPU the
C restatement is switched to the DEVICE build's shift semantics (oracle/aql_oracle.c:297-305:
`1 << (rho + 14)` is an int shift — x86 wraps the count, the GPU yields 0), which is what the
engine implements.
"""
import ctypes as C

import numpy as np
import pytest

import harness as H
import reference_golden as R
from reference_golden import reference_results  # noqa: F401  (autouse fixture)
from aresdb_b200 import cabi as A
from aresdb_b200 import columns, expr as E, synth
from aresdb_b200.executor import Batch, LegacyBatchExecutor
from aresdb_b200.query import AggQuery, Measure
from test_pipeline_parity import CITY, FARE, STATUS, TS, upload


def hll_queries():
    return {
        # ~50 groups x a few hundred registers each: every group stays sparse
        "sparse_by_city": AggQuery([E.eq(STATUS, E.Lit(1))], [CITY], Measure("countdistincthll", TS)),
        # 4 groups x thousands of registers: dense vectors (>= 4096 registers) next to sparse ones
        "dense_by_status": AggQuery([], [STATUS], Measure("countdistincthll", TS)),
        # two dims (4-byte bucket + 1-byte enum), hashed column narrower than 4 bytes
        "two_dims": AggQuery([E.gt(FARE, E.Lit(10.0))], [E.floor(TS, E.Lit(86400)), STATUS],
                             Measure("countdistincthll", CITY)),
    }


BATCHES = [(0, 20000), (1, 7001), (2, 26000)]


@pytest.fixture(scope="module")
def host_batches():
    return [synth.generate_batch(day, rows, num_cities=50, null_rate=0.02) for day, rows in BATCHES]


def run_hll_query(be, q, host_batches):
    ex = LegacyBatchExecutor(be.lib, be.space, q)
    for i, hb in enumerate(host_batches):
        ex.process_batch(upload(be, hb), is_last=i == len(host_batches) - 1)
    return ex.hll


def assert_same_hll(got, exp, ctx=""):
    assert got.groups == exp.groups, f"{ctx}: {got.groups} groups vs {exp.groups}"
    assert got.dims.rows == exp.dims.rows, f"{ctx}: dimension rows / order differ"
    assert got.counts.tolist() == exp.counts.tolist(), f"{ctx}: register counts differ"
    assert got.regs.tobytes() == exp.regs.tobytes(), f"{ctx}: register vector differs"


def set_oracle_device_semantics(on: bool):
    orc = H.get_backend("oracle")
    fn = orc.lib.alg.OracleSetDeviceSemantics
    fn.argtypes, fn.restype = [C.c_int], None
    fn(1 if on else 0)


def hll_summary(r) -> dict:
    """What assert_same_hll compares, plus the sizes the test asserts on."""
    return {"groups": r.groups, "rows": r.dims.packed_rows(), "counts": r.counts, "regs": r.regs,
            "dense_groups": int((r.counts >= 4096).sum()), "regs_size": int(r.regs.size)}


@pytest.mark.parametrize("name", list(hll_queries()))
def test_hll_sequence_oracle_vs_reference(name, host_batches):
    orc = H.get_backend("oracle")
    set_oracle_device_semantics(False)
    q = hll_queries()[name]
    exp = R.expected(lambda ref: hll_summary(run_hll_query(ref, q, host_batches)))
    got = run_hll_query(orc, q, host_batches)
    assert exp["groups"] > 0
    if name == "dense_by_status":
        assert exp["dense_groups"] > 0 and exp["regs_size"] >= 16384
    R.assert_same(hll_summary(got), exp, name)
    # the decoded registers are consistent with the counts
    for dense, c in zip(got.dense_registers().values(), got.counts):
        assert int((dense != 0).sum()) == int(c)


def test_hll_single_batch_equals_three_batches(host_batches):
    """Carrying (key, value) rows across batches does not change the registers."""
    orc = H.get_backend("oracle")
    set_oracle_device_semantics(False)
    q = hll_queries()["two_dims"]
    three = run_hll_query(orc, q, host_batches)
    merged = synth.HostBatch([np.concatenate([hb.values[c] for hb in host_batches]) for c in range(4)],
                             [np.concatenate([hb.valid[c] for hb in host_batches]) for c in range(4)],
                             sum(hb.num_rows for hb in host_batches), 0)
    one = run_hll_query(orc, q, [merged])
    assert one.dense_registers().keys() == three.dense_registers().keys()
    for k, v in one.dense_registers().items():
        assert v.tobytes() == three.dense_registers()[k].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(hll_queries()))
def test_hll_sequence_on_b200(name, host_batches):
    eng, orc = H.get_backend("b200"), H.get_backend("oracle")
    q = hll_queries()[name]
    set_oracle_device_semantics(True)
    try:
        exp = run_hll_query(orc, q, host_batches)
    finally:
        set_oracle_device_semantics(False)
    got = run_hll_query(eng, q, host_batches)
    assert_same_hll(got, exp, name)


def _hll_values(be, values: np.ndarray) -> np.ndarray:
    """GetHLLValue over a uint32 column through UnaryTransform into a scratch vector."""
    n = values.size
    buf, vp = columns.make_column(be.space, A.Uint32, values)
    out = be.zeros(5 * n)
    idx = be.put(np.arange(n, dtype=np.uint32))
    be.lib.UnaryTransform(A.vp_input(vp), A.scratch_output(out.ptr, 4 * n, A.Uint32), idx.ptr, n, None, 0,
                          A.GetHLLValue, be.space.stream, be.device)
    return out.get(np.uint32, n)


def _long_rho_inputs():
    """uint32 inputs whose 64-bit hash has bits 14..31 clear, i.e. rho >= 18: the two builds of the
    reference disagree on exactly these (found by scanning with the C restatement)."""
    orc = H.get_backend("oracle")
    vals = np.arange(1, 3_000_001, dtype=np.uint32)
    set_oracle_device_semantics(False)
    host = _hll_values(orc, vals)
    set_oracle_device_semantics(True)
    dev = _hll_values(orc, vals)
    set_oracle_device_semantics(False)
    differ = np.nonzero(host != dev)[0]
    return vals[differ], host[differ], dev[differ]


def test_hll_value_host_shift_semantics_match_reference():
    vals, host, dev = _long_rho_inputs()
    assert vals.size >= 3, "expected ~11 inputs with rho >= 18 among 3e6"
    assert (host >> 16 >= 18).all() and (dev >> 16 >= 18).all()
    R.assert_same(host, R.expected(lambda ref: _hll_values(ref, vals)), "GetHLLValue, rho >= 18")


@pytest.mark.gpu
def test_hll_value_device_shift_semantics_on_b200():
    eng = H.get_backend("b200")
    vals, host, dev = _long_rho_inputs()
    assert vals.size >= 3
    assert _hll_values(eng, vals).tolist() == dev.tolist()


# ---- the fused path: ExecuteBatchPlan into an AGGR_HLL state, AggStateFinalizeHLL --------------------
ENTRY_MODE, DENSE_MODE = 100000, 0   # AggSpec.ExpectedGroups: > 4096 -> (group, register) entries; else dense registers


def run_hll_fused(be, q, host_batches, expected_groups=DENSE_MODE):
    from aresdb_b200.executor import FusedBatchExecutor
    ex = FusedBatchExecutor(be.lib, be.space, q, expected_groups)
    keep = []
    for hb in host_batches:
        b = upload(be, hb)
        keep.append(b)
        ex.process_batch(b)
    r = ex.hll_result()
    ex.close()
    return r


def _device_oracle(q, host_batches):
    orc = H.get_backend("oracle")
    set_oracle_device_semantics(True)
    try:
        return run_hll_query(orc, q, host_batches)
    finally:
        set_oracle_device_semantics(False)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [ENTRY_MODE, DENSE_MODE], ids=["entries", "dense"])
@pytest.mark.parametrize("name", list(hll_queries()))
def test_hll_fused_plan_on_b200(name, mode, host_batches):
    """One fused kernel per batch + AggStateFinalizeHLL == the reference's per-batch HyperLogLog
    sequence, byte for byte (dims, order, register counts, sparse/dense vectors), in both table modes."""
    eng = H.get_backend("b200")
    q = hll_queries()[name]
    assert_same_hll(run_hll_fused(eng, q, host_batches, mode), _device_oracle(q, host_batches), f"{name}/{mode}")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [ENTRY_MODE, DENSE_MODE], ids=["entries", "dense"])
def test_hll_fused_states_merge_through_carried_rows(mode, host_batches):
    """Two HLL states (two GPUs' worth of batches) combine through AggStateFinalize (carried rows:
    one per (group, register) entry) + AggStateMerge — the multi-GPU exchange step for hll queries."""
    from aresdb_b200.executor import FusedBatchExecutor, _ResultBuffers
    eng = H.get_backend("b200")
    q = hll_queries()["two_dims"]
    a, b = FusedBatchExecutor(eng.lib, eng.space, q, mode), FusedBatchExecutor(eng.lib, eng.space, q, mode)
    keep = [upload(eng, hb) for hb in host_batches]
    a.process_batch(keep[0])
    a.process_batch(keep[1])
    b.process_batch(keep[2])
    n, carried = b.finalize_into()
    assert n == b.group_count() and n > 0
    values = carried.measures.get(np.uint32, n)
    assert (np.diff(carried.hash.get(np.uint64, n).astype(np.uint64)) > 0).all()      # key-ascending, one row per key
    assert ((carried.hash.get(np.uint64, n) & 0x3FFF) == (values & 0x3FFF)).all()    # key carries the register
    a.merge(carried.dimension_vector(q), carried.measures.ptr, n)
    assert_same_hll(a.hll_result(), _device_oracle(q, host_batches), "merged")
    a.close()
    b.close()


@pytest.mark.gpu
def test_hll_fused_empty_result():
    eng = H.get_backend("b200")
    q = AggQuery([E.eq(STATUS, E.Lit(99))], [CITY], Measure("countdistincthll", TS))
    r = run_hll_fused(eng, q, [synth.generate_batch(0, 5000)])
    assert r.groups == 0 and r.regs.size == 0
