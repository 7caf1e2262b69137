/* abi_probe.c — prints size / field offsets of every by-value struct and the values of the ABI enums of the cgo boundary.
 * Compiled against the REFERENCE's own headers (-DUSE_REFERENCE -I<reference tree>: query/time_series_aggregate.h +
 * cgoutils/memory.h), its output is tests/golden/abi_layout_reference.txt; tests/test_abi_vs_reference_headers.py
 * compiles it against include/aresdb_b200/*.h and requires the same output.  It also LINKS this file against
 * aresdb_b200/lib/libalgorithm.so + libmem.so and calls entry points through the declared prototypes. */
#include <stddef.h>
#include <stdio.h>
#ifdef USE_REFERENCE
#include "query/time_series_aggregate.h"
#include "cgoutils/memory.h"
#else
#include "aresdb_b200/aql_abi.h"
#include "aresdb_b200/device_memory.h"
#endif

#define S(T) printf("sizeof %s %zu\n", #T, sizeof(T))
#define F(T, f) printf("offsetof %s.%s %zu\n", #T, #f, offsetof(T, f))
#define E(v) printf("enum %s %d\n", #v, (int)(v))

int main(int argc, char **argv) {
  S(CGoCallResHandle); F(CGoCallResHandle, res); F(CGoCallResHandle, pStrErr);
  S(RecordID); S(CuckooHashIndex); F(CuckooHashIndex, buckets); F(CuckooHashIndex, seeds); F(CuckooHashIndex, keyBytes);
  F(CuckooHashIndex, numHashes); F(CuckooHashIndex, numBuckets);
  S(GeoPointT); S(UUIDT); S(DefaultValue); F(DefaultValue, HasDefault); F(DefaultValue, Value);
  S(VectorPartySlice); F(VectorPartySlice, BasePtr); F(VectorPartySlice, NullsOffset); F(VectorPartySlice, ValuesOffset);
  F(VectorPartySlice, StartingIndex); F(VectorPartySlice, DataType); F(VectorPartySlice, DefaultValue); F(VectorPartySlice, Length);
  S(ScratchSpaceVector); F(ScratchSpaceVector, Values); F(ScratchSpaceVector, NullsOffset); F(ScratchSpaceVector, DataType);
  S(ConstantVector); F(ConstantVector, Value); F(ConstantVector, IsValid); F(ConstantVector, DataType);
  S(ForeignColumnVector); F(ForeignColumnVector, RecordIDs); F(ForeignColumnVector, Batches); F(ForeignColumnVector, BaseBatchID);
  F(ForeignColumnVector, NumBatches); F(ForeignColumnVector, NumRecordsInLastBatch); F(ForeignColumnVector, TimezoneLookup); F(ForeignColumnVector, TimezoneLookupSize);
  F(ForeignColumnVector, DataType); F(ForeignColumnVector, DefaultValue);
  S(ArrayVectorPartySlice); F(ArrayVectorPartySlice, OffsetLengthVector); F(ArrayVectorPartySlice, ValueOffsetAdj);
  F(ArrayVectorPartySlice, DataType); F(ArrayVectorPartySlice, Length); E(ArrayVectorPartyInput);
  S(InputVector); F(InputVector, Vector); F(InputVector, Type);
  S(DimensionVector); F(DimensionVector, DimValues); F(DimensionVector, HashValues); F(DimensionVector, IndexVector);
  F(DimensionVector, VectorCapacity); F(DimensionVector, NumDimsPerDimWidth);
  S(DimensionOutputVector); F(DimensionOutputVector, DimValues); F(DimensionOutputVector, DimNulls); F(DimensionOutputVector, DataType);
  S(MeasureOutputVector); F(MeasureOutputVector, Values); F(MeasureOutputVector, DataType); F(MeasureOutputVector, AggFunc);
  S(OutputVector); F(OutputVector, Vector); F(OutputVector, Type);
  S(GeoShapeBatch);
  E(NUM_DIM_WIDTH); E(MAX_DIMENSION_BYTES); E(HLL_BITS); E(HLL_DENSE_SIZE); E(HLL_DENSE_THRESHOLD);
  E(AGGR_SUM_UNSIGNED); E(AGGR_SUM_SIGNED); E(AGGR_SUM_FLOAT); E(AGGR_MIN_UNSIGNED); E(AGGR_MIN_SIGNED); E(AGGR_MIN_FLOAT);
  E(AGGR_MAX_UNSIGNED); E(AGGR_MAX_SIGNED); E(AGGR_MAX_FLOAT); E(AGGR_AVG_FLOAT); E(AGGR_HLL);
  E(Bool); E(Int8); E(Uint8); E(Int16); E(Uint16); E(Int32); E(Uint32); E(Float32); E(Int64); E(Uint64); E(GeoPoint); E(UUID); E(Float64);
  E(ConstInt); E(ConstFloat); E(ConstGeoPoint);
  E(Negate); E(Not); E(BitwiseNot); E(IsNull); E(IsNotNull); E(Noop); E(GetWeekStart); E(GetMonthStart); E(GetQuarterStart);
  E(GetYearStart); E(GetDayOfMonth); E(GetDayOfYear); E(GetMonthOfYear); E(GetQuarterOfYear); E(GetHLLValue);
  E(And); E(Or); E(Equal); E(NotEqual); E(LessThan); E(LessThanOrEqual); E(GreaterThan); E(GreaterThanOrEqual); E(Plus); E(Minus);
  E(Multiply); E(Divide); E(Mod); E(BitwiseAnd); E(BitwiseOr); E(BitwiseXor); E(Floor);
  E(VectorPartyInput); E(ScratchSpaceInput); E(ConstantInput); E(ForeignColumnInput);
  E(ScratchSpaceOutput); E(MeasureOutput); E(DimensionOutput);
  if (argc > 1) { /* link check: the prototypes come from whichever header set was compiled in */
    CGoCallResHandle h = GetDeviceCount();
    printf("link GetDeviceCount err=%d\n", h.pStrErr != NULL);
    printf("link GetFlags %u\n", (unsigned)GetFlags());
    /* only the addresses are taken: proves the symbols resolve with the reference's signatures */
    printf("link symbols %d\n", (int)((void *)InitIndexVector != NULL) + ((void *)UnaryTransform != NULL) + ((void *)BinaryFilter != NULL) +
           ((void *)Sort != NULL) + ((void *)Reduce != NULL) + ((void *)HashReduce != NULL) + ((void *)HyperLogLog != NULL) +
           ((void *)HashLookup != NULL) + ((void *)DeviceAllocate != NULL) + ((void *)AsyncCopyHostToDevice != NULL));
  }
  return 0;
}
