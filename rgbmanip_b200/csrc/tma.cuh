// Host side of the TMA tensor maps of the tcgen05 kernels (defined in tc_conv.cu).
#pragma once
#include "common.cuh"

namespace adp {

// Resolves the driver's cuTensorMapEncodeTiled once; every plan that encodes a tensor map calls it first.
int tma_init_driver();

// Tensor map over a densely packed tensor of `rank` dims (dims[0] innermost, esize bytes per element): the byte strides are
// the running products of the dims.  estr = nullptr: unit element strides.  Failures name `what` in adp_last_error.
int tma_encode(CUtensorMap* tm, CUtensorMapDataType dt, int rank, const void* ptr, const cuuint64_t* dims, int esize,
               const cuuint32_t* box, const cuuint32_t* estr, CUtensorMapSwizzle swizzle, CUtensorMapL2promotion l2,
               const char* what);

// element type of a 16-bit activation or weight plane
inline CUtensorMapDataType tma_type16(int f16) { return f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16; }

}  // namespace adp
