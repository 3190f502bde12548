// Block-wide (value, index) selection shared by the beam-search step (decode.cu) and the row top-k (classify.cu).
#pragma once
#include "vtx_common.cuh"

namespace vtx {

// Selection order, the argmax rule of vtx_argmax_rows: NaN ranks above every number, then larger value, then lower
// index (also among NaNs).
__device__ __forceinline__ bool rank_better(float v, int i, float bv, int bi) {
  const bool vn = isnan(v), bn = isnan(bv);
  if (vn != bn) return vn;
  return v > bv || ((v == bv || vn) && i < bi);
}

// Block-wide best (value, index) of one offer per thread; every thread gets the winner.  sv / si: 32 shared slots.
__device__ __forceinline__ void block_best(float& v, int& i, float* sv, int* si) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int oi = __shfl_xor_sync(0xffffffffu, i, o);
    if (rank_better(ov, oi, v, i)) { v = ov; i = oi; }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();  // sv / si may still be read from the previous call
  if (lane == 0) { sv[warp] = v; si[warp] = i; }
  __syncthreads();
  v = lane < nw ? sv[lane] : -INFINITY;
  i = lane < nw ? si[lane] : 0x7fffffff;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int oi = __shfl_xor_sync(0xffffffffu, i, o);
    if (rank_better(ov, oi, v, i)) { v = ov; i = oi; }
  }
}

}  // namespace vtx
