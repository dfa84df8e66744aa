// Pieces shared by the two kernels that compute the skinning matrices M[v,f] = sum_j W[v,j] G'[f,j] on tcgen05
// (skin_tc3.cu: fused with the blend contraction; lbs_tc.cu: standalone skinning): the fp16 hi | lo operand formats.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace sb
{
namespace skin
{
constexpr int KJ = 32;              // joints padded to two K = 16 steps
constexpr int W_EXP = 10, G_EXP = 4; // power-of-two pre-scales: lo = x - hi stays a normal fp16 (undone in the epilogue)

__device__ __forceinline__ uint32_t pack_half2(float lo16, float hi16)
{
  const __half2 h = __floats2half2_rn(lo16, hi16);
  return *reinterpret_cast<const uint32_t *>(&h);
}

// One vertex's row of the dense skinning weights (24 floats) -> the A operand of the skinning GEMM in TMEM: lane =
// vertex, 32 joints = 16 packed fp16x2 columns per part, hi at taddr, lo at taddr + 16.  The caller follows with
// tmem_st_wait + tcgen05.fence::before_thread_sync before signalling the MMA warp.
__device__ __forceinline__ void store_w_row_tmem(const float * __restrict__ wrow, uint32_t taddr)
{
  float w[KJ];
  const float4 * wp = reinterpret_cast<const float4 *>(wrow);
#pragma unroll
  for(int i = 0; i < kJoints / 4; i++)
  {
    const float4 t = __ldg(wp + i);
    w[4 * i] = t.x, w[4 * i + 1] = t.y, w[4 * i + 2] = t.z, w[4 * i + 3] = t.w;
  }
#pragma unroll
  for(int j = kJoints; j < KJ; j++) w[j] = 0.f;
  uint32_t hi[KJ / 2], lo[KJ / 2];
#pragma unroll
  for(int i = 0; i < KJ / 2; i++)
  {
    const float a = w[2 * i] * static_cast<float>(1 << W_EXP), b = w[2 * i + 1] * static_cast<float>(1 << W_EXP);
    const float ah = __half2float(__float2half_rn(a)), bh = __half2float(__float2half_rn(b));
    hi[i] = pack_half2(ah, bh);
    lo[i] = pack_half2(a - ah, b - bh);
  }
  ptx::tmem_st_x16(taddr, hi);
  ptx::tmem_st_x16(taddr + KJ / 2, lo);
}
} // namespace skin
} // namespace sb
