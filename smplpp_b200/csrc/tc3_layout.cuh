// Shared-memory / stage-image layout of K2''' (skin_tc3.cu), shared with K1 (forward.cu), which writes the per-call
// coefficient and transform stage images directly.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"
#include "skin_common.cuh"

namespace tc3
{
using namespace sb;
constexpr int MV = 128;                          // vertices per tile (UMMA M)
constexpr int NF = 96;                           // frames per block (UMMA N of GEMM 1)
constexpr int ROWB = 64;                         // bytes of K per shared-memory row (one SWIZZLE_64B span = 32 fp16)
constexpr int KP = kBlendK;                      // 224
constexpr int KUSED = kPoseDim + kShapeDim;      // 217: the template column is excluded
constexpr int NKB = KP * 2 / ROWB;               // 7 K-blocks of 32
constexpr int A_PART = 3 * MV * ROWB;            // 24576: one part (hi or lo) of the basis tile, 3 planes
constexpr int B_PART = NF * ROWB;                // 6144
constexpr int STAGE = 2 * A_PART + 2 * B_PART;   // 61440
constexpr int SUBF = 8;                          // frames per skinning sub-batch
constexpr int SUBN = SUBF * kXformFloats;        // 96 = UMMA N of GEMM 2
constexpr int KJ = skin::KJ;                     // joints padded to two K = 16 steps
constexpr int G_PART = SUBN * ROWB;              // 6144
constexpr int G_STAGE = 2 * G_PART;              // 12288
constexpr int NSUB = NF / SUBF;                  // 12 sub-batches per item
constexpr int EPI_WARPS = 16;
constexpr int EPI_FR = 2;                        // frames of a sub-batch handled by one epilogue warp
constexpr int FR_WARP = NSUB * EPI_FR;           // 24 frames of an item per epilogue warp
constexpr int CTRL_WARPS = 4;                     // one warpgroup: producer, MMA issuer, two idle
constexpr int THREADS = 32 * (CTRL_WARPS + EPI_WARPS);
// shared memory: [ST GEMM 1 stages][GS transform sub-batch slots][barriers]
template<int ST, int GS>
struct Layout
{
  static constexpr int OFF_G = ST * STAGE;
  static constexpr int OFF_BAR = OFF_G + GS * G_STAGE;
  static constexpr int SMEM_BYTES = 1024 + OFF_BAR + 512;
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};
constexpr int TMEM_COLS = 512;
constexpr int COL_M = 3 * NF;                    // 288
constexpr int COL_W = COL_M + 2 * SUBN;          // 480
constexpr int TRIPLES = NKB * 6;                 // GEMM 1 = 42 (K-block, product, K-step) triples of 3 MMAs (planes)
constexpr int COEF_EXP = 6, W_EXP = skin::W_EXP, G_EXP = skin::G_EXP;
static_assert(COL_W + 2 * (KJ / 2) == TMEM_COLS, "TMEM column map");
static_assert(STAGE % 1024 == 0 && G_STAGE % 1024 == 0, "swizzle atoms stay aligned");

// frame n of a 96-frame block -> row of the block in the fp16 coefficient operand (= accumulator column of GEMM 1):
// the 24 frames epilogue warp group fp owns (frame pair fp of every 8-frame sub-batch) become adjacent columns
__host__ __device__ constexpr int coef_row(int n)
{
  return ((n % SUBF) / EPI_FR) * FR_WARP + (n / SUBF) * EPI_FR + (n % EPI_FR);
}


// byte offset inside a 1024-byte aligned stage region -> SWIZZLE_64B position (16-byte chunk index XOR bits [7,9) of the
// offset: what a tiled TMA load with CU_TENSOR_MAP_SWIZZLE_64B writes and what the UMMA descriptor expects)
__host__ __device__ constexpr uint32_t swz64(uint32_t o)
{
  return o ^ (((o >> 7) & 3u) << 4);
}

// eight consecutive K values of one operand row -> fp16 hi | lo 16-byte chunks at their (swizzled) places
__device__ __forceinline__ void split8_store(const float (&x)[8], uint8_t * hi_dst, uint8_t * lo_dst)
{
  uint32_t h[4], l[4];
#pragma unroll
  for(int i = 0; i < 4; i++)
  {
    const float a = x[2 * i], b = x[2 * i + 1];
    const float ah = __half2float(__float2half_rn(a)), bh = __half2float(__float2half_rn(b));
    h[i] = skin::pack_half2(ah, bh);
    l[i] = skin::pack_half2(a - ah, b - bh);
  }
  *reinterpret_cast<uint4 *>(hi_dst) = make_uint4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<uint4 *>(lo_dst) = make_uint4(l[0], l[1], l[2], l[3]);
}

// byte offsets of the two per-call images inside the scratch area of tc3_frame_operand_bytes(batch)
inline size_t img_g_offset(int Bpad)
{
  return align_up(static_cast<size_t>(2) * Bpad * KP * sizeof(__half));
}
} // namespace tc3
