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
constexpr int KW = 16;                           // joint slots per window (one K = 16 step of GEMM 2)
constexpr int NWIN = 2;                          // joint windows per model
constexpr int KJ = NWIN * KW;                    // 32 slots per transform row
constexpr int ROWG = KW * 2;                     // bytes of one window's row (one SWIZZLE_32B span = 16 fp16)
constexpr int G_PART = SUBN * ROWG;              // 3072: one part (hi or lo) of one window of a sub-batch
constexpr int G_WIN = 2 * G_PART;                // 6144: one window of a sub-batch = one transform ring slot
constexpr int G_SUB = NWIN * G_WIN;              // 12288: one sub-batch of the transform image
constexpr int NSUB = NF / SUBF;                  // 12 sub-batches per item
constexpr int EPI_WARPS = 16;
constexpr int EPI_FR = 2;                        // frames of a sub-batch handled by one epilogue warp
constexpr int FR_WARP = NSUB * EPI_FR;           // 24 frames of an item per epilogue warp
constexpr int CTRL_WARPS = 4;                     // one warpgroup: producer, MMA issuer, two idle
constexpr int THREADS = 32 * (CTRL_WARPS + EPI_WARPS);
// shared memory: [ST GEMM 1 stages][GS transform window slots][barriers]
template<int ST, int GS>
struct Layout
{
  static constexpr int OFF_G = ST * STAGE;
  static constexpr int OFF_BAR = OFF_G + GS * G_WIN;
  static constexpr int SMEM_BYTES = 1024 + OFF_BAR + 512;
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};
constexpr int TMEM_COLS = 512;
constexpr int COL_M = 3 * NF;                    // 288
constexpr int COL_W = COL_M + 2 * SUBN;          // 480
constexpr int TRIPLES = NKB * 6;                 // GEMM 1 = 42 (K-block, product, K-step) triples of 3 MMAs (planes)
constexpr int COEF_EXP = 6, W_EXP = skin::W_EXP, G_EXP = skin::G_EXP;
static_assert(COL_W + NWIN * KW == TMEM_COLS, "TMEM column map: window w at COL_W + 16 w (8 hi | 8 lo columns)");
static_assert(STAGE % 1024 == 0 && G_WIN % 1024 == 0 && G_PART % 256 == 0, "swizzle atoms stay aligned");

// The two joint windows of a model (chosen by tc3_prepare_model from its skinning weights): slot s of the transform
// image belongs to window s / KW and holds joint[s], or zeros for -1.  A joint may sit in both windows.
struct WindowMap
{
  int8_t joint[KJ];
};
// joints of slots 8 c .. 8 c + 7 for a run-time c (0..3): selects between constant indices, so that the map (a kernel
// parameter) is not copied to local memory
__device__ __forceinline__ void chunk_joints(const WindowMap & m, int c, int (&j)[8])
{
#pragma unroll
  for(int jj = 0; jj < 8; jj++)
  {
    j[jj] = m.joint[jj];
#pragma unroll
    for(int q = 1; q < KJ / 8; q++) j[jj] = c == q ? m.joint[8 * q + jj] : j[jj];
  }
}
static_assert(sizeof(ModelDev::tc3_slot_joint) == KJ, "slot map of the model");
inline WindowMap window_map(const ModelDev & d)
{
  WindowMap m;
  for(int s = 0; s < KJ; s++) m.joint[s] = d.tc3_slot_joint[s];
  return m;
}

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
// the same for SWIZZLE_32B (16-byte chunk index XOR bit 7 of the offset), inside a 256-byte aligned region
__host__ __device__ constexpr uint32_t swz32(uint32_t o)
{
  return o ^ (((o >> 7) & 1u) << 4);
}

// transform image [frame block][sub-batch][window][hi | lo][96 rows][16 slots], SWIZZLE_32B: byte offset of the hi
// 16-byte chunk with slots 8 c .. 8 c + 7 (c = 0..3, window c / 2) of element e (0..11) of frame f; lo is G_PART further
__host__ __device__ inline size_t g_chunk_offset(long long f, int e, int c)
{
  const long long fb = f / NF;
  const int nf = static_cast<int>(f - fb * NF);
  const size_t blk = ((static_cast<size_t>(fb) * NSUB + nf / SUBF) * NWIN + c / 2) * G_WIN;
  return blk + swz32(static_cast<uint32_t>(((nf % SUBF) * kXformFloats + e) * ROWG + (c % 2) * 16));
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
