// SMPL forward pass on sm_100a: pose features + kinematic chain (K1), fused blend-shape contraction +
// linear blend skinning (K2, FFMA variant), standalone skinning (K3) and the generic per-module kernels.
//
// Reference semantics (file:line in the reference tree):
//   rodrigues           src/BlendShape.cpp:803-844     (a = ||theta + 1e-8||, u = theta / a)
//   pose feature        src/BlendShape.cpp:865-928     (vec(R_1..R_23) - vec(I))
//   pose / shape blend  src/BlendShape.cpp:764, 670-683
//   rest shape, joints  src/JointRegression.cpp:551-598 (joints exclude the pose blend)
//   kinematic chain     src/WorldTransformation.cpp:508-677
//   skinning            src/LinearBlendSkinning.cpp:445-553 (homogeneous divide kept, root translation added)
#include "common.cuh"
#include "forward.cuh"
#include "ik2.cuh"
#include "ik_poseblend.cuh"
#include "ik_solve.cuh"
#include "tc3_layout.cuh"
#include "vposer.cuh"

using namespace sb;

namespace sb
{
std::atomic<int> g_forward_variant{0};
std::atomic<int> g_lbs_variant{2};
}

// ------------------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------------------

// BlendShape::rodrigues for one joint.  R row-major.
__device__ __forceinline__ void rodrigues3(float x, float y, float z, float * R)
{
  const float eps = 1e-8f;
  float ax = x + eps, ay = y + eps, az = z + eps;
  float a = sqrtf(ax * ax + ay * ay + az * az);
  float ux = x / a, uy = y / a, uz = z / a;
  float s, c;
  sincosf(a, &s, &c);
  float oc = 1.f - c;
  // K = [u]x ; K^2 computed entry-wise exactly as matmul(skew, skew)
  R[0] = 1.f + oc * (-(uz * uz) - uy * uy);
  R[1] = s * (-uz) + oc * (uy * ux);
  R[2] = s * uy + oc * (uz * ux);
  R[3] = s * uz + oc * (ux * uy);
  R[4] = 1.f + oc * (-(uz * uz) - ux * ux);
  R[5] = s * (-ux) + oc * (uz * uy);
  R[6] = s * (-uy) + oc * (ux * uz);
  R[7] = s * ux + oc * (uy * uz);
  R[8] = 1.f + oc * (-(uy * uy) - ux * ux);
}

// ------------------------------------------------------------------------------------------------------------
// K1: pose features + joints + kinematic chain.  One warp per frame, lane j = joint j (24 of 32 lanes).
// ------------------------------------------------------------------------------------------------------------
constexpr int kChainWarps = 8;

__global__ void __launch_bounds__(kChainWarps * 32)
    pose_chain_kernel(ChainTopo topo, const float * __restrict__ joint_template,
                      const float * __restrict__ joint_shape, int B, const float * __restrict__ beta,
                      long long beta_stride, const float * __restrict__ theta, float * __restrict__ coef,
                      float * __restrict__ xforms, float * __restrict__ joints_out, float * __restrict__ xforms44_out,
                      uint8_t * __restrict__ img_b, uint8_t * __restrict__ img_g, int Bpad, tc3::WindowMap wmap)
{
  __shared__ float sG[kChainWarps][kJoints][12];
  __shared__ float sJ[kChainWarps][kJoints][3];
  __shared__ float sC[kChainWarps][kBlendK];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long b = static_cast<long long>(blockIdx.x) * kChainWarps + warp;
  if(b >= B)
  {
    // padding frames of the last 96-frame block: their rows of the K2''' stage images are zero
    if(img_b && b < Bpad)
    {
      const long long fb = b / tc3::NF;
      const int nf = static_cast<int>(b - fb * tc3::NF);
      const uint4 z = make_uint4(0u, 0u, 0u, 0u);
      if(lane < tc3::KP / 8)
      {
        uint8_t * blk = img_b + (static_cast<size_t>(fb) * tc3::NKB + lane / 4) * (2 * tc3::B_PART);
        const uint32_t o = static_cast<uint32_t>(tc3::coef_row(nf) * tc3::ROWB + (lane % 4) * 16);
        *reinterpret_cast<uint4 *>(blk + tc3::swz64(o)) = z;
        *reinterpret_cast<uint4 *>(blk + tc3::swz64(tc3::B_PART + o)) = z;
      }
      for(int c = lane; c < kXformFloats * 4; c += 32)
      {
        uint8_t * dst = img_g + tc3::g_chunk_offset(b, c / 4, c % 4);
        *reinterpret_cast<uint4 *>(dst) = z;
        *reinterpret_cast<uint4 *>(dst + tc3::G_PART) = z;
      }
    }
    return; // whole warp leaves together; only __syncwarp below
  }

  const float * bp = beta + b * beta_stride;
  float R[9], Jt[3] = {0.f, 0.f, 0.f}, t[3];
  if(lane < kJoints)
  {
    const float * th = theta + (b * (kJoints + 1) + 1 + lane) * 3;
    rodrigues3(th[0], th[1], th[2], R);
#pragma unroll
    for(int k = 0; k < 3; k++)
    {
      float acc = joint_template[lane * 3 + k];
#pragma unroll
      for(int i = 0; i < kShapeDim; i++) acc = fmaf(joint_shape[(lane * 3 + k) * kShapeDim + i], bp[i], acc);
      Jt[k] = acc;
      sJ[warp][lane][k] = acc;
    }
  }
  __syncwarp();
  const int parent = lane < kJoints ? topo.parent[lane] : -1;
  const int depth = lane < kJoints ? topo.depth[lane] : -1;
  if(lane < kJoints)
  {
#pragma unroll
    for(int k = 0; k < 3; k++) t[k] = parent >= 0 ? Jt[k] - sJ[warp][parent][k] : Jt[k];
  }
  // global transforms, level by level (parents always precede: WorldTransformation.cpp:583-610)
  float G[12];
  for(int d = 0; d <= topo.max_depth; d++)
  {
    if(depth == d)
    {
      if(parent < 0)
      {
#pragma unroll
        for(int r = 0; r < 3; r++)
        {
          G[4 * r + 0] = R[3 * r + 0];
          G[4 * r + 1] = R[3 * r + 1];
          G[4 * r + 2] = R[3 * r + 2];
          G[4 * r + 3] = t[r];
        }
      }
      else
      {
        const float * P = sG[warp][parent];
#pragma unroll
        for(int r = 0; r < 3; r++)
        {
          float p0 = P[4 * r + 0], p1 = P[4 * r + 1], p2 = P[4 * r + 2], p3 = P[4 * r + 3];
#pragma unroll
          for(int c = 0; c < 3; c++) G[4 * r + c] = p0 * R[c] + p1 * R[3 + c] + p2 * R[6 + c];
          G[4 * r + 3] = p0 * t[0] + p1 * t[1] + p2 * t[2] + p3;
        }
      }
#pragma unroll
      for(int e = 0; e < 12; e++) sG[warp][lane][e] = G[e];
    }
    __syncwarp();
  }
  if(lane < kJoints)
  {
    // relativeTransform (WorldTransformation.cpp:657-677): t' = tg - Rg * Jt
#pragma unroll
    for(int r = 0; r < 3; r++) G[4 * r + 3] -= G[4 * r + 0] * Jt[0] + G[4 * r + 1] * Jt[1] + G[4 * r + 2] * Jt[2];
    if(xforms)
    {
      float4 * dst = reinterpret_cast<float4 *>(xforms + (b * kJoints + lane) * 12);
      dst[0] = make_float4(G[0], G[1], G[2], G[3]);
      dst[1] = make_float4(G[4], G[5], G[6], G[7]);
      dst[2] = make_float4(G[8], G[9], G[10], G[11]);
    }
    if(xforms44_out)
    {
      float4 * dst = reinterpret_cast<float4 *>(xforms44_out + (b * kJoints + lane) * 16);
      dst[0] = make_float4(G[0], G[1], G[2], G[3]);
      dst[1] = make_float4(G[4], G[5], G[6], G[7]);
      dst[2] = make_float4(G[8], G[9], G[10], G[11]);
      dst[3] = make_float4(0.f, 0.f, 0.f, 1.f);
    }
    if(joints_out)
    {
#pragma unroll
      for(int k = 0; k < 3; k++) joints_out[(b * kJoints + lane) * 3 + k] = Jt[k];
    }
  }
  if(img_g)
  {
    // transform stage image of K2''' (tc3::g_chunk_offset: row = frame in its 8-frame sub-batch * 12 + element, two
    // 16-slot joint windows, fp16 hi | lo x 2^4, SWIZZLE_32B): the relative transforms go back to shared memory and
    // every lane writes 16-byte chunks (8 slots of one element); this replaces a separate pass over the fp32 transforms
    __syncwarp();
    if(lane < kJoints)
    {
#pragma unroll
      for(int e = 0; e < 12; e++) sG[warp][lane][e] = G[e];
    }
    __syncwarp();
    for(int c = lane; c < kXformFloats * 4; c += 32)
    {
      const int e = c / 4, cj = c % 4;
      float x[8];
      int js[8];
      tc3::chunk_joints(wmap, cj, js);
#pragma unroll
      for(int jj = 0; jj < 8; jj++)
        x[jj] = js[jj] >= 0 ? sG[warp][js[jj] < 0 ? 0 : js[jj]][e] * static_cast<float>(1 << tc3::G_EXP) : 0.f;
      uint8_t * dst = img_g + tc3::g_chunk_offset(b, e, cj);
      tc3::split8_store(x, dst, dst + tc3::G_PART);
    }
  }
  if(coef)
  {
    if(lane >= 1 && lane < kJoints)
    {
#pragma unroll
      for(int e = 0; e < 9; e++) sC[warp][9 * (lane - 1) + e] = R[e] - ((e == 0 || e == 4 || e == 8) ? 1.f : 0.f);
    }
    if(lane < kShapeDim) sC[warp][kPoseDim + lane] = bp[lane];
    if(lane >= kShapeDim && lane < kShapeDim + 1 + (kBlendK - kBlendKUsed))
      sC[warp][kPoseDim + lane] = lane == kShapeDim ? 1.f : 0.f;
    __syncwarp();
    for(int i = lane; i < kBlendK; i += 32) coef[b * kBlendK + i] = sC[warp][i];
    if(img_b && lane < tc3::KP / 8)
    {
      // coefficient stage image (rows of a 96-frame block permuted by coef_row, fp16 hi | lo x 2^6); the template
      // column and the padding stay out of the tensor-core product
      float x[8];
#pragma unroll
      for(int e = 0; e < 8; e++) x[e] = lane * 8 + e < tc3::KUSED ? sC[warp][lane * 8 + e] * static_cast<float>(1 << tc3::COEF_EXP) : 0.f;
      const long long fb = b / tc3::NF;
      const int r = tc3::coef_row(static_cast<int>(b - fb * tc3::NF));
      uint8_t * blk = img_b + (static_cast<size_t>(fb) * tc3::NKB + lane / 4) * (2 * tc3::B_PART);
      const uint32_t o = static_cast<uint32_t>(r * tc3::ROWB + (lane % 4) * 16);
      tc3::split8_store(x, blk + tc3::swz64(o), blk + tc3::swz64(tc3::B_PART + o));
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// K2 (FFMA): rest = coef (B x 224) . basis^T (224 x 3V) with skinning fused in the epilogue.
//   tile 64 frames x 64 vertices (192 columns), 256 threads, 4 frames x 4 vertices per thread.
// ------------------------------------------------------------------------------------------------------------
namespace k2
{
constexpr int BM = 64, BNV = 64, BN = BNV * 3, BK = 16, THREADS = 256;
constexpr int TM = 4, TNV = 4, TN = TNV * 3;
constexpr int AS_LD = BM + 4, BS_LD = BN + 4;
constexpr int GS_LD = kJoints * 12;
constexpr size_t SMEM_AB = sizeof(float) * 2 * BK * (AS_LD + BS_LD);
constexpr size_t SMEM_G = sizeof(float) * BM * GS_LD;
constexpr size_t SMEM_TOTAL = SMEM_AB + SMEM_G;
} // namespace k2

__device__ __forceinline__ void cp_async16(void * smem, const void * gmem)
{
  unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem));
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit()
{
  asm volatile("cp.async.commit_group;\n" ::);
}
__device__ __forceinline__ void cp_async_wait_all()
{
  asm volatile("cp.async.wait_all;\n" ::);
}

template<bool kSkin>
__global__ void __launch_bounds__(k2::THREADS, 2)
    blend_skin_ffma_kernel(const float * __restrict__ basis, const uint8_t * __restrict__ lbs_joint,
                           const float * __restrict__ lbs_weight, const float * __restrict__ lbs_wsum, int V, int Vpad,
                           int kmax, int B, const float * __restrict__ coef, const float * __restrict__ xforms,
                           const float * __restrict__ theta, float * __restrict__ out)
{
  using namespace k2;
  extern __shared__ __align__(16) float smem[];
  float * As = smem;                    // [2][BK][AS_LD]
  float * Bs = smem + 2 * BK * AS_LD;   // [2][BK][BS_LD]
  float * Gs = smem + 2 * BK * (AS_LD + BS_LD); // [BM][24*12]

  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int v0 = blockIdx.x * BNV;
  const int m0 = blockIdx.y * BM;

  if(kSkin)
  {
    // prefetch the tile's 64 x 24 relative transforms; consumed only in the epilogue
    for(int i = tid; i < BM * GS_LD / 4; i += THREADS)
    {
      int row = i / (GS_LD / 4), q = i % (GS_LD / 4);
      int b = min(m0 + row, B - 1);
      cp_async16(Gs + row * GS_LD + q * 4, xforms + static_cast<size_t>(b) * GS_LD + q * 4);
    }
    cp_async_commit();
  }

  // global -> register staging of one K chunk
  const int a_row = tid >> 2, a_q = tid & 3;
  const float * a_src = coef + static_cast<size_t>(min(m0 + a_row, B - 1)) * kBlendK + a_q * 4;
  const float * b_src[3];
  int b_row[3], b_q[3];
#pragma unroll
  for(int i = 0; i < 3; i++)
  {
    int idx = tid + i * THREADS;
    b_row[i] = idx >> 2;
    b_q[i] = idx & 3;
    b_src[i] = basis + (static_cast<size_t>(v0) * 3 + b_row[i]) * kBlendK + b_q[i] * 4;
  }
  float4 a_reg, b_reg[3];
  auto load_chunk = [&](int kc) {
    a_reg = __ldg(reinterpret_cast<const float4 *>(a_src + kc * BK));
#pragma unroll
    for(int i = 0; i < 3; i++) b_reg[i] = __ldg(reinterpret_cast<const float4 *>(b_src[i] + kc * BK));
  };
  auto store_chunk = [&](int buf) {
    float * as = As + buf * BK * AS_LD + (a_q * 4) * AS_LD + a_row;
    as[0] = a_reg.x;
    as[AS_LD] = a_reg.y;
    as[2 * AS_LD] = a_reg.z;
    as[3 * AS_LD] = a_reg.w;
#pragma unroll
    for(int i = 0; i < 3; i++)
    {
      float * bs = Bs + buf * BK * BS_LD + (b_q[i] * 4) * BS_LD + b_row[i];
      bs[0] = b_reg[i].x;
      bs[BS_LD] = b_reg[i].y;
      bs[2 * BS_LD] = b_reg[i].z;
      bs[3 * BS_LD] = b_reg[i].w;
    }
  };

  float acc[TM][TN];
#pragma unroll
  for(int i = 0; i < TM; i++)
#pragma unroll
    for(int j = 0; j < TN; j++) acc[i][j] = 0.f;

  constexpr int NK = kBlendK / BK;
  load_chunk(0);
  store_chunk(0);
  __syncthreads();
  for(int kc = 0; kc < NK; kc++)
  {
    const int buf = kc & 1;
    if(kc + 1 < NK) load_chunk(kc + 1);
    const float * as = As + buf * BK * AS_LD + ty * TM;
    const float * bs = Bs + buf * BK * BS_LD + tx * TN;
#pragma unroll
    for(int k = 0; k < BK; k++)
    {
      float4 a4 = *reinterpret_cast<const float4 *>(as + k * AS_LD);
      float4 b0 = *reinterpret_cast<const float4 *>(bs + k * BS_LD);
      float4 b1 = *reinterpret_cast<const float4 *>(bs + k * BS_LD + 4);
      float4 b2 = *reinterpret_cast<const float4 *>(bs + k * BS_LD + 8);
      float a[TM] = {a4.x, a4.y, a4.z, a4.w};
      float bb[TN] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w, b2.x, b2.y, b2.z, b2.w};
#pragma unroll
      for(int i = 0; i < TM; i++)
#pragma unroll
        for(int j = 0; j < TN; j++) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
    if(kc + 1 < NK)
    {
      store_chunk(buf ^ 1);
      __syncthreads();
    }
  }

  // ---- epilogue ----
  const int vbase = v0 + tx * TNV;
  const bool vec_ok = (V & 1) == 0; // float2 stores need (b V + v) 3 even
  if(kSkin)
  {
    cp_async_wait_all();
    __syncthreads();
    uint8_t jn[TNV][4];
    float jw[TNV][4], inv_ws[TNV];
    if(kmax <= 4)
    {
#pragma unroll
      for(int jv = 0; jv < TNV; jv++)
      {
#pragma unroll
        for(int k = 0; k < 4; k++)
        {
          bool on = k < kmax;
          jn[jv][k] = on ? lbs_joint[static_cast<size_t>(k) * Vpad + vbase + jv] : 0;
          jw[jv][k] = on ? lbs_weight[static_cast<size_t>(k) * Vpad + vbase + jv] : 0.f;
        }
        inv_ws[jv] = 1.f / lbs_wsum[vbase + jv];
      }
    }
#pragma unroll
    for(int i = 0; i < TM; i++)
    {
      const int b = m0 + ty * TM + i;
      if(b >= B) continue;
      const float * g = Gs + (ty * TM + i) * GS_LD;
      const float * tr = theta + static_cast<size_t>(b) * (kJoints + 1) * 3;
      const float trx = tr[0], try_ = tr[1], trz = tr[2];
      float o[TN];
#pragma unroll
      for(int jv = 0; jv < TNV; jv++)
      {
        const float rx = acc[i][3 * jv], ry = acc[i][3 * jv + 1], rz = acc[i][3 * jv + 2];
        float ox = 0.f, oy = 0.f, oz = 0.f, iw;
        if(kmax <= 4)
        {
#pragma unroll
          for(int k = 0; k < 4; k++)
          {
            const float4 * gj = reinterpret_cast<const float4 *>(g + jn[jv][k] * 12);
            float4 r0 = gj[0], r1 = gj[1], r2 = gj[2];
            float w = jw[jv][k];
            ox = fmaf(w, fmaf(r0.x, rx, fmaf(r0.y, ry, fmaf(r0.z, rz, r0.w))), ox);
            oy = fmaf(w, fmaf(r1.x, rx, fmaf(r1.y, ry, fmaf(r1.z, rz, r1.w))), oy);
            oz = fmaf(w, fmaf(r2.x, rx, fmaf(r2.y, ry, fmaf(r2.z, rz, r2.w))), oz);
          }
          iw = inv_ws[jv];
        }
        else
        {
          const int v = vbase + jv;
          for(int k = 0; k < kmax; k++)
          {
            const float4 * gj = reinterpret_cast<const float4 *>(g + lbs_joint[static_cast<size_t>(k) * Vpad + v] * 12);
            float4 r0 = gj[0], r1 = gj[1], r2 = gj[2];
            float w = lbs_weight[static_cast<size_t>(k) * Vpad + v];
            ox = fmaf(w, fmaf(r0.x, rx, fmaf(r0.y, ry, fmaf(r0.z, rz, r0.w))), ox);
            oy = fmaf(w, fmaf(r1.x, rx, fmaf(r1.y, ry, fmaf(r1.z, rz, r1.w))), oy);
            oz = fmaf(w, fmaf(r2.x, rx, fmaf(r2.y, ry, fmaf(r2.z, rz, r2.w))), oz);
          }
          iw = 1.f / lbs_wsum[v];
        }
        o[3 * jv] = fmaf(ox, iw, trx);
        o[3 * jv + 1] = fmaf(oy, iw, try_);
        o[3 * jv + 2] = fmaf(oz, iw, trz);
      }
      float * dst = out + (static_cast<size_t>(b) * V + vbase) * 3;
      if(vbase + TNV <= V && vec_ok)
      {
#pragma unroll
        for(int q = 0; q < TN / 2; q++) reinterpret_cast<float2 *>(dst)[q] = make_float2(o[2 * q], o[2 * q + 1]);
      }
      else
      {
        for(int q = 0; q < TN; q++)
          if(vbase + q / 3 < V) dst[q] = o[q];
      }
    }
  }
  else
  {
#pragma unroll
    for(int i = 0; i < TM; i++)
    {
      const int b = m0 + ty * TM + i;
      if(b >= B) continue;
      float * dst = out + (static_cast<size_t>(b) * V + vbase) * 3;
      if(vbase + TNV <= V && vec_ok)
      {
#pragma unroll
        for(int q = 0; q < TN / 2; q++) reinterpret_cast<float2 *>(dst)[q] = make_float2(acc[i][2 * q], acc[i][2 * q + 1]);
      }
      else
      {
        for(int q = 0; q < TN; q++)
          if(vbase + q / 3 < V) dst[q] = acc[i][q];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// K3: standalone linear blend skinning (HBM-bound).  CTA = 512 vertices x FR frames; 2 vertices per thread.
//   kAffine: transforms are 3x4 [R|t'] rows (12 floats/joint, internal format); else full 4x4 (16 floats/joint,
//   LinearBlendSkinning's input format) including the homogeneous row.
// ------------------------------------------------------------------------------------------------------------
namespace k3
{
constexpr int THREADS = 256, VPL = kGroupVerts, VPC = THREADS * VPL; // 4 vertices per lane, 1024 per CTA
constexpr int FR = 16;                                               // frames per CTA (weights stay in registers)
}

// Shared-memory bandwidth bounds skinning: every (vertex, frame, influence) needs 12-16 floats of a transform.  A lane
// therefore owns 4 CONSECUTIVE vertices and walks the union of their joints (3.7 on average for a coherent mesh):
// each transform row is fetched once and applied to all 4 vertices from registers.
// kVec2: 8-byte global accesses (needs even V); otherwise scalar accesses.
template<bool kAffine, bool kVec2>
__global__ void __launch_bounds__(k3::THREADS, 2)
    lbs_kernel(const uint8_t * __restrict__ lbs_joint, const float * __restrict__ lbs_weight,
               const float * __restrict__ lbs_wsum, const int8_t * __restrict__ group_nj,
               const uint8_t * __restrict__ group_joint, const float * __restrict__ group_w, int V, int Vpad, int kmax,
               int B, const float * __restrict__ rest, const float * __restrict__ xforms,
               const float * __restrict__ root, int root_stride, float * __restrict__ out)
{
  using namespace k3;
  constexpr int XF = kAffine ? 12 : 16;
  // per-joint stride in shared memory: 12 and 20 floats both map the 8 joint residues to distinct 4-bank groups
  constexpr int XFP = kAffine ? 12 : 20;
  __shared__ __align__(16) float Gs[FR][kJoints * XFP];
  const int tid = threadIdx.x;
  const int b0 = blockIdx.y * FR;
  const int nfr = min(FR, B - b0);
  for(int i = tid; i < nfr * kJoints * XF / 4; i += THREADS)
  {
    const int fr = i / (kJoints * XF / 4), rem = i % (kJoints * XF / 4);
    const int j = rem / (XF / 4), q = rem % (XF / 4);
    *reinterpret_cast<float4 *>(&Gs[fr][j * XFP + 4 * q]) =
        __ldg(reinterpret_cast<const float4 *>(xforms + static_cast<size_t>(b0) * kJoints * XF) + i);
  }
  const int v = (blockIdx.x * THREADS + tid) * VPL; // first of this lane's 4 vertices
  const int g = v / VPL;
  const int nvalid = min(VPL, V - v);               // <= 0: lane idle
  int nj = -1;
  float gw[kGroupJoints][VPL], iw[VPL];
  unsigned gj_lo = 0, gj_hi = 0;
  if(nvalid > 0)
  {
    nj = group_nj ? group_nj[g] : -1;
#pragma unroll
    for(int u = 0; u < VPL; u++) iw[u] = 1.f / lbs_wsum[min(v + u, V - 1)];
    if(nj >= 0)
    {
      const uint2 jj = __ldg(reinterpret_cast<const uint2 *>(group_joint + static_cast<size_t>(g) * kGroupJoints));
      gj_lo = jj.x, gj_hi = jj.y;
#pragma unroll
      for(int k = 0; k < kGroupJoints; k++)
      {
        const float4 w = __ldg(reinterpret_cast<const float4 *>(group_w + (static_cast<size_t>(g) * kGroupJoints + k) * VPL));
        gw[k][0] = w.x, gw[k][1] = w.y, gw[k][2] = w.z, gw[k][3] = w.w;
      }
    }
  }
  __syncthreads();
  if(nvalid <= 0) return;
  const bool full = nvalid == VPL;
  // software pipeline: the loads of frame f + 1 are in flight while frame f is skinned
  float rn[3 * VPL];
  auto load_frame = [&](int f) {
    const size_t base = (static_cast<size_t>(b0 + f) * V + v) * 3;
    if(kVec2 && full)
    {
      const float2 * src = reinterpret_cast<const float2 *>(rest + base);
#pragma unroll
      for(int q = 0; q < 6; q++)
      {
        const float2 t = __ldcs(src + q);
        rn[2 * q] = t.x, rn[2 * q + 1] = t.y;
      }
    }
    else
    {
#pragma unroll
      for(int q = 0; q < 3 * VPL; q++) rn[q] = q < 3 * nvalid ? rest[base + q] : 0.f;
    }
  };
  load_frame(0);
  for(int f = 0; f < nfr; f++)
  {
    const size_t base = (static_cast<size_t>(b0 + f) * V + v) * 3;
    float r[3 * VPL];
#pragma unroll
    for(int q = 0; q < 3 * VPL; q++) r[q] = rn[q];
    if(f + 1 < nfr) load_frame(f + 1);
    float tx = 0.f, ty = 0.f, tz = 0.f;
    if(root)
    {
      const float * rp = root + static_cast<size_t>(b0 + f) * root_stride;
      tx = rp[0], ty = rp[1], tz = rp[2];
    }
    float o[3 * VPL], ow[VPL];
#pragma unroll
    for(int q = 0; q < 3 * VPL; q++) o[q] = 0.f;
#pragma unroll
    for(int u = 0; u < VPL; u++) ow[u] = 0.f;
    if(nj >= 0)
    {
#pragma unroll
      for(int k = 0; k < kGroupJoints; k++)
      {
        if(k < nj)
        {
          const int j = ((k < 4 ? gj_lo : gj_hi) >> (8 * (k & 3))) & 0xff;
          const float4 * gjp = reinterpret_cast<const float4 *>(&Gs[f][j * XFP]);
          const float4 r0 = gjp[0], r1 = gjp[1], r2 = gjp[2];
          float4 r3 = make_float4(0.f, 0.f, 0.f, 1.f);
          if(!kAffine) r3 = gjp[3];
#pragma unroll
          for(int u = 0; u < VPL; u++)
          {
            const float w = gw[k][u];
            const float rx = r[3 * u], ry = r[3 * u + 1], rz = r[3 * u + 2];
            o[3 * u] = fmaf(w, fmaf(r0.x, rx, fmaf(r0.y, ry, fmaf(r0.z, rz, r0.w))), o[3 * u]);
            o[3 * u + 1] = fmaf(w, fmaf(r1.x, rx, fmaf(r1.y, ry, fmaf(r1.z, rz, r1.w))), o[3 * u + 1]);
            o[3 * u + 2] = fmaf(w, fmaf(r2.x, rx, fmaf(r2.y, ry, fmaf(r2.z, rz, r2.w))), o[3 * u + 2]);
            if(!kAffine) ow[u] = fmaf(w, fmaf(r3.x, rx, fmaf(r3.y, ry, fmaf(r3.z, rz, r3.w))), ow[u]);
          }
        }
      }
    }
    else
    {
      // generic path: per-vertex influence slots (more than kGroupJoints joints in the group, or no group tables)
      for(int u = 0; u < nvalid; u++)
      {
        const float rx = r[3 * u], ry = r[3 * u + 1], rz = r[3 * u + 2];
        float ox = 0.f, oy = 0.f, oz = 0.f, o4 = 0.f;
        for(int k = 0; k < kmax; k++)
        {
          const float w = lbs_weight[static_cast<size_t>(k) * Vpad + v + u];
          const float4 * gjp = reinterpret_cast<const float4 *>(&Gs[f][lbs_joint[static_cast<size_t>(k) * Vpad + v + u] * XFP]);
          const float4 r0 = gjp[0], r1 = gjp[1], r2 = gjp[2];
          ox = fmaf(w, fmaf(r0.x, rx, fmaf(r0.y, ry, fmaf(r0.z, rz, r0.w))), ox);
          oy = fmaf(w, fmaf(r1.x, rx, fmaf(r1.y, ry, fmaf(r1.z, rz, r1.w))), oy);
          oz = fmaf(w, fmaf(r2.x, rx, fmaf(r2.y, ry, fmaf(r2.z, rz, r2.w))), oz);
          if(!kAffine)
          {
            const float4 r3 = gjp[3];
            o4 = fmaf(w, fmaf(r3.x, rx, fmaf(r3.y, ry, fmaf(r3.z, rz, r3.w))), o4);
          }
        }
#pragma unroll
        for(int uu = 0; uu < VPL; uu++)
          if(uu == u) o[3 * uu] = ox, o[3 * uu + 1] = oy, o[3 * uu + 2] = oz, ow[uu] = o4;
      }
    }
#pragma unroll
    for(int u = 0; u < VPL; u++)
    {
      const float inv = kAffine ? iw[u] : 1.f / ow[u];
      o[3 * u] = fmaf(o[3 * u], inv, tx);
      o[3 * u + 1] = fmaf(o[3 * u + 1], inv, ty);
      o[3 * u + 2] = fmaf(o[3 * u + 2], inv, tz);
    }
    if(kVec2 && full)
    {
      float2 * dst = reinterpret_cast<float2 *>(out + base);
#pragma unroll
      for(int q = 0; q < 6; q++) __stcs(dst + q, make_float2(o[2 * q], o[2 * q + 1]));
    }
    else
    {
#pragma unroll
      for(int q = 0; q < 3 * VPL; q++)
        if(q < 3 * nvalid) out[base + q] = o[q];
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// Generic per-module kernels (any V, caller tensors; used by the module-level API and the Tester KATs).
// ------------------------------------------------------------------------------------------------------------
__global__ void rodrigues_kernel(long long n, const float * __restrict__ theta, float * __restrict__ rot)
{
  long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if(i >= n) return;
  float R[9];
  rodrigues3(theta[3 * i], theta[3 * i + 1], theta[3 * i + 2], R);
#pragma unroll
  for(int e = 0; e < 9; e++) rot[9 * i + e] = R[e];
}

// one thread per (b, v, k): pose blend 207-dot and shape blend 10-dot
__global__ void blend_generic_kernel(int B, int V, const float * __restrict__ beta, const float * __restrict__ rot,
                                     const float * __restrict__ shape_basis, const float * __restrict__ pose_basis,
                                     float * __restrict__ shape_bs, float * __restrict__ pose_bs)
{
  long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if(i >= static_cast<long long>(B) * V * 3) return;
  int b = static_cast<int>(i / (static_cast<long long>(V) * 3));
  long long vk = i % (static_cast<long long>(V) * 3);
  const float * pb = pose_basis + vk * kPoseDim;
  const float * r = rot + static_cast<size_t>(b) * kJoints * 9 + 9; // skip the root rotation
  float acc = 0.f;
  for(int d = 0; d < kPoseDim; d++)
  {
    int e = d % 9;
    float c = r[d] - ((e == 0 || e == 4 || e == 8) ? 1.f : 0.f);
    acc = fmaf(c, pb[d], acc);
  }
  pose_bs[i] = acc;
  const float * sb_ = shape_basis + vk * kShapeDim;
  float s = 0.f;
  for(int d = 0; d < kShapeDim; d++) s = fmaf(beta[b * kShapeDim + d], sb_[d], s);
  shape_bs[i] = s;
}

__global__ void linear_combine_kernel(long long n, long long vk_count, const float * __restrict__ templ,
                                      const float * __restrict__ shape_bs, const float * __restrict__ pose_bs,
                                      float * __restrict__ rest)
{
  long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if(i >= n) return;
  rest[i] = templ[i % vk_count] + shape_bs[i] + pose_bs[i];
}

// one warp per (b, j, k): joints = Jreg . (T + S)
__global__ void joint_regress_kernel(int B, int V, const float * __restrict__ templ, const float * __restrict__ jreg,
                                     const float * __restrict__ shape_bs, float * __restrict__ joints)
{
  int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if(w >= B * kJoints * 3) return;
  int b = w / (kJoints * 3), j = (w / 3) % kJoints, k = w % 3;
  float acc = 0.f;
  for(int v = lane; v < V; v += 32)
    acc = fmaf(jreg[static_cast<size_t>(j) * V + v], templ[3 * v + k] + shape_bs[(static_cast<size_t>(b) * V + v) * 3 + k], acc);
#pragma unroll
  for(int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if(lane == 0) joints[w] = acc;
}

// WorldTransformation::transform on caller-supplied rotations (any 3x3, the Tester KAT feeds non-rotations)
__global__ void world_transform_kernel(int B, const long long * __restrict__ kine_tree, const float * __restrict__ joints,
                                       const float * __restrict__ rot, float * __restrict__ out)
{
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if(b >= B) return;
  float G[kJoints][12];
  const float * J = joints + static_cast<size_t>(b) * kJoints * 3;
  const float * R = rot + static_cast<size_t>(b) * kJoints * 9;
  for(int j = 0; j < kJoints; j++)
  {
    long long p = kine_tree[j];
    const float * Rj = R + 9 * j;
    if(j == 0 || p < 0 || p >= kJoints)
    {
      for(int r = 0; r < 3; r++)
      {
        for(int c = 0; c < 3; c++) G[j][4 * r + c] = Rj[3 * r + c];
        G[j][4 * r + 3] = J[3 * j + r];
      }
    }
    else
    {
      float t[3] = {J[3 * j] - J[3 * p], J[3 * j + 1] - J[3 * p + 1], J[3 * j + 2] - J[3 * p + 2]};
      for(int r = 0; r < 3; r++)
      {
        float p0 = G[p][4 * r], p1 = G[p][4 * r + 1], p2 = G[p][4 * r + 2], p3 = G[p][4 * r + 3];
        for(int c = 0; c < 3; c++) G[j][4 * r + c] = p0 * Rj[c] + p1 * Rj[3 + c] + p2 * Rj[6 + c];
        G[j][4 * r + 3] = p0 * t[0] + p1 * t[1] + p2 * t[2] + p3;
      }
    }
  }
  float * o = out + static_cast<size_t>(b) * kJoints * 16;
  for(int j = 0; j < kJoints; j++)
  {
    for(int r = 0; r < 3; r++)
    {
      for(int c = 0; c < 3; c++) o[16 * j + 4 * r + c] = G[j][4 * r + c];
      o[16 * j + 4 * r + 3] =
          G[j][4 * r + 3] - (G[j][4 * r] * J[3 * j] + G[j][4 * r + 1] * J[3 * j + 1] + G[j][4 * r + 2] * J[3 * j + 2]);
    }
    o[16 * j + 12] = 0.f, o[16 * j + 13] = 0.f, o[16 * j + 14] = 0.f, o[16 * j + 15] = 1.f;
  }
}

// dense-weight skinning with the full homogeneous row (LinearBlendSkinning.cpp:463-467, 545-550)
__global__ void lbs_dense_kernel(int B, int V, const float * __restrict__ weights, const float * __restrict__ rest,
                                 const float * __restrict__ xf, const float * __restrict__ root,
                                 float * __restrict__ out)
{
  long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if(i >= static_cast<long long>(B) * V) return;
  int b = static_cast<int>(i / V), v = static_cast<int>(i % V);
  float rx = rest[3 * i], ry = rest[3 * i + 1], rz = rest[3 * i + 2];
  float M[16];
  for(int e = 0; e < 16; e++) M[e] = 0.f;
  for(int j = 0; j < kJoints; j++)
  {
    float w = weights[static_cast<size_t>(v) * kJoints + j];
    const float * g = xf + (static_cast<size_t>(b) * kJoints + j) * 16;
    for(int e = 0; e < 16; e++) M[e] = fmaf(w, g[e], M[e]);
  }
  float h[4];
  for(int r = 0; r < 4; r++) h[r] = M[4 * r] * rx + M[4 * r + 1] * ry + M[4 * r + 2] * rz + M[4 * r + 3];
  for(int k = 0; k < 3; k++) out[3 * i + k] = h[k] / h[3] + (root ? root[3 * b + k] : 0.f);
}

// ------------------------------------------------------------------------------------------------------------
// Normals (SMPL::calcNormal / calcVertexNormal, src/SMPL.cpp:518-535), batched: one thread per (frame, item).
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void normalize3(float & x, float & y, float & z)
{
  // torch::nn::functional::normalize: v / max(||v||, 1e-12)
  float n = fmaxf(sqrtf(x * x + y * y + z * z), 1e-12f);
  x /= n, y /= n, z /= n;
}

__device__ __forceinline__ void face_normal(const float * __restrict__ verts, const int32_t * __restrict__ faces, int f,
                                            float & nx, float & ny, float & nz)
{
  const float * a = verts + 3 * faces[3 * f], *b = verts + 3 * faces[3 * f + 1], *c = verts + 3 * faces[3 * f + 2];
  float e1x = b[0] - a[0], e1y = b[1] - a[1], e1z = b[2] - a[2];
  float e2x = c[0] - a[0], e2y = c[1] - a[1], e2z = c[2] - a[2];
  nx = e1y * e2z - e1z * e2y;
  ny = e1z * e2x - e1x * e2z;
  nz = e1x * e2y - e1y * e2x;
  normalize3(nx, ny, nz);
}

__global__ void normals_kernel(const int32_t * __restrict__ faces, const int32_t * __restrict__ adj_offset,
                               const int32_t * __restrict__ adj_faces, int V, int F, int B,
                               const float * __restrict__ verts, int nF, const long long * __restrict__ face_idx,
                               float * __restrict__ fn, int nV, const long long * __restrict__ vert_idx,
                               float * __restrict__ vn)
{
  long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int per = nF + nV;
  if(i >= static_cast<long long>(B) * per) return;
  int b = static_cast<int>(i / per), it = static_cast<int>(i % per);
  const float * vb = verts + static_cast<size_t>(b) * V * 3;
  if(it < nF)
  {
    long long f = face_idx[it];
    float x = 0.f, y = 0.f, z = 0.f;
    if(f >= 0 && f < F) face_normal(vb, faces, static_cast<int>(f), x, y, z);
    float * o = fn + (static_cast<size_t>(b) * nF + it) * 3;
    o[0] = x, o[1] = y, o[2] = z;
  }
  else
  {
    it -= nF;
    long long v = vert_idx[it];
    float ax = 0.f, ay = 0.f, az = 0.f;
    if(v >= 0 && v < V)
    {
      int s = adj_offset[v], e = adj_offset[v + 1];
      float w = 1.f / static_cast<float>(e - s);
      for(int k = s; k < e; k++)
      {
        float x, y, z;
        face_normal(vb, faces, adj_faces[k], x, y, z);
        ax = fmaf(w, x, ax), ay = fmaf(w, y, ay), az = fmaf(w, z, az);
      }
      normalize3(ax, ay, az);
    }
    float * o = vn + (static_cast<size_t>(b) * nV + it) * 3;
    o[0] = ax, o[1] = ay, o[2] = az;
  }
}

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
namespace sb
{
ChainTopo make_topo(const ModelDev & d)
{
  ChainTopo t;
  for(int j = 0; j < kJoints; j++)
  {
    t.parent[j] = d.parent[j];
    t.depth[j] = d.depth[j];
  }
  t.max_depth = d.max_depth;
  return t;
}

int launch_pose_chain(const ModelDev & d, cudaStream_t st, int B, const float * beta, long long beta_stride,
                      const float * theta, float * coef, float * xforms, float * joints, float * xforms44,
                      void * tc3_scratch)
{
  // with tc3_scratch the kernel also writes the coefficient / transform stage images of K2''' (and zero rows for the
  // frames that pad the last 96-frame block)
  const int Bpad = tc3_scratch ? static_cast<int>(align_up(static_cast<size_t>(B), tc3::NF)) : B;
  uint8_t * img_b = static_cast<uint8_t *>(tc3_scratch);
  uint8_t * img_g = tc3_scratch ? img_b + tc3::img_g_offset(Bpad) : nullptr;
  int grid = (Bpad + kChainWarps - 1) / kChainWarps;
  pose_chain_kernel<<<grid, kChainWarps * 32, 0, st>>>(make_topo(d), d.joint_template, d.joint_shape, B, beta,
                                                       beta_stride, theta, coef, xforms, joints, xforms44, img_b, img_g, Bpad,
                                                       tc3::window_map(d));
  SB_LAUNCHED();
  return SMPLPP_OK;
}

int launch_blend_skin_ffma(const ModelDev & d, cudaStream_t st, int B, const float * coef, const float * xforms,
                           const float * theta, float * out, bool skin)
{
  static bool configured[64] = {};
  if(first_call_on_device(configured))
  {
    SB_CUDA(cudaFuncSetAttribute(blend_skin_ffma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(k2::SMEM_TOTAL)));
    SB_CUDA(cudaFuncSetAttribute(blend_skin_ffma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(k2::SMEM_AB)));
  }
  dim3 grid(d.Vpad / k2::BNV, (B + k2::BM - 1) / k2::BM);
  if(skin)
    blend_skin_ffma_kernel<true><<<grid, k2::THREADS, k2::SMEM_TOTAL, st>>>(
        d.basis, d.lbs_joint, d.lbs_weight, d.lbs_wsum, d.V, d.Vpad, d.kmax, B, coef, xforms, theta, out);
  else
    blend_skin_ffma_kernel<false><<<grid, k2::THREADS, k2::SMEM_AB, st>>>(
        d.basis, d.lbs_joint, d.lbs_weight, d.lbs_wsum, d.V, d.Vpad, d.kmax, B, coef, xforms, theta, out);
  SB_LAUNCHED();
  return SMPLPP_OK;
}

int launch_lbs(const ModelDev & d, cudaStream_t st, int B, const float * rest, const float * xforms, bool affine,
               const float * root, int root_stride, float * out)
{
  if(affine && g_lbs_variant == 2 && lbs_tc_usable(d, rest, out, xforms))
    return launch_lbs_tc(d, st, B, rest, xforms, kXformFloats, root, root_stride, out);
  if(affine && g_lbs_variant == 0 && lbs_tma_usable(d, rest, out, xforms))
    return launch_lbs_tma(d, st, B, rest, xforms, root, root_stride, out);
  dim3 grid((d.V + k3::VPC - 1) / k3::VPC, (B + k3::FR - 1) / k3::FR);
  const bool vec2 = (d.V & 1) == 0 && (reinterpret_cast<uintptr_t>(rest) & 7) == 0 && (reinterpret_cast<uintptr_t>(out) & 7) == 0;
#define SB_LBS(AFF, VEC)                                                                                               \
  lbs_kernel<AFF, VEC><<<grid, k3::THREADS, 0, st>>>(d.lbs_joint, d.lbs_weight, d.lbs_wsum, d.group_nj, d.group_joint, \
                                                     d.group_w, d.V, d.Vpad, d.kmax, B, rest, xforms, root,           \
                                                     root_stride, out)
  if(affine && vec2)
    SB_LBS(true, true);
  else if(affine)
    SB_LBS(true, false);
  else if(vec2)
    SB_LBS(false, true);
  else
    SB_LBS(false, false);
#undef SB_LBS
  SB_LAUNCHED();
  return SMPLPP_OK;
}
} // namespace sb

extern "C" int smplpp_set_forward_variant(int variant)
{
  // 200 / 201 / 202: standalone skinning kernel (FFMA per-warp TMA pipelines / FFMA register-pipelined kernel / skinning
  // matrices on tcgen05, the default; the FFMA kernels are bound by FFMA issue at ~3.2 TB/s, see DESIGN.md §4)
  if(variant == 300 || variant == 301) // VPoser Jacobian: 300 tensor cores (default), 301 FFMA kernel
  {
    g_vposer_jac_variant = variant - 300;
    return SMPLPP_OK;
  }
  if(variant >= 200 && variant <= 202)
  {
    g_lbs_variant = variant - 200;
    return SMPLPP_OK;
  }
  // IK step: 400 auto (two kernels for a shared attachment topology, the fused kernel for per-frame attachments),
  // 401 two kernels, 402 fused kernel for every call
  if(variant >= 400 && variant <= 402)
  {
    g_ik_variant = variant - 400;
    return SMPLPP_OK;
  }
  // normal equations + solve of the two-kernel IK path: 410 auto (fp64 tensor-core kernel where the shape allows),
  // 411 the scalar ik_solve_kernel always
  if(variant == 410 || variant == 411)
  {
    g_solve_variant = variant - 410;
    return SMPLPP_OK;
  }
  // pose-blend columns of the IK Jacobian: 420 auto (ik_poseblend_tc_kernel, tcgen05), 421 the FFMA phase of ik_jacobian_kernel
  if(variant >= 420 && variant <= 422) // 422: tcgen05 pose-blend columns on the FFMA rest shape (isolates the two in tests)
  {
    g_poseblend_variant = variant - 420;
    return SMPLPP_OK;
  }
  if(variant != 0 && variant != 1 && variant != 3 && variant != 6)
    return fail(SMPLPP_ERR_INVALID, "SMPL", "unknown forward variant");
  g_forward_variant = variant;
  return SMPLPP_OK;
}

extern "C" size_t smplpp_forward_workspace_bytes(const smplpp_model_t * model, int64_t batch)
{
  if(!model || batch < 1) return 0;
  size_t bpad = align_up(static_cast<size_t>(batch), 128);
  size_t bytes = 512;
  bytes += align_up(bpad * kBlendK * sizeof(float));         // coefficients (A operand)
  bytes += align_up(bpad * kJoints * 12 * sizeof(float));    // relative transforms 3x4
  bytes += tc3_frame_operand_bytes(batch);                  // fp16 hi / lo coefficient + transform stage images (variant 6)
  bytes += align_up(static_cast<size_t>(batch) * model->d.V * 3 * sizeof(float)); // rest shape (unfused variant)
  return bytes;
}

extern "C" int smplpp_forward(const smplpp_model_t * model, void * stream, int64_t batch, const float * beta,
                              int64_t beta_stride, const float * theta, float * vertices, float * joints,
                              float * transforms, float * rest_shape, void * workspace, size_t workspace_bytes)
{
  if(!model || batch < 1 || !beta || !theta) return fail(SMPLPP_ERR_INVALID, "SMPL", "Cannot launch a SMPL model!");
  if(batch > (1ll << 24)) return fail(SMPLPP_ERR_INVALID, "SMPL", "Cannot launch a SMPL model! (batch too large)");
  if(!workspace || workspace_bytes < smplpp_forward_workspace_bytes(model, batch))
    return fail(SMPLPP_ERR_INVALID, "SMPL", "Cannot launch a SMPL model! (workspace too small)");
  const ModelDev & d = model->d;
  const int B = static_cast<int>(batch);
  cudaStream_t st = as_stream(stream);
  size_t bpad = align_up(static_cast<size_t>(batch), 128);
  char * ws = align_up_ptr<char>(workspace);
  float * coef = reinterpret_cast<float *>(ws);
  ws += align_up(bpad * kBlendK * sizeof(float));
  float * xforms = reinterpret_cast<float *>(ws);
  ws += align_up(bpad * kJoints * 12 * sizeof(float));
  void * tc3_scratch = ws;
  ws += tc3_frame_operand_bytes(batch);
  float * rest_ws = reinterpret_cast<float *>(ws);

  const bool need_verts = vertices != nullptr;
  const bool need_rest = rest_shape != nullptr;
  int variant = g_forward_variant;
  if(variant == 0) variant = model->d.tc3_ready ? 6 : 1;
  if(variant == 6 && !model->d.tc3_ready)
    return fail(SMPLPP_ERR_INVALID, "SMPL", "tcgen05 blend variant is not available for this model");
  // K1 writes the stage images of K2''' itself when that kernel follows
  const bool fused_images = variant == 6 && need_verts && !need_rest;
  int rc = launch_pose_chain(d, st, B, beta, beta_stride, theta, (need_verts || need_rest) ? coef : nullptr, xforms,
                             joints, transforms, fused_images ? tc3_scratch : nullptr);
  if(rc != SMPLPP_OK) return rc;
  if(need_rest || (need_verts && variant == 3))
  {
    float * rest = need_rest ? rest_shape : rest_ws;
    rc = launch_blend_skin_ffma(d, st, B, coef, xforms, theta, rest, false);
    if(rc != SMPLPP_OK) return rc;
    if(need_verts) rc = launch_lbs(d, st, B, rest, xforms, true, theta, (kJoints + 1) * 3, vertices);
    return rc;
  }
  if(need_verts)
  {
    if(variant == 6)
      rc = launch_blend_skin_tc3(d, st, B, coef, xforms, tc3_scratch, theta, vertices, /*images_ready=*/true);
    else
      rc = launch_blend_skin_ffma(d, st, B, coef, xforms, theta, vertices, true);
  }
  return rc;
}

// ---- module-level API ----

extern "C" int smplpp_blend_shape(void * stream, int64_t batch, int64_t V, const float * beta, const float * theta,
                                  const float * shape_basis, const float * pose_basis, float * shape_bs, float * pose_bs,
                                  float * pose_rot)
{
  if(batch < 1 || V < 1 || !beta) return fail(SMPLPP_ERR_INVALID, "BlendShape", "Failed to set beta!");
  if(!theta) return fail(SMPLPP_ERR_INVALID, "BlendShape", "Failed to set theta!");
  if(!shape_basis || !pose_basis || !shape_bs || !pose_bs || !pose_rot)
    return fail(SMPLPP_ERR_INVALID, "BlendShape", "Cannot blend pose-dependented shape!");
  cudaStream_t st = as_stream(stream);
  long long n = batch * kJoints;
  rodrigues_kernel<<<static_cast<unsigned>((n + 127) / 128), 128, 0, st>>>(n, theta, pose_rot);
  SB_LAUNCHED();
  long long total = batch * V * 3;
  blend_generic_kernel<<<static_cast<unsigned>((total + 127) / 128), 128, 0, st>>>(
      static_cast<int>(batch), static_cast<int>(V), beta, pose_rot, shape_basis, pose_basis, shape_bs, pose_bs);
  SB_LAUNCHED();
  return SMPLPP_OK;
}

extern "C" int smplpp_joint_regression(void * stream, int64_t batch, int64_t V, const float * templ, const float * jreg,
                                       const float * shape_bs, const float * pose_bs, float * rest, float * joints)
{
  if(batch < 1 || V < 1 || !templ || !shape_bs || !pose_bs || !rest)
    return fail(SMPLPP_ERR_INVALID, "JointRegression", "Cannot linearly combine shapes!");
  if(!jreg || !joints) return fail(SMPLPP_ERR_INVALID, "JointRegression", "Cannot regress vertices to joints!");
  cudaStream_t st = as_stream(stream);
  long long n = batch * V * 3;
  linear_combine_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(n, V * 3, templ, shape_bs, pose_bs, rest);
  SB_LAUNCHED();
  long long warps = batch * kJoints * 3;
  joint_regress_kernel<<<static_cast<unsigned>((warps * 32 + 127) / 128), 128, 0, st>>>(
      static_cast<int>(batch), static_cast<int>(V), templ, jreg, shape_bs, joints);
  SB_LAUNCHED();
  return SMPLPP_OK;
}

extern "C" int smplpp_world_transformation(void * stream, int64_t batch, const int64_t * kine_tree, const float * joints,
                                           const float * pose_rot, float * transforms)
{
  if(batch < 1 || !kine_tree || !joints || !pose_rot || !transforms)
    return fail(SMPLPP_ERR_INVALID, "WorldTransformation", "Cannot transform bones locally!");
  world_transform_kernel<<<static_cast<unsigned>((batch + 63) / 64), 64, 0, as_stream(stream)>>>(
      static_cast<int>(batch), reinterpret_cast<const long long *>(kine_tree), joints, pose_rot, transforms);
  SB_LAUNCHED();
  return SMPLPP_OK;
}

extern "C" int smplpp_linear_blend_skinning(void * stream, int64_t batch, int64_t V, const float * weights,
                                            const float * rest, const float * transforms, const float * root_pos,
                                            float * vertices)
{
  if(batch < 1 || V < 1 || !weights) return fail(SMPLPP_ERR_INVALID, "LinearBlendSkinning", "Failed to set weights!");
  if(!rest || !transforms || !vertices)
    return fail(SMPLPP_ERR_INVALID, "LinearBlendSkinning", "Cannot convert Cartesian coordinates to homogeneous one!");
  long long n = batch * V;
  lbs_dense_kernel<<<static_cast<unsigned>((n + 127) / 128), 128, 0, as_stream(stream)>>>(
      static_cast<int>(batch), static_cast<int>(V), weights, rest, transforms, root_pos, vertices);
  SB_LAUNCHED();
  return SMPLPP_OK;
}

extern "C" int smplpp_model_skinning(const smplpp_model_t * model, void * stream, int64_t batch, const float * rest,
                                     const float * transforms, const float * root_pos, float * vertices)
{
  if(!model || batch < 1 || !rest || !transforms || !vertices)
    return fail(SMPLPP_ERR_INVALID, "LinearBlendSkinning", "Failed to get vertices of new pose!");
  return launch_lbs(model->d, as_stream(stream), static_cast<int>(batch), rest, transforms, false, root_pos, 3, vertices);
}

extern "C" int smplpp_normals(const smplpp_model_t * model, void * stream, int64_t batch, const float * vertices,
                              int64_t n_faces, const int64_t * face_idx, float * face_normals, int64_t n_verts,
                              const int64_t * vert_idx, float * vertex_normals)
{
  if(!model || batch < 1 || !vertices || n_faces < 0 || n_verts < 0 || (n_faces > 0 && (!face_idx || !face_normals))
     || (n_verts > 0 && (!vert_idx || !vertex_normals)))
    return fail(SMPLPP_ERR_INVALID, "SMPL", "Failed to get face indices!");
  long long total = batch * (n_faces + n_verts);
  if(total == 0) return SMPLPP_OK;
  const ModelDev & d = model->d;
  normals_kernel<<<static_cast<unsigned>((total + 127) / 128), 128, 0, as_stream(stream)>>>(
      d.faces, d.adj_offset, d.adj_faces, d.V, d.F, static_cast<int>(batch), vertices, static_cast<int>(n_faces),
      reinterpret_cast<const long long *>(face_idx), face_normals, static_cast<int>(n_verts),
      reinterpret_cast<const long long *>(vert_idx), vertex_normals);
  SB_LAUNCHED();
  return SMPLPP_OK;
}

extern "C" int smplpp_model_skinning34(const smplpp_model_t * model, void * stream, int64_t batch, const float * rest,
                                       const float * transforms34, const float * root_pos, float * vertices)
{
  if(!model || batch < 1 || !rest || !transforms34 || !vertices)
    return fail(SMPLPP_ERR_INVALID, "LinearBlendSkinning", "Failed to get vertices of new pose!");
  return launch_lbs(model->d, as_stream(stream), static_cast<int>(batch), rest, transforms34, true, root_pos, 3, vertices);
}
