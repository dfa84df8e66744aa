// K3' : standalone linear blend skinning as per-warp TMA pipelines (HBM-bound row of SURVEY.md §8d).
//
// Reference semantics: LinearBlendSkinning::skinning (src/LinearBlendSkinning.cpp:445-483) with cart2homo / homo2cart
// (:505-553): vert = (sum_j W[v,j] G'_j [rest_v; 1])[:3] / sum_j W[v,j] + root translation.
//
// Each warp owns 128 consecutive vertices (1536 contiguous bytes per frame) and walks the CTA's frames with a ring of
// bulk copies: cp.async.bulk global->shared fills stage s (completion on the warp's own mbarrier), the lanes skin
// their 4 consecutive vertices IN PLACE (each joint transform of the group is fetched once and applied to all 4
// vertices from registers), and cp.async.bulk shared->global drains the same stage.  Memory traffic is decoupled
// from registers (3 frames of loads in flight per warp, 16 warps per SM), both directions move whole 16-byte-aligned
// lines, and there is no CTA-wide synchronisation after the transforms of the CTA's frames were staged.
//
// A frame is V * 12 bytes = 82 680 B for SMPL, i.e. 8 mod 16: every other frame starts 8 bytes off a 16-byte
// boundary.  Loads copy the enclosing aligned range (data lands at stage + lo, lo in {0, 8}); stores send the
// aligned interior with the bulk copy and the 8-byte head / tail with ordinary stores.
#include "forward.cuh"
#include "tc_ptx.cuh"

using namespace sb;

namespace k3t
{
constexpr int WARPS = 8;
constexpr int THREADS = WARPS * 32;
constexpr int VPL = kGroupVerts;               // 4 consecutive vertices per lane
constexpr int SLICE = 32 * VPL;                // 128 vertices per warp
constexpr int STAGE_BYTES = SLICE * 12 + 16;   // + room for the 8-byte misalignment

template<int FRC, int S>
struct Layout
{
  static constexpr int XF_FLOATS = FRC * kJoints * kXformFloats;
  static constexpr int OFF_ROOT = XF_FLOATS * 4;
  static constexpr int OFF_RING = OFF_ROOT + FRC * 16;
  static constexpr int OFF_BAR = OFF_RING + WARPS * S * STAGE_BYTES;
  static constexpr int BYTES = OFF_BAR + WARPS * S * 8 + 128;
};
} // namespace k3t

// One frame of one warp: skin the lane's 4 vertices in place.  NJ = number of joint slots walked (the warp-wide
// maximum of the lanes' union sizes, so the loop is branch-free; lanes with fewer joints carry zero weights).
template<int NJ>
__device__ __forceinline__ void skin_in_place(uint32_t my, uint32_t lo, uint32_t gf, const uint32_t (&joff)[kGroupJoints],
                                              const float (&gw)[kGroupJoints][k3t::VPL], const float (&iw)[k3t::VPL],
                                              float tx, float ty, float tz)
{
  constexpr int VPL = k3t::VPL;
  float r[3 * VPL];
  if(lo == 0)
  {
#pragma unroll
    for(int q = 0; q < 3; q++)
    {
      const float4 t = ptx::lds128(my + 16 * q);
      r[4 * q] = t.x, r[4 * q + 1] = t.y, r[4 * q + 2] = t.z, r[4 * q + 3] = t.w;
    }
  }
  else
  {
    const float2 h = ptx::lds64(my);
    const float4 m0 = ptx::lds128(my + 8), m1 = ptx::lds128(my + 24);
    const float2 t = ptx::lds64(my + 40);
    r[0] = h.x, r[1] = h.y, r[2] = m0.x, r[3] = m0.y, r[4] = m0.z, r[5] = m0.w;
    r[6] = m1.x, r[7] = m1.y, r[8] = m1.z, r[9] = m1.w, r[10] = t.x, r[11] = t.y;
  }
  float o[3 * VPL];
#pragma unroll
  for(int q = 0; q < 3 * VPL; q++) o[q] = 0.f;
#pragma unroll
  for(int k = 0; k < NJ; k++)
  {
    const uint32_t gj = gf + joff[k];
    const float4 r0 = ptx::lds128(gj), r1 = ptx::lds128(gj + 16), r2 = ptx::lds128(gj + 32);
#pragma unroll
    for(int u = 0; u < VPL; u++)
    {
      const float w = gw[k][u];
      const float rx = r[3 * u], ry = r[3 * u + 1], rz = r[3 * u + 2];
      o[3 * u] = fmaf(w, fmaf(r0.x, rx, fmaf(r0.y, ry, fmaf(r0.z, rz, r0.w))), o[3 * u]);
      o[3 * u + 1] = fmaf(w, fmaf(r1.x, rx, fmaf(r1.y, ry, fmaf(r1.z, rz, r1.w))), o[3 * u + 1]);
      o[3 * u + 2] = fmaf(w, fmaf(r2.x, rx, fmaf(r2.y, ry, fmaf(r2.z, rz, r2.w))), o[3 * u + 2]);
    }
  }
#pragma unroll
  for(int u = 0; u < VPL; u++)
  {
    o[3 * u] = fmaf(o[3 * u], iw[u], tx);
    o[3 * u + 1] = fmaf(o[3 * u + 1], iw[u], ty);
    o[3 * u + 2] = fmaf(o[3 * u + 2], iw[u], tz);
  }
  if(lo == 0)
  {
#pragma unroll
    for(int q = 0; q < 3; q++) ptx::sts128(my + 16 * q, make_float4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]));
  }
  else
  {
    ptx::sts64(my, make_float2(o[0], o[1]));
    ptx::sts128(my + 8, make_float4(o[2], o[3], o[4], o[5]));
    ptx::sts128(my + 24, make_float4(o[6], o[7], o[8], o[9]));
    ptx::sts64(my + 40, make_float2(o[10], o[11]));
  }
}

template<int FRC, int S>
__global__ void __launch_bounds__(k3t::THREADS, 2)
    lbs_tma_kernel(const uint8_t * __restrict__ lbs_joint, const float * __restrict__ lbs_weight,
                   const float * __restrict__ lbs_wsum, const int8_t * __restrict__ group_nj,
                   const uint8_t * __restrict__ group_joint, const float * __restrict__ group_w, int V, int Vpad, int kmax,
                   int B, const float * __restrict__ rest, const float * __restrict__ xforms, const float * __restrict__ root,
                   int root_stride, float * __restrict__ out)
{
  using namespace k3t;
  using L = Layout<FRC, S>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t * smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~uintptr_t(127));
  float * Gs = reinterpret_cast<float *>(smem);
  float * Tr = reinterpret_cast<float *>(smem + L::OFF_ROOT);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint8_t * ring = smem + L::OFF_RING + warp * S * STAGE_BYTES;
  uint64_t * full = reinterpret_cast<uint64_t *>(smem + L::OFF_BAR) + warp * S;

  const int b0 = blockIdx.y * FRC;
  const int nfr = min(FRC, B - b0);
  const int v0 = (blockIdx.x * WARPS + warp) * SLICE;
  const int nv = min(SLICE, V - v0); // <= 0: this warp has no vertices
  const unsigned long long total_bytes = static_cast<unsigned long long>(B) * V * 12ull;
  const unsigned long long frame_bytes = static_cast<unsigned long long>(V) * 12ull;
  const unsigned long long a0 = (static_cast<unsigned long long>(b0) * V + v0) * 12ull; // chunk of frame 0
  const uint32_t data_bytes = static_cast<uint32_t>(max(nv, 0)) * 12u;
  const uint8_t * rest_b = reinterpret_cast<const uint8_t *>(rest);
  uint8_t * out_b = reinterpret_cast<uint8_t *>(out);

  // bulk load of this warp's chunk of frame f: the enclosing 16-byte aligned range, clipped to the tensor
  auto issue_load = [&](int f) {
    const unsigned long long a = a0 + static_cast<unsigned long long>(f) * frame_bytes;
    const uint32_t lo = static_cast<uint32_t>(a) & 15u;
    const unsigned long long ga = a - lo;
    const unsigned long long avail = (total_bytes - ga) & ~15ull;
    const uint32_t nb = static_cast<uint32_t>(min(static_cast<unsigned long long>((lo + data_bytes + 15u) & ~15u), avail));
    const int s = f % S;
    ptx::mbar_expect_tx(&full[s], nb);
    ptx::bulk_load_1d(ring + s * STAGE_BYTES, rest_b + ga, nb, &full[s]);
  };

  if(lane == 0)
  {
    for(int s = 0; s < S; s++) ptx::mbar_init(&full[s], 1);
    ptx::fence_barrier_init();
    if(nv > 0)
      for(int f = 0; f < min(S - 1, nfr); f++) issue_load(f);
  }
  // transforms and root translations of the CTA's frames (shared by its 8 warps)
  for(int i = tid; i < nfr * kJoints * kXformFloats / 4; i += THREADS)
    reinterpret_cast<float4 *>(Gs)[i] = __ldg(reinterpret_cast<const float4 *>(xforms + static_cast<size_t>(b0) * kJoints * kXformFloats) + i);
  for(int i = tid; i < nfr * 3; i += THREADS)
  {
    const int f = i / 3, k = i - 3 * f;
    Tr[4 * f + k] = root ? root[static_cast<size_t>(b0 + f) * root_stride + k] : 0.f;
  }
  // per-lane group tables: union of the joints of the lane's 4 vertices + dense weights over it.  A group with more
  // than kGroupJoints distinct joints (nj < 0) takes the generic per-vertex path below.
  const int v = v0 + lane * VPL;
  const int nvalid = max(0, min(VPL, V - v));
  int nj = 0;
  float gw[kGroupJoints][VPL], iw[VPL];
  uint32_t joff[kGroupJoints];
#pragma unroll
  for(int u = 0; u < VPL; u++) iw[u] = 1.f;
#pragma unroll
  for(int k = 0; k < kGroupJoints; k++)
  {
    joff[k] = 0;
#pragma unroll
    for(int u = 0; u < VPL; u++) gw[k][u] = 0.f;
  }
  if(nvalid > 0)
  {
    const int g = v / VPL;
    nj = group_nj[g];
#pragma unroll
    for(int u = 0; u < VPL; u++) iw[u] = 1.f / lbs_wsum[min(v + u, V - 1)];
    if(nj >= 0)
    {
      const uint2 jj = __ldg(reinterpret_cast<const uint2 *>(group_joint + static_cast<size_t>(g) * kGroupJoints));
#pragma unroll
      for(int k = 0; k < kGroupJoints; k++)
      {
        if(k < nj)
        {
          joff[k] = (((k < 4 ? jj.x : jj.y) >> (8 * (k & 3))) & 0xffu) * (kXformFloats * 4);
          const float4 w = __ldg(reinterpret_cast<const float4 *>(group_w + (static_cast<size_t>(g) * kGroupJoints + k) * VPL));
          gw[k][0] = w.x, gw[k][1] = w.y, gw[k][2] = w.z, gw[k][3] = w.w;
        }
      }
    }
  }
  const bool any_generic = __any_sync(0xffffffffu, nj < 0);
  const int nj_max = __reduce_max_sync(0xffffffffu, max(nj, 0));
  __syncthreads();
  if(nv <= 0) return;

  const uint32_t gs_addr = ptx::smem_u32(Gs);
  const uint32_t ring_addr = ptx::smem_u32(ring);
  unsigned long long a = a0;
  for(int f = 0; f < nfr; f++, a += frame_bytes)
  {
    const int s = f % S;
    const uint32_t lo = static_cast<uint32_t>(a) & 15u;
    const unsigned long long ga = a - lo;
    const uint32_t need = lo + data_bytes;
    const uint32_t st_addr = ring_addr + s * STAGE_BYTES;
    uint8_t * stage = ring + s * STAGE_BYTES;
    ptx::mbar_wait(&full[s], (f / S) & 1);
    if(ga + ((need + 15u) & ~15u) > total_bytes)
    {
      // the very last chunk of the tensor: the aligned range would end past the allocation; fetch the tail words
      const uint32_t nb = static_cast<uint32_t>((total_bytes - ga) & ~15ull);
      for(uint32_t w = nb / 4 + lane; w < need / 4; w += 32)
        reinterpret_cast<float *>(stage)[w] = reinterpret_cast<const float *>(rest_b + ga)[w];
      __syncwarp();
    }
    // ---- this lane's 4 vertices: 48 bytes at stage + lo + 48 lane, skinned in place ----
    const uint32_t my = st_addr + lo + 48u * lane;
    const uint32_t gf = gs_addr + static_cast<uint32_t>(f) * (kJoints * kXformFloats * 4);
    const float tx = Tr[4 * f], ty = Tr[4 * f + 1], tz = Tr[4 * f + 2];
    switch(nj_max)
    {
      case 0:
      case 1: skin_in_place<1>(my, lo, gf, joff, gw, iw, tx, ty, tz); break;
      case 2: skin_in_place<2>(my, lo, gf, joff, gw, iw, tx, ty, tz); break;
      case 3: skin_in_place<3>(my, lo, gf, joff, gw, iw, tx, ty, tz); break;
      case 4: skin_in_place<4>(my, lo, gf, joff, gw, iw, tx, ty, tz); break;
      case 5: skin_in_place<5>(my, lo, gf, joff, gw, iw, tx, ty, tz); break;
      case 6: skin_in_place<6>(my, lo, gf, joff, gw, iw, tx, ty, tz); break;
      case 7: skin_in_place<7>(my, lo, gf, joff, gw, iw, tx, ty, tz); break;
      default: skin_in_place<8>(my, lo, gf, joff, gw, iw, tx, ty, tz); break;
    }
    if(any_generic && nj < 0)
    {
      // more than kGroupJoints distinct joints in the group: per-vertex influence slots, straight from the ELL tables
      for(int u = 0; u < nvalid; u++)
      {
        const uint32_t pv = my + 12u * u;
        // the in-place pass above wrote tx/ty/tz here (all weights zero); the rest position is re-read from global
        const float * rp = reinterpret_cast<const float *>(rest_b + a) + 3 * (lane * VPL + u);
        const float rx = rp[0], ry = rp[1], rz = rp[2];
        float ox = 0.f, oy = 0.f, oz = 0.f;
        for(int k = 0; k < kmax; k++)
        {
          const float w = lbs_weight[static_cast<size_t>(k) * Vpad + v + u];
          const uint32_t gj = gf + lbs_joint[static_cast<size_t>(k) * Vpad + v + u] * (kXformFloats * 4);
          const float4 r0 = ptx::lds128(gj), r1 = ptx::lds128(gj + 16), r2 = ptx::lds128(gj + 32);
          ox = fmaf(w, fmaf(r0.x, rx, fmaf(r0.y, ry, fmaf(r0.z, rz, r0.w))), ox);
          oy = fmaf(w, fmaf(r1.x, rx, fmaf(r1.y, ry, fmaf(r1.z, rz, r1.w))), oy);
          oz = fmaf(w, fmaf(r2.x, rx, fmaf(r2.y, ry, fmaf(r2.z, rz, r2.w))), oz);
        }
        ptx::sts32(pv, fmaf(ox, iw[u], tx));
        ptx::sts32(pv + 4, fmaf(oy, iw[u], ty));
        ptx::sts32(pv + 8, fmaf(oz, iw[u], tz));
      }
    }
    ptx::fence_proxy_async(); // generic-proxy writes -> visible to the bulk copy engine
    __syncwarp();
    // ---- drain: aligned interior by bulk copy, 8-byte head / tail by ordinary stores ----
    const uint32_t head = (16u - lo) & 15u;
    const uint32_t sa = lo + head;
    const uint32_t interior = (need - sa) & ~15u;
    const uint32_t tail = need - sa - interior;
    if(lane == 0)
    {
      if(interior) ptx::bulk_store_1d(out_b + ga + sa, st_addr + sa, interior);
      ptx::bulk_commit();
    }
    if(lane < head / 4) reinterpret_cast<float *>(out_b + a)[lane] = reinterpret_cast<const float *>(stage + lo)[lane];
    if(lane < tail / 4)
      reinterpret_cast<float *>(out_b + ga + sa + interior)[lane] = reinterpret_cast<const float *>(stage + sa + interior)[lane];
    // ---- refill the stage drained one iteration ago (frame f - 1) with frame f + S - 1 ----
    if(f + S - 1 < nfr)
    {
      if(lane == 0 && f >= 1) ptx::bulk_wait_read<1>(); // the store of frame f-1 no longer reads its stage
      __syncwarp();                                     // (also orders the other lanes' head/tail reads of that stage)
      if(lane == 0) issue_load(f + S - 1);
    }
  }
  if(lane == 0) ptx::bulk_wait_read<0>();
  __syncwarp();
}

namespace sb
{
namespace
{
constexpr int kFrc = 16, kStages = 4;
}

bool lbs_tma_usable(const ModelDev & d, const float * rest, const float * out, const float * xforms)
{
  return (d.V & 1) == 0 && d.group_nj && (reinterpret_cast<uintptr_t>(rest) & 15) == 0
         && (reinterpret_cast<uintptr_t>(out) & 15) == 0 && (reinterpret_cast<uintptr_t>(xforms) & 15) == 0 && rest != out;
}

int launch_lbs_tma(const ModelDev & d, cudaStream_t st, int B, const float * rest, const float * xforms, const float * root,
                   int root_stride, float * out)
{
  const int slices = (d.V + k3t::SLICE - 1) / k3t::SLICE;
  using L = k3t::Layout<kFrc, kStages>;
  SB_CUDA(cudaFuncSetAttribute(lbs_tma_kernel<kFrc, kStages>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::BYTES));
  dim3 grid((slices + k3t::WARPS - 1) / k3t::WARPS, (B + kFrc - 1) / kFrc);
  lbs_tma_kernel<kFrc, kStages><<<grid, k3t::THREADS, L::BYTES, st>>>(d.lbs_joint, d.lbs_weight, d.lbs_wsum, d.group_nj,
                                                                      d.group_joint, d.group_w, d.V, d.Vpad, d.kmax, B,
                                                                      rest, xforms, root, root_stride, out);
  SB_LAUNCHED();
  return SMPLPP_OK;
}
} // namespace sb
