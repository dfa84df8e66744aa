// K3'' : standalone linear blend skinning with the skinning matrices on tcgen05 (HBM-bound row of SURVEY.md §8d).
//
// Reference semantics: LinearBlendSkinning::skinning (src/LinearBlendSkinning.cpp:445-483) with cart2homo / homo2cart
// (:505-553): vert = (sum_j W[v,j] G'_j [rest_v; 1])[:3] / sum_j W[v,j] + root translation.
//
// The FFMA kernels (lbs_kernel, lbs_tma_kernel) spend ~44 FMAs per vertex and frame on forming
// sum_j W[v,j] G'_j and are bound by FFMA issue at ~3.2 TB/s.  Here M[v,f] = sum_j W[v,j] G'[f,j] is a GEMM on the
// tensor cores (128 vertices x (8 frames x 12), K = 24 -> 32, fp16 hi | lo split, three products, fp32 accumulate in
// TMEM; same operand split as skin_tc3.cu, skin_common.cuh) and the CUDA cores only apply M to the rest position:
// 12 FMAs per vertex and frame.
//
// CTA = 128 vertices x a chunk of frames, walked in 8-frame sub-batches:
//   warps 0, 18-20 producers (producer i owns sub-batches i, i+4, ...; lane t issues frame t's copy): per sub-batch one ring slot = the transforms (TMA tensor load, fp16 hi | lo, K-major) + the
//            8 rest rows of the tile (cp.async.bulk, 1536 contiguous bytes each; a frame is 82 680 B = 8 mod 16, so
//            the enclosing 16-byte aligned range is copied and the data sits at slot + lo, lo in {0, 8})
//   warp 1   MMA issuer: 6 tcgen05.mma (A = W tile in TMEM, written once by the epilogue threads) per sub-batch into one
//            of FIVE 96-column TMEM buffers, so the tensor pipe runs ahead of the epilogue
//   warps 2-17 epilogue: lane = vertex (TMEM lane); four groups of four warps (one per lane quadrant), group g owns the
//            sub-batches g, g+4, ... so that four sub-batches are in flight on the CUDA cores at any time (one warp's
//            serial latency per sub-batch is ~1500 cycles, the HBM budget ~1100): rest from the ring slot (ld.shared,
//            stride 12 B: conflict-free), M from TMEM, 12 FMAs, staged and written as 384 contiguous bytes per warp
//            and frame.
#include <cuda.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <mutex>

#include "forward.cuh"
#include "skin_common.cuh"
#include "tc_ptx.cuh"

using namespace sb;

namespace k3c
{
constexpr int MV = 128;
constexpr int SUBF = 8;                          // frames per sub-batch
constexpr int SUBN = SUBF * kXformFloats;        // 96 = UMMA N
constexpr int ROWB = 64;                         // 32 fp16 joints per K-major row (SWIZZLE_64B)
constexpr int G_PART = SUBN * ROWB;              // 6144
constexpr int REST_ROW = MV * 12 + 16;           // 1552: one frame's rest rows of the tile + misalignment room
constexpr int OFF_REST = 2 * G_PART;             // 12288
constexpr int SLOT = 25 * 1024;                  // 12288 + 8 * 1552 = 24704 -> 25600 (keeps G' 1024-byte aligned)
constexpr int RS = 8;                            // ring slots (8 x 24.7 KB of loads in flight per SM)
constexpr int MBUF = 5;                          // TMEM matrix buffers
constexpr int EPI_WARPS = 16;
constexpr int EPI_FR = 4;                         // frames per TMEM read (a warp walks its sub-batch in two halves)
constexpr int EPI_GROUPS = EPI_WARPS / 4;         // warp groups (one warp per lane quadrant); group g owns sub-batches g, g+4, ...
constexpr int PRODUCERS = 4;                      // TMA issue from one warp costs ~150 cycles per copy: 10 copies per sub-batch
constexpr int THREADS = 32 * (2 + EPI_WARPS + PRODUCERS - 1);
constexpr int STG_FLOATS = EPI_FR * 32 * 3;
constexpr int OFF_STG = RS * SLOT;
constexpr int OFF_BAR = OFF_STG + EPI_WARPS * STG_FLOATS * 4;
constexpr int SMEM_BYTES = 1024 + OFF_BAR + 256;
constexpr int TMEM_COLS = 512;
constexpr int COL_W = MBUF * SUBN;               // 480
static_assert(OFF_REST + SUBF * REST_ROW <= SLOT, "ring slot");
static_assert(COL_W + skin::KJ == TMEM_COLS, "TMEM column map");

struct Params
{
  int V, B, Bpad, chunk;        // chunk: frames per CTA (multiple of SUBF)
  float scale_m;                // 2^-(W_EXP + G_EXP)
  const float * weights;        // (V, 24) dense
  const float * wsum;           // (Vpad)
  const float * rest;           // (B, V, 3)
  const float * root;           // (B, root_stride) or null
  int root_stride;
  float * out;                  // (B, V, 3)
};
} // namespace k3c

// xforms (B,24,XF) fp32 (XF = 12: 3x4 rows, XF = 16: 4x4 whose bottom row is (0,0,0,1)) -> xf16 [part][Bpad*12][32] fp16
__global__ void split_xforms_kernel(const float * __restrict__ xforms, int xf_floats, int B, int Bpad, __half * __restrict__ xf16)
{
  const long long o = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long n_xf = static_cast<long long>(Bpad) * kXformFloats * skin::KJ;
  if(o >= n_xf) return;
  const int j = static_cast<int>(o % skin::KJ);
  const long long row = o / skin::KJ;
  const int e = static_cast<int>(row % kXformFloats);
  const long long f = row / kXformFloats;
  const float x = (f < B && j < kJoints) ? xforms[(f * kJoints + j) * xf_floats + e] * static_cast<float>(1 << skin::G_EXP) : 0.f;
  const __half hi = __float2half_rn(x);
  xf16[o] = hi;
  xf16[n_xf + o] = __float2half_rn(x - __half2float(hi));
}

__global__ void __launch_bounds__(k3c::THREADS, 1) lbs_tc_kernel(const __grid_constant__ CUtensorMap tmG, const k3c::Params p)
{
  using namespace k3c;
  extern __shared__ uint8_t smem_raw[];
  uint8_t * smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float * stg = reinterpret_cast<float *>(smem + OFF_STG);
  uint64_t * bars = reinterpret_cast<uint64_t *>(smem + OFF_BAR);
  uint64_t * s_full = bars;              // [RS]    TMA -> MMA + epilogue
  uint64_t * s_empty = s_full + RS;      // [RS]    MMA (commit) + the 4 warps of the owning group -> TMA
  uint64_t * m_full = s_empty + RS;      // [MBUF]  MMA -> epilogue
  uint64_t * m_empty = m_full + MBUF;    // [MBUF]  epilogue -> MMA
  uint64_t * w_ready = m_empty + MBUF;   //         epilogue -> MMA (W tile stored in TMEM)
  uint32_t * tmem_slot = reinterpret_cast<uint32_t *>(w_ready + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = blockIdx.y;
  const int f0 = blockIdx.x * p.chunk;
  const int nfr = min(p.chunk, p.B - f0);
  const int nsub = (nfr + SUBF - 1) / SUBF;
  const int v0 = tile * MV;
  const int nv = min(MV, p.V - v0);
  const unsigned long long total_bytes = static_cast<unsigned long long>(p.B) * p.V * 12ull;
  const unsigned long long frame_bytes = static_cast<unsigned long long>(p.V) * 12ull;
  const uint32_t data_bytes = static_cast<uint32_t>(nv) * 12u;

  if(warp == 0 && lane == 0)
  {
    ptx::prefetch_tensormap(&tmG);
    for(int s = 0; s < RS; s++)
    {
      ptx::mbar_init(&s_full[s], 1);
      ptx::mbar_init(&s_empty[s], 1 + 4);
    }
    for(int i = 0; i < MBUF; i++)
    {
      ptx::mbar_init(&m_full[i], 1);
      ptx::mbar_init(&m_empty[i], 4);
    }
    ptx::mbar_init(w_ready, 4);
    ptx::fence_barrier_init();
  }
  if(warp == 1) ptx::tmem_alloc<TMEM_COLS>(tmem_slot);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if(warp == 0 || warp >= 2 + EPI_WARPS)
  {
    // producers (warp 0 and the last three warps; producer i owns the sub-batches i, i + 4, ...: issuing the 10 copies
    // of a sub-batch from one warp costs more than the ~1100-cycle HBM budget of a sub-batch): lane t issues the bulk
    // copy of frame t (address arithmetic in parallel), lane 0 the barrier bookkeeping and the transforms' tensor loads
    const int prod = warp == 0 ? 0 : warp - (1 + EPI_WARPS);
    const uint8_t * rest_b = reinterpret_cast<const uint8_t *>(p.rest);
    for(int sb = prod; sb < nsub; sb += PRODUCERS)
    {
      const int s = sb % RS;
      if(lane == 0) ptx::mbar_wait(&s_empty[s], ((sb / RS) & 1) ^ 1);
      __syncwarp();
      uint8_t * slot = smem + s * SLOT;
      const int fa = f0 + sb * SUBF;
      const int live = min(SUBF, p.B - fa);
      // enclosing 16-byte aligned range of this lane's frame, clipped to the tensor
      unsigned long long ga = 0;
      uint32_t nb = 0;
      if(lane < live)
      {
        const unsigned long long a = (static_cast<unsigned long long>(fa + lane) * p.V + v0) * 12ull;
        const uint32_t lo = static_cast<uint32_t>(a) & 15u;
        ga = a - lo;
        nb = static_cast<uint32_t>(min(static_cast<unsigned long long>((lo + data_bytes + 15u) & ~15u), (total_bytes - ga) & ~15ull));
      }
      const uint32_t tx = 2 * G_PART + __reduce_add_sync(0xffffffffu, nb);
      if(lane == 0)
      {
        ptx::mbar_expect_tx(&s_full[s], tx);
#pragma unroll
        for(int part = 0; part < 2; part++)
          ptx::tma_load_2d(slot + part * G_PART, &tmG, 0, (part * p.Bpad + fa) * kXformFloats, &s_full[s]);
      }
      __syncwarp();
      if(lane < live) ptx::bulk_load_1d(slot + OFF_REST + lane * REST_ROW, rest_b + ga, nb, &s_full[s]);
    }
  }
  else if(warp == 1)
  {
    if(ptx::elect_one())
    {
      constexpr uint32_t idesc = ptx::make_idesc_f16(MV, SUBN);
      ptx::mbar_wait(w_ready, 0);
      ptx::tc_fence_after();
      for(int sb = 0; sb < nsub; sb++)
      {
        const int s = sb % RS, b = sb % MBUF;
        ptx::mbar_wait(&s_full[s], (sb / RS) & 1);
        ptx::mbar_wait(&m_empty[b], ((sb / MBUF) & 1) ^ 1);
        ptx::tc_fence_after();
        const uint32_t sg = ptx::smem_u32(smem + s * SLOT);
#pragma unroll
        for(int prod = 0; prod < 3; prod++)
        {
          const int pa = prod == 1 ? 1 : 0, pb = prod == 2 ? 1 : 0; // hi.hi, lo.hi, hi.lo
#pragma unroll
          for(int ks = 0; ks < 2; ks++)
          {
            const uint64_t bdesc = ptx::make_smem_desc<ROWB>(sg + pb * G_PART + ks * 32);
            ptx::umma_f16_ts(tmem_base + b * SUBN, tmem_base + COL_W + pa * (skin::KJ / 2) + ks * 8, bdesc, idesc,
                             (prod | ks) != 0 ? 1u : 0u);
          }
        }
        ptx::tc_commit(&s_empty[s]); // the transforms of the slot are consumed once these MMAs have completed
        ptx::tc_commit(&m_full[b]);
      }
    }
  }
  else
  {
    const int ew = warp - 2;
    const int q = warp & 3;  // TMEM lane quadrant (hardware rule: warp id % 4)
    const int grp = ew >> 2; // warp group: owns sub-batches grp, grp + 4, ... (all 8 frames, in two halves of 4)
    const int wv0 = v0 + q * 32;
    const int v = wv0 + lane;
    const int vc = min(v, p.V - 1);
    const int nvalid = max(0, min(32, p.V - wv0));
    const uint32_t lane_taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    if(ew < 4)
    {
      skin::store_w_row_tmem(p.weights + static_cast<size_t>(vc) * kJoints, lane_taddr + COL_W);
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if(lane == 0) ptx::mbar_arrive(w_ready);
    }
    const float sm = p.scale_m / p.wsum[vc]; // homogeneous divide (LinearBlendSkinning.cpp:545-550) folded into the scale
    const uint32_t my_stg = ptx::smem_u32(stg + ew * STG_FLOATS);
    // everything that does not depend on the sub-batch is computed once
    const uint32_t row0 = ptx::smem_u32(smem) + OFF_REST + static_cast<uint32_t>(q * 32 + lane) * 12u;
    const uint32_t lo0 = static_cast<uint32_t>((static_cast<unsigned long long>(f0) * p.V + v0) * 12ull) & 15u;
    const uint32_t dlo = static_cast<uint32_t>(frame_bytes) & 15u; // misalignment step per frame (8 for SMPL)
    // only the CTA that owns the last rows of the tensor can see a clipped bulk copy
    const bool may_clip = (tile == static_cast<int>(gridDim.y) - 1) && (f0 + nfr == p.B);
    constexpr int NST = EPI_FR * 48 / 32; // float2 stores per lane and half
    int st_ofs[NST], st_t[NST];
    bool st_ok[NST];
#pragma unroll
    for(int i = 0; i < NST; i++)
    {
      const int idx = 32 * i + lane; // float2 index over EPI_FR frames x 48
      st_t[i] = idx / 48;
      const int w2 = idx - 48 * st_t[i];
      st_ofs[i] = st_t[i] * (p.V * 3 / 2) + w2; // in float2 units from the half's first frame (V is even)
      st_ok[i] = 2 * w2 < 3 * nvalid;
    }

    for(int sb = grp; sb < nsub; sb += EPI_GROUPS)
    {
      const int s = sb % RS, b = sb % MBUF;
      ptx::mbar_wait(&s_full[s], (sb / RS) & 1);
      // rest positions of this vertex for all 8 frames -> registers, then the slot goes straight back to the producer
      // (memory-level parallelism: a slot held through the whole visit left only ~4 slots of loads in flight per SM)
      float r[SUBF][3];
#pragma unroll
      for(int t = 0; t < SUBF; t++)
      {
        // the frame's rows sit at slot + lo (lo = misalignment of the frame's chunk)
        const uint32_t lo = (lo0 + static_cast<uint32_t>(sb * SUBF + t) * dlo) & 15u;
        const uint32_t addr = row0 + s * SLOT + t * REST_ROW + lo;
        r[t][0] = ptx::lds32(addr), r[t][1] = ptx::lds32(addr + 4), r[t][2] = ptx::lds32(addr + 8);
      }
      if(may_clip && f0 + sb * SUBF + SUBF > p.B - 1 && v < p.V)
      {
        // the very last rows of the tensor: the aligned bulk copy stops short of the allocation's end
        const int t = p.B - 1 - (f0 + sb * SUBF);
        if(t >= 0 && t < SUBF)
        {
          const unsigned long long a = (static_cast<unsigned long long>(p.B - 1) * p.V + v0) * 12ull;
          const uint32_t lo = static_cast<uint32_t>(a) & 15u;
          const uint32_t nb = static_cast<uint32_t>((total_bytes - (a - lo)) & ~15ull);
          const uint32_t off = lo + static_cast<uint32_t>(q * 32 + lane) * 12u;
#pragma unroll
          for(int tt = 0; tt < SUBF; tt++)
#pragma unroll
            for(int k = 0; k < 3; k++)
              if(tt == t && off + 4u * k + 4u > nb) r[tt][k] = p.rest[(static_cast<size_t>(p.B - 1) * p.V + v) * 3 + k];
        }
      }
      __syncwarp();
      if(lane == 0) ptx::mbar_arrive(&s_empty[s]);
      bool m_ready = false;
#pragma unroll
      for(int half = 0; half < SUBF / EPI_FR; half++)
      {
        const int fl = sb * SUBF + half * EPI_FR; // first frame of the half within the chunk
        float tr[EPI_FR][3];
#pragma unroll
        for(int t = 0; t < EPI_FR; t++)
        {
          tr[t][0] = tr[t][1] = tr[t][2] = 0.f;
          if(p.root && fl + t < nfr)
          {
            const float * trp = p.root + static_cast<size_t>(f0 + fl + t) * p.root_stride;
            tr[t][0] = __ldg(trp), tr[t][1] = __ldg(trp + 1), tr[t][2] = __ldg(trp + 2);
          }
        }
        // ---- skinning matrices of the half's four frames ----
        if(!m_ready)
        {
          ptx::mbar_wait(&m_full[b], (sb / MBUF) & 1);
          ptx::tc_fence_after();
          m_ready = true;
        }
        float M[EPI_FR * kXformFloats];
        const uint32_t mcol = lane_taddr + b * SUBN + half * (EPI_FR * kXformFloats);
        ptx::tmem_ld_x16(mcol, M);
        ptx::tmem_ld_x16(mcol + 16, M + 16);
        ptx::tmem_ld_x16(mcol + 32, M + 32);
        ptx::tmem_ld_wait();
        if(half == SUBF / EPI_FR - 1)
        {
          ptx::tc_fence_before();
          __syncwarp();
          if(lane == 0) ptx::mbar_arrive(&m_empty[b]);
        }
#pragma unroll
        for(int t = 0; t < EPI_FR; t++)
        {
          const float * m = M + kXformFloats * t;
          const float * rr = r[half * EPI_FR + t];
          const float ox = fmaf(m[0], rr[0], fmaf(m[1], rr[1], fmaf(m[2], rr[2], m[3])));
          const float oy = fmaf(m[4], rr[0], fmaf(m[5], rr[1], fmaf(m[6], rr[2], m[7])));
          const float oz = fmaf(m[8], rr[0], fmaf(m[9], rr[1], fmaf(m[10], rr[2], m[11])));
          const uint32_t sa = my_stg + (t * 96 + lane * 3) * 4;
          ptx::sts32(sa, fmaf(ox, sm, tr[t][0]));
          ptx::sts32(sa + 4, fmaf(oy, sm, tr[t][1]));
          ptx::sts32(sa + 8, fmaf(oz, sm, tr[t][2]));
        }
        __syncwarp();
        float2 * out_h = reinterpret_cast<float2 *>(p.out + (static_cast<size_t>(f0 + fl) * p.V + wv0) * 3);
#pragma unroll
        for(int i = 0; i < NST; i++)
        {
          const float2 val = ptx::lds64(my_stg + (32 * i + lane) * 8);
          if(st_ok[i] && fl + st_t[i] < nfr) __stcs(out_h + st_ofs[i], val);
        }
        __syncwarp();
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if(warp == 1) ptx::tmem_dealloc<TMEM_COLS>(tmem_base);
}

namespace sb
{
EncodeTiledFn encode_fn()
{
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void * p = nullptr;
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    if(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess
       && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
    else
      cudaGetLastError();
  });
  return fn;
}

bool lbs_tc_usable(const ModelDev & d, const float * rest, const float * out, const float * xforms)
{
  return d.tc3_ready && (d.V & 1) == 0 && d.V >= k3c::MV && (reinterpret_cast<uintptr_t>(rest) & 15) == 0
         && (reinterpret_cast<uintptr_t>(out) & 7) == 0 && (reinterpret_cast<uintptr_t>(xforms) & 15) == 0 && rest != out
         && encode_fn() != nullptr;
}

// xf_floats: 12 (affine 3x4) or 16 (4x4 with bottom row (0,0,0,1))
int launch_lbs_tc(const ModelDev & d, cudaStream_t st, int B, const float * rest, const float * xforms, int xf_floats,
                  const float * root, int root_stride, float * out)
{
  static bool configured[64] = {};
  if(first_call_on_device(configured))
  {
    SB_CUDA(cudaFuncSetAttribute(lbs_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, k3c::SMEM_BYTES));
    // the per-call transform scratch comes from the stream-ordered pool: keep freed blocks cached across synchronisations
    int dev = 0;
    cudaMemPool_t pool = nullptr;
    if(cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess)
    {
      uint64_t keep = 1ull << 30;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaGetLastError();
  }
  const int Bpad = static_cast<int>(align_up(static_cast<size_t>(B), k3c::SUBF));
  const size_t xf_bytes = static_cast<size_t>(2) * Bpad * kXformFloats * skin::KJ * sizeof(__half);
  void * xf16 = nullptr;
  SB_CUDA(cudaMallocAsync(&xf16, xf_bytes, st)); // stream-ordered scratch: the entry point has no workspace argument
  const long long n = static_cast<long long>(Bpad) * kXformFloats * skin::KJ;
  split_xforms_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(xforms, xf_floats, B, Bpad, static_cast<__half *>(xf16));
  SB_LAUNCHED();
  alignas(64) CUtensorMap tmG;
  {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(skin::KJ), static_cast<cuuint64_t>(2) * Bpad * kXformFloats};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(skin::KJ) * 2};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(skin::KJ), static_cast<cuuint32_t>(k3c::SUBN)};
    cuuint32_t estr[2] = {1, 1};
    if(encode_fn()(&tmG, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, xf16, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE)
       != CUDA_SUCCESS)
    {
      cudaFreeAsync(xf16, st);
      return fail(SMPLPP_ERR_CUDA, "CUDA", "cuTensorMapEncodeTiled failed for the skinning transforms");
    }
  }
  const int ntiles = (d.V + k3c::MV - 1) / k3c::MV;
  // frames per CTA: long chunks (the TMEM / W-tile set-up is paid once per CTA) sized so that the grid fills whole waves
  int sms = 148;
  {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  }
  const int want = std::max(1, (B + 511) / 512);                                   // ~512 frames per CTA
  const int waves = std::max(1, (ntiles * want + sms - 1) / sms);
  int nchunks = std::max(1, std::min((waves * sms) / ntiles, (B + k3c::SUBF - 1) / k3c::SUBF));
  int chunk = static_cast<int>(align_up(static_cast<size_t>((B + nchunks - 1) / nchunks), k3c::SUBF));
  nchunks = (B + chunk - 1) / chunk;
  k3c::Params p;
  p.V = d.V;
  p.B = B;
  p.Bpad = Bpad;
  p.chunk = chunk;
  p.scale_m = ldexpf(1.f, -(skin::W_EXP + skin::G_EXP));
  p.weights = d.weights_dense;
  p.wsum = d.lbs_wsum;
  p.rest = rest;
  p.root = root;
  p.root_stride = root_stride;
  p.out = out;
  lbs_tc_kernel<<<dim3(nchunks, ntiles), k3c::THREADS, k3c::SMEM_BYTES, st>>>(tmG, p);
  SB_LAUNCHED();
  SB_CUDA(cudaFreeAsync(xf16, st));
  return SMPLPP_OK;
}
} // namespace sb
