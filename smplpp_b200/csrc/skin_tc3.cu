// K2''' (tcgen05, persistent + pipelined): fused blend-shape contraction + linear blend skinning, both products on the
// tensor cores, with the contraction of work item i+1 running UNDER the skinning GEMM + epilogue of work item i.
//
// Reference semantics: BlendShape::poseBlend / shapeBlend (src/BlendShape.cpp:764, 670-683), the rest shape
// T + S + P (src/JointRegression.cpp:551-565) and LinearBlendSkinning::skinning (src/LinearBlendSkinning.cpp:445-553).
//
//   rest[v,f]   = T[v] + sum_k basis[v,k] coef[f,k]                 GEMM 1: (128 vertices x 3 planes) x 96 frames, K = 224
//   M[v,f]      = sum_j W[v,j] G'[f,j]  (3x4 per vertex and frame)  GEMM 2: 128 vertices x (8 frames x 12), K = 16 or 32
//   vert[v,f]   = M[v,f] [rest; 1] / sum_j W[v,j] + trans[f]        epilogue: 12 FMA per vertex and frame
//
// Work and pipeline (DESIGN.md 4.1 has the measurements):
//   * one persistent CTA per SM walks a contiguous range of (vertex tile, frame block) work items;
//   * when GEMM 1 of an item completes, the sixteen epilogue warps DRAIN its 288 accumulator columns into registers
//     (72 per thread, pre-scaled by 1 / sum_j W), which frees the TMEM columns: one thread then issues the 126 MMAs of
//     the NEXT item's GEMM 1 while another issues the 12 sub-batches of this item's GEMM 2;
//   * joint windows: the model's 24 joints are covered by two 16-slot windows (chosen from its weights at create time).
//     A vertex tile whose joints all sit in one window runs GEMM 2 at K = 16 (3 MMAs per sub-batch, 6 KB of transforms);
//     any other tile runs both windows (6 MMAs, 12 KB), its weights in each joint's primary slot only.  Exact: the
//     dropped products multiply zero weights;
//   * two TMA producer threads, one per ring (2 x 60 KB GEMM 1 stages, 6 x 6 KB transform window slots), so neither
//     ring can starve the other;
//   * the frames of a 96-frame block are permuted in the fp16 coefficient operand so that the 24 frames an epilogue
//     warp owns are 24 adjacent accumulator columns (6 tcgen05.ld per drain instead of 36).
//   * every operand tile is stored in global memory as the exact (SWIZZLE_64B) shared-memory image of its pipeline
//     stage, so a stage is two contiguous cp.async.bulk copies (48 KB basis + 12 KB coefficients) and a transform
//     sub-batch is one (6 or 12 KB, SWIZZLE_32B): no tensor maps, a handful of large copies per item.
// Precision: both GEMMs are fp32 in the reference.  Every operand is split into fp16 hi + lo (power-of-two pre-scaled
// so that lo stays a normal fp16) and three products are accumulated in fp32 TMEM, hi.hi + lo.hi + hi.lo (~2^-22
// relative).  The ~1 m template stays out of GEMM 1 and is added in fp32.
//
// TMEM (512 columns): [0,288) rest accumulators (x | y | z planes x 96 frames), [288,480) two 96-column buffers of
// skinning matrices (8 frames x 12), [480,512) the W tile (A operand of GEMM 2: window w at 480 + 16 w, fp16 hi | lo).
// warp 0: TMA producer of the GEMM 1 stages | warp 1: TMEM allocator + issuer of GEMM 2 | warp 2: TMA producer of the transform
// sub-batches | warp 3: issuer of GEMM 1 (the first warpgroup hands its registers back with setmaxnreg) | warps 4-19: epilogue,
// 112 registers each (four per TMEM lane quadrant, one per frame pair of an 8-frame sub-batch).
#include <cuda.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <vector>

#include "forward.cuh"
#include "skin_common.cuh"
#include "tc3_layout.cuh"
#include "tc_ptx.cuh"

using namespace sb;

namespace tc3
{
struct Params
{
  int V, B, Bpad, ntiles, nfb, nitems;
  float scale_p, scale_m;       // 2^-(basis_exp + COEF_EXP), 2^-(W_EXP + G_EXP)
  const uint8_t * img_a;        // [tile][K-block][part][plane][128][64 B]   stage image of the fp16 basis
  const uint8_t * img_b;        // [frame block][K-block][part][96][64 B]   stage image of the fp16 coefficients
  const uint8_t * img_g;        // [frame block][sub-batch][window][part][96][32 B] stage image of the fp16 transforms
  const uint8_t * tile_mode;    // (ntiles) 0 / 1: the tile's joints fit window 0 / 1, 2: both windows
  const float * basis;          // (3 Vpad, 224): column 217 = template
  const float * weights;        // (V, 24) dense
  const float * wsum;           // (Vpad)
  const float * theta;          // (B, 25, 3): row 0 = root translation
  float * out;                  // (B, V, 3)
  WindowMap wmap;               // transform-image slot -> joint
  uint32_t primary;             // bit s: slot s is the primary slot of its joint (W tile of a both-window tile)
};

// One vertex's row of the dense skinning weights -> the W tile (A operand of GEMM 2) in TMEM: lane = vertex, window w
// at taddr + 16 w (8 hi | 8 lo packed fp16x2 columns).  A window tile (mode 0 / 1) writes its window's joints; a
// both-window tile (mode 2) puts every joint in its primary slot only, so a joint of both windows counts once.  The
// caller follows with tmem_st_wait + tcgen05.fence::before_thread_sync before signalling the MMA warp.
__device__ __forceinline__ void store_w_windows(const float * __restrict__ wrow, uint32_t taddr, const WindowMap wmap,
                                                uint32_t primary, int mode)
{
  uint32_t c[NWIN][KW]; // [window][hi 8 | lo 8]
#pragma unroll
  for(int i = 0; i < KJ / 2; i++)
  {
    float x[2];
#pragma unroll
    for(int h = 0; h < 2; h++)
    {
      const int s = 2 * i + h, j = wmap.joint[s];
      const bool keep = j >= 0 && (mode == 2 ? ((primary >> s) & 1u) != 0 : s / KW == mode);
      x[h] = keep ? __ldg(wrow + (j < 0 ? 0 : j)) * static_cast<float>(1 << W_EXP) : 0.f;
    }
    const float ah = __half2float(__float2half_rn(x[0])), bh = __half2float(__float2half_rn(x[1]));
    c[i / (KW / 2)][i % (KW / 2)] = skin::pack_half2(ah, bh);
    c[i / (KW / 2)][KW / 2 + i % (KW / 2)] = skin::pack_half2(x[0] - ah, x[1] - bh);
  }
  ptx::tmem_st_x16(taddr, c[0]);
  ptx::tmem_st_x16(taddr + KW, c[1]);
}

} // namespace tc3

// basis (3 Vpad, 224) fp32 -> stage images [tile][K-block][part hi | lo][plane][128 rows][32 fp16], scaled by 2^e
__global__ void basis_image_f16_kernel(const float * __restrict__ basis, int V, int ntiles, float scale, uint8_t * __restrict__ img)
{
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long n = static_cast<long long>(ntiles) * 3 * tc3::MV * tc3::KP;
  if(i >= n) return;
  const int k = static_cast<int>(i % tc3::KP);
  const long long row = i / tc3::KP;
  const int r = static_cast<int>(row % tc3::MV);
  const int plane = static_cast<int>((row / tc3::MV) % 3);
  const int tile = static_cast<int>(row / (3 * tc3::MV));
  const int v = tile * tc3::MV + r;
  const float x = (v < V && k < tc3::KUSED) ? basis[(static_cast<size_t>(3) * v + plane) * kBlendK + k] * scale : 0.f;
  const __half hi = __float2half_rn(x);
  const __half lo = __float2half_rn(x - __half2float(hi));
  uint8_t * blk = img + (static_cast<size_t>(tile) * tc3::NKB + k / 32) * (2 * tc3::A_PART);
  const uint32_t o = static_cast<uint32_t>(plane * tc3::MV * tc3::ROWB + r * tc3::ROWB + (k % 32) * 2);
  *reinterpret_cast<__half *>(blk + tc3::swz64(o)) = hi;
  *reinterpret_cast<__half *>(blk + tc3::swz64(tc3::A_PART + o)) = lo;
}

// per-call operands: coef (B,224) fp32 -> img_b (rows of every 96-frame block permuted by coef_row, x 2^6);
// xforms (B,24,12) fp32 -> img_g (row = frame in sub-batch * 12 + element of the 3x4, column = joint slot of the two
// windows, x 2^4).  Padding (frames >= B, K >= 217, empty slots) is zero-filled.  One thread per 16-byte chunk (8 fp16 of one row:
// the swizzle moves whole chunks), hi and lo written as one 16-byte store each.
__global__ void frame_images3_kernel(const float * __restrict__ coef, const float * __restrict__ xforms, int B, int Bpad,
                                     uint8_t * __restrict__ img_b, uint8_t * __restrict__ img_g, const tc3::WindowMap wmap)
{
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  constexpr int CK = tc3::KP / 8;   // 28 chunks per coefficient row
  constexpr int CJ = tc3::KJ / 8;   // 4 chunks per transform row
  const long long n_coef = static_cast<long long>(Bpad) * CK;
  const long long n_xf = static_cast<long long>(Bpad) * kXformFloats * CJ;
  float x[8];
  if(i < n_coef)
  {
    const int ck = static_cast<int>(i % CK);
    const long long f = i / CK;
    if(f < B)
    {
      const float4 a = __ldg(reinterpret_cast<const float4 *>(coef + f * tc3::KP + ck * 8));
      const float4 b = __ldg(reinterpret_cast<const float4 *>(coef + f * tc3::KP + ck * 8 + 4));
      x[0] = a.x, x[1] = a.y, x[2] = a.z, x[3] = a.w, x[4] = b.x, x[5] = b.y, x[6] = b.z, x[7] = b.w;
    }
#pragma unroll
    for(int e = 0; e < 8; e++) x[e] = (f < B && ck * 8 + e < tc3::KUSED) ? x[e] * static_cast<float>(1 << tc3::COEF_EXP) : 0.f;
    const long long fb = f / tc3::NF;
    const int r = tc3::coef_row(static_cast<int>(f - fb * tc3::NF));
    uint8_t * blk = img_b + (static_cast<size_t>(fb) * tc3::NKB + ck / 4) * (2 * tc3::B_PART);
    const uint32_t o = static_cast<uint32_t>(r * tc3::ROWB + (ck % 4) * 16);
    tc3::split8_store(x, blk + tc3::swz64(o), blk + tc3::swz64(tc3::B_PART + o));
  }
  else if(i < n_coef + n_xf)
  {
    const long long q = i - n_coef;
    const int cj = static_cast<int>(q % CJ);
    const long long row = q / CJ;
    const int e = static_cast<int>(row % kXformFloats);
    const long long f = row / kXformFloats;
    int js[8];
    tc3::chunk_joints(wmap, cj, js);
#pragma unroll
    for(int jj = 0; jj < 8; jj++)
      x[jj] = (f < B && js[jj] >= 0)
                  ? __ldg(xforms + (f * kJoints + (js[jj] < 0 ? 0 : js[jj])) * kXformFloats + e) * static_cast<float>(1 << tc3::G_EXP)
                  : 0.f;
    uint8_t * dst = img_g + tc3::g_chunk_offset(f, e, cj);
    tc3::split8_store(x, dst, dst + tc3::G_PART);
  }
}

template<int STAGES, int GSLOTS>
__global__ void __launch_bounds__(tc3::THREADS, 1)
    blend_skin_tc3_kernel(const tc3::Params p)
{
  using namespace tc3;
  using L = Layout<STAGES, GSLOTS>;
  constexpr int OFF_G = L::OFF_G, OFF_BAR = L::OFF_BAR;
  extern __shared__ uint8_t smem_raw[];
  uint8_t * smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t * bars = reinterpret_cast<uint64_t *>(smem + OFF_BAR);
  // the same base as a 32-bit shared-window address, aligned in that space (the window base is itself 1 KB aligned): the
  // hot loops address stages and barriers as smem32 + constant instead of converting a generic pointer at every use
  const uint32_t smem32 = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar32 = smem32 + OFF_BAR;
  uint64_t * full = bars;                // [STAGES]  TMA -> MMA (GEMM 1 stages)
  uint64_t * empty = full + STAGES;      // [STAGES]  MMA -> TMA
  uint64_t * g_full = empty + STAGES;    // [GSLOTS]  TMA -> MMA (transform windows of a sub-batch)
  uint64_t * g_empty = g_full + GSLOTS;  // [GSLOTS]  MMA -> TMA
  uint64_t * m_full = g_empty + GSLOTS;  // [2]       MMA -> epilogue (skinning matrices of a sub-batch)
  uint64_t * m_empty = m_full + 2;       // [2]       epilogue -> MMA
  uint64_t * p_full = m_empty + 2;       //           MMA -> epilogue (rest accumulators of an item complete)
  uint64_t * rest_free = p_full + 1;     //           epilogue -> MMA (accumulators drained into registers)
  uint64_t * w_ready = rest_free + 1;    //           epilogue -> MMA (W tile stored in TMEM)
  uint32_t * tmem_slot = reinterpret_cast<uint32_t *>(w_ready + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // contiguous range of work items, vertex tile major / frame block minor: a CTA changes its vertex tile (W tile,
  // template, 1 / sum w) at most a couple of times
  const int it0 = static_cast<int>(static_cast<long long>(blockIdx.x) * p.nitems / gridDim.x);
  const int it1 = static_cast<int>(static_cast<long long>(blockIdx.x + 1) * p.nitems / gridDim.x);
  const int nit = it1 - it0;

  if(warp == 0 && lane == 0)
  {
    for(int s = 0; s < STAGES; s++)
    {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for(int s = 0; s < GSLOTS; s++)
    {
      ptx::mbar_init(&g_full[s], 1);
      ptx::mbar_init(&g_empty[s], 1);
    }
    for(int i = 0; i < 2; i++)
    {
      ptx::mbar_init(&m_full[i], 1);
      ptx::mbar_init(&m_empty[i], EPI_WARPS);
    }
    ptx::mbar_init(p_full, 1);
    ptx::mbar_init(rest_free, EPI_WARPS);
    ptx::mbar_init(w_ready, 4);
    ptx::fence_barrier_init();
  }
  if(warp == 1) ptx::tmem_alloc<TMEM_COLS>(tmem_slot);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if(warp < CTRL_WARPS)
  {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
  if(warp == 0)
  {
    // ---- producer of the GEMM 1 stage ring ----
    // (Measured, scripts/ubench/ubench_tma.cu: [expect_tx, copy] groups issued back to back by ONE thread onto different
    // barriers retire ~410 cycles apart whatever their size, so a group is as large as a stage, and each ring has its own
    // producer thread with plain blocking waits.  A single polling producer over both rings performed the same.)
    if(ptx::elect_one())
    {
      const int total_kb = nit * NKB;
      // (An L2 prefetch of all seven K-blocks of the first item at kernel start was measured: no gain.)
      // The reload of a stage is on the critical path of the GEMM 1 issuer (a quarter of its samples are stage waits):
      // source addresses (two integer divisions) are ready BEFORE the wait, barriers and stages are 32-bit shared addresses.
      int kb = 0, tile = it0 / p.nfb, fb = it0 % p.nfb;
      for(int kbn = 0; kbn < total_kb; kbn++)
      {
        const uint32_t s = static_cast<uint32_t>(kbn % STAGES);
        const uint8_t * srca = p.img_a + (static_cast<size_t>(tile) * NKB + kb) * (2 * A_PART);
        const uint8_t * srcb = p.img_b + (static_cast<size_t>(fb) * NKB + kb) * (2 * B_PART);
        const uint32_t dst = smem32 + s * STAGE, fbar = bar32 + 8 * s;
        ptx::mbar_wait_a(bar32 + 8 * (STAGES + s), ((kbn / STAGES) & 1) ^ 1);
        ptx::mbar_expect_tx_a(fbar, STAGE);
        ptx::bulk_load_1d_a(dst, srca, 2 * A_PART, fbar);
        ptx::bulk_load_1d_a(dst + 2 * A_PART, srcb, 2 * B_PART, fbar);
        if(++kb == NKB)
        {
          kb = 0;
          if(++fb == p.nfb) fb = 0, tile++;
        }
      }
    }
  }
  else if(warp == 2)
  {
    // ---- producer of the transform ring: per sub-batch one 6 KB entry (the tile's window) or, for a both-window
    //      tile, two consecutive entries filled by ONE 12 KB copy signalled on the first (the second barrier gets a
    //      plain arrival so that every entry completes one phase) ----
    if(ptx::elect_one())
    {
      int gn = 0, fb = it0 % p.nfb, tile = it0 / p.nfb;
      for(int k = 0; k < nit; k++)
      {
        const int mode = p.tile_mode[tile], nw = mode == 2 ? 2 : 1;
        const uint8_t * src = p.img_g + static_cast<size_t>(fb) * NSUB * G_SUB + (mode == 1 ? G_WIN : 0);
        for(int sb = 0; sb < NSUB; sb++, gn += nw)
        {
          const uint32_t s = static_cast<uint32_t>(gn % GSLOTS), par = ((gn / GSLOTS) & 1) ^ 1;
          const uint32_t fbar = bar32 + 8 * (2 * STAGES + s), ebar = bar32 + 8 * (2 * STAGES + GSLOTS + s);
          ptx::mbar_wait_a(ebar, par);
          if(nw == 2) ptx::mbar_wait_a(ebar + 8, par);
          ptx::mbar_expect_tx_a(fbar, nw * G_WIN);
          ptx::bulk_load_1d_a(smem32 + OFF_G + s * G_WIN, src + static_cast<size_t>(sb) * G_SUB, nw * G_WIN, fbar);
          if(nw == 2) ptx::mbar_arrive_a(fbar + 8);
        }
        if(++fb == p.nfb) fb = 0, tile++;
      }
    }
  }
  else if(warp == 1 || warp == 3)
  {
    if(ptx::elect_one())
    {
      constexpr uint32_t idesc1 = ptx::make_idesc_f16(MV, NF);
      constexpr uint32_t idesc2 = ptx::make_idesc_f16(MV, SUBN);
      // Every instruction between two tcgen05.mma is on the critical path of its issuing thread.  ncu's source page of the
      // single-issuer version (r02h) had that thread at 1800 instructions per item for 198 MMAs and blocked on a full
      // tensor queue in only a quarter of its samples: the tensor pipe starved behind the issue loop.  Hence (a) TWO
      // issuing threads - warp 3 the 126 GEMM 1 MMAs of the next item, warp 1 the 36 (window tile) or 72 (both-window
      // tile) GEMM 2 MMAs of this one; the tensor
      // queue interleaves them (0.1725 -> 0.1607 ms per launch) - and (b) lean streams: the sub-batches and half K-blocks
      // are unrolled, so that ring slots, parities and operand offsets are compile-time constants; only the stage of a
      // K-block (ring position over all items) and the item parity are run-time values, and barriers are 32-bit shared
      // addresses.  Descriptor = constant high word | (shared address >> 4).
      static_assert(NSUB % GSLOTS == 0 && ((NSUB / GSLOTS) & 1) == 0 && GSLOTS % 2 == 0,
                    "transform ring (12 or 24 entries per item): slot and parity of an entry do not depend on the item, "
                    "and the two entries of a both-window sub-batch are adjacent slots");
      static_assert((NSUB & 3) == 0, "matrix buffers: parity of a sub-batch does not depend on the item");
      constexpr uint32_t DHI = ptx::smem_desc_hi<ROWB>(), DHI_G = ptx::smem_desc_hi<ROWG>();
      const uint32_t smem16 = smem32 >> 4;
      const uint32_t a_full = bar32; // one base register, every other barrier at a compile-time offset
      const uint32_t a_empty = a_full + 8 * STAGES, a_gfull = a_empty + 8 * STAGES, a_gempty = a_gfull + 8 * GSLOTS,
                     a_mfull = a_gempty + 8 * GSLOTS, a_mempty = a_mfull + 16, a_pfull = a_mempty + 16, a_rest = a_pfull + 8,
                     a_wready = a_rest + 8;
      // MMA i (0..8) of a half K-block: triple i / 3 (operand parts and K step), plane i % 3.
      //   half 0: (hi.hi, ks 0), (hi.hi, ks 1), (lo.hi, ks 0)      half 1: (lo.hi, ks 1), (hi.lo, ks 0), (hi.lo, ks 1)
      auto g1_mma = [&](uint32_t st16, int hpar, int i, uint32_t acc) {
        const int t = i / 3, c = i % 3;
        const int a_part = hpar == 0 ? (t == 2 ? 1 : 0) : (t == 0 ? 1 : 0);
        const int b_part = hpar == 0 ? 0 : (t == 0 ? 0 : 1);
        const int ks = hpar == 0 ? (t == 1 ? 1 : 0) : (t == 1 ? 0 : 1);
        ptx::umma_f16_ss_lo(tmem_base + c * NF, st16 + ((a_part * A_PART + c * MV * ROWB + ks * 32) >> 4),
                            st16 + ((2 * A_PART + b_part * B_PART + ks * 32) >> 4), DHI, idesc1, acc);
      };
      // GEMM 2 of sub-batch sb (compile-time after unrolling) over nw windows: hi.hi, lo.hi, hi.lo at K = 16 per window.
      // nw = 1: ring entry sb, aw = the tile's window of the W tile; nw = 2 (both-window tile): entries 2 sb, 2 sb + 1,
      // whose data the first barrier covers, aw = window 0
      auto g2_sub = [&](int sb, int nw, uint32_t aw) {
        const int b = sb & 1, e0 = sb * nw, gs0 = e0 % GSLOTS;
        ptx::mbar_wait_a(a_gfull + 8 * gs0, (e0 / GSLOTS) & 1);
        ptx::mbar_wait_a(a_mempty + 8 * b, ((sb >> 1) & 1) ^ 1);
        ptx::tc_fence_after();
        const uint32_t dm = tmem_base + COL_M + b * SUBN;
#pragma unroll
        for(int w = 0; w < nw; w++)
        {
          const uint32_t sg16 = smem16 + ((OFF_G + (gs0 + w) * G_WIN) >> 4);
#pragma unroll
          for(int prod = 0; prod < 3; prod++)
          {
            const int pa = prod == 1 ? 1 : 0, pb = prod == 2 ? 1 : 0;
            ptx::umma_f16_ts_lo(dm, aw + w * KW + pa * (KW / 2), sg16 + ((pb * G_PART) >> 4), DHI_G, idesc2,
                                (w | prod) != 0 ? 1u : 0u);
          }
        }
        ptx::tc_commit_a(a_mfull + 8 * b);
#pragma unroll
        for(int w = 0; w < nw; w++) ptx::tc_commit_a(a_gempty + 8 * (gs0 + w));
      };
      // half K-block h (compile-time after unrolling: K-block h / 2, operand half h % 2) of the GEMM 1 whose first K-block
      // has ring position kbn0 (run-time).  The even half waits for the TMA data, the odd half hands the stage back.
      auto g1_half = [&](int h, int kbn0) {
        const int kbn = kbn0 + (h >> 1);
        const uint32_t s = static_cast<uint32_t>(kbn % STAGES);
        const uint32_t st16 = smem16 + s * (STAGE >> 4);
        if((h & 1) == 0)
        {
          ptx::mbar_wait_a(a_full + 8 * s, (kbn / STAGES) & 1);
          ptx::tc_fence_after();
#pragma unroll
          for(int i = 0; i < 9; i++) g1_mma(st16, 0, i, (h == 0 && i < 3) ? 0u : 1u);
        }
        else
        {
#pragma unroll
          for(int i = 0; i < 9; i++) g1_mma(st16, 1, i, 1u);
          ptx::tc_commit_a(a_empty + 8 * s);
        }
      };
      if(nit > 0 && warp == 3)
      {
#pragma unroll
        for(int h = 0; h < 2 * NKB; h++) g1_half(h, 0);
        ptx::tc_commit_a(a_pfull);
      }
      if(warp == 3)
      {
        // ---- GEMM 1 issuer: the 126 MMAs of item k + 1 as soon as item k's accumulators have been drained into the epilogue
        //      warps' registers; the stage ring and the tensor queue pace it ----
        for(int k = 0; k + 1 < nit; k++)
        {
          ptx::mbar_wait_a(a_rest, k & 1);
          ptx::tc_fence_after();
#pragma unroll
          for(int h = 0; h < 2 * NKB; h++) g1_half(h, (k + 1) * NKB);
          ptx::tc_commit_a(a_pfull);
        }
      }
      // ---- GEMM 2 issuer (warp 1): the twelve sub-batches of every item, two matrix buffers; the tile mode selects
      //      one of two unrolled streams once per item ----
      int wcount = 0, prev_tile = -1, mode = 0;
      for(int k = 0; k < (warp == 3 ? 0 : nit); k++)
      {
        const int tile = (it0 + k) / p.nfb;
        if(tile != prev_tile)
        {
          mode = p.tile_mode[tile];
          ptx::mbar_wait_a(a_wready, wcount & 1);
          ptx::tc_fence_after();
          wcount++;
          prev_tile = tile;
        }
        if(mode == 2)
        {
#pragma unroll
          for(int sb = 0; sb < NSUB; sb++) g2_sub(sb, 2, tmem_base + COL_W);
        }
        else
        {
          const uint32_t aw = tmem_base + COL_W + KW * mode;
#pragma unroll
          for(int sb = 0; sb < NSUB; sb++) g2_sub(sb, 1, aw);
        }
      }
    }
  }
  }
  else
  {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
    const int ew = warp - CTRL_WARPS;
    const int q = warp & 3;        // TMEM lane quadrant this warp may access (hardware rule: warp id % 4)
    const int fp = ew >> 2;        // which frame pair of every 8-frame sub-batch
    const uint32_t lane_taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const float sp = p.scale_p;
    // barriers as 32-bit shared addresses, frame stride and validity bounds hoisted: the r02h source page showed ~120
    // instructions per sub-batch and warp for 24 FMA + 6 stores (cvta sequences, 64-bit store addresses rebuilt from the
    // kernel parameters for every frame)
    const uint32_t a_mfull = bar32 + 16 * (STAGES + GSLOTS); // one base register, compile-time offsets
    const uint32_t a_mempty = a_mfull + 16, a_pfull = a_mempty + 16, a_rest = a_pfull + 8, a_wready = a_rest + 8;
    const unsigned fstride = static_cast<unsigned>(p.V) * 3u; // floats per frame of the output
    // (At 112 registers ptxas rebuilds part of this state in the first sub-batches instead of keeping it; forcing it into
    // registers with opaque asm operands gave 72 instead of 75-120 instructions per sub-batch and was 2 % SLOWER.)
    int prev_tile = -1;
    int wv0 = 0, nvalid = 0;
    float T0 = 0.f, T1 = 0.f, T2 = 0.f, sm = 0.f;
    for(int k = 0; k < nit; k++)
    {
      const int item = it0 + k;
      const int tile = item / p.nfb, f0 = (item - tile * p.nfb) * NF;
      if(tile != prev_tile)
      {
        prev_tile = tile;
        wv0 = tile * MV + q * 32;
        const int vc = min(wv0 + lane, p.V - 1);
        nvalid = max(0, min(32, p.V - wv0));
        if(ew < 4)
        {
          // every MMA that read the previous W tile has completed: this warp has seen m_full of the item's last sub-batch
          store_w_windows(p.weights + static_cast<size_t>(vc) * kJoints, lane_taddr + COL_W, p.wmap, p.primary,
                          p.tile_mode[tile]);
          ptx::tmem_st_wait();
          ptx::tc_fence_before();
          __syncwarp();
          if(lane == 0) ptx::mbar_arrive_a(a_wready);
        }
        sm = p.scale_m / p.wsum[vc]; // homogeneous divide (LinearBlendSkinning.cpp:545-550) folded into the scale
        const float * tp = p.basis + static_cast<size_t>(3) * vc * kBlendK + KUSED;
        T0 = __ldg(tp) * sm, T1 = __ldg(tp + kBlendK) * sm, T2 = __ldg(tp + 2 * kBlendK) * sm;
      }
      // root translations (theta row 0, SMPL.cpp:726-727) of this warp's 24 frames: lane l holds frame pair l / 2, frame
      // l % 2; fetched once per item (in flight during the p_full wait) and broadcast by shuffles in the sub-batch loop
      float trx = 0.f, try_ = 0.f, trz = 0.f;
      if(lane < FR_WARP)
      {
        const int f = min(f0 + (lane >> 1) * SUBF + fp * EPI_FR + (lane & 1), p.B - 1);
        const float * tq = p.theta + static_cast<size_t>(f) * ((kJoints + 1) * 3);
        trx = __ldg(tq), try_ = __ldg(tq + 1), trz = __ldg(tq + 2);
      }
      // ---- drain the rest accumulators of this item: 24 frames x (x, y, z), pre-multiplied by scale / sum w ----
      float R[3][FR_WARP];
      ptx::mbar_wait_a(a_pfull, k & 1);
      ptx::tc_fence_after();
#pragma unroll
      for(int c = 0; c < 3; c++)
      {
        ptx::tmem_ld_x16(lane_taddr + c * NF + fp * FR_WARP, R[c]);
        ptx::tmem_ld_x8p(lane_taddr + c * NF + fp * FR_WARP + 16, R[c] + 16);
      }
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if(lane == 0) ptx::mbar_arrive_a(a_rest);
      {
        const float s = sp * sm;
#pragma unroll
        for(int i = 0; i < FR_WARP; i++)
        {
          R[0][i] = fmaf(R[0][i], s, T0);
          R[1][i] = fmaf(R[1][i], s, T1);
          R[2][i] = fmaf(R[2][i], s, T2);
        }
      }
      float * outp = p.out + (static_cast<size_t>(f0 + fp * EPI_FR) * p.V + wv0) * 3;
      float * outl = outp + lane * 3;                                  // this lane's vertex in the warp's first frame
      const int nfv = lane < nvalid ? p.B - f0 - fp * EPI_FR : 0;      // frame slots (sb * SUBF + t) below nfv are stored
#pragma unroll
      for(int sb = 0; sb < NSUB; sb++)
      {
        const int h = sb & 1; // matrix buffer of this sub-batch (NSUB is even: the same for every item)
        float tr[EPI_FR][3];
#pragma unroll
        for(int t = 0; t < EPI_FR; t++)
        {
          tr[t][0] = __shfl_sync(0xffffffffu, trx, sb * EPI_FR + t);
          tr[t][1] = __shfl_sync(0xffffffffu, try_, sb * EPI_FR + t);
          tr[t][2] = __shfl_sync(0xffffffffu, trz, sb * EPI_FR + t);
        }
        ptx::mbar_wait_a(a_mfull + 8 * h, (sb >> 1) & 1); // 6 ring rounds per item: the parity does not depend on the item
        ptx::tc_fence_after();
        float M[EPI_FR * kXformFloats];
        const uint32_t mcol = lane_taddr + COL_M + h * SUBN + fp * (EPI_FR * kXformFloats);
        ptx::tmem_ld_x16(mcol, M);
        ptx::tmem_ld_x8p(mcol + 16, M + 16);
        ptx::tmem_ld_wait();
        ptx::tc_fence_before();
        __syncwarp();
        if(lane == 0) ptx::mbar_arrive_a(a_mempty + 8 * h); // the MMA warp may overwrite this matrix buffer
#pragma unroll
        for(int t = 0; t < EPI_FR; t++)
        {
          const float rx = R[0][sb * EPI_FR + t], ry = R[1][sb * EPI_FR + t], rz = R[2][sb * EPI_FR + t];
          const float * m = M + kXformFloats * t;
          const float ox = fmaf(m[0], rx, fmaf(m[1], ry, fmaf(m[2], rz, fmaf(m[3], sm, tr[t][0]))));
          const float oy = fmaf(m[4], rx, fmaf(m[5], ry, fmaf(m[6], rz, fmaf(m[7], sm, tr[t][1]))));
          const float oz = fmaf(m[8], rx, fmaf(m[9], ry, fmaf(m[10], rz, fmaf(m[11], sm, tr[t][2]))));
          // no staging: three 4-byte streaming stores per vertex and frame (a warp's 32 vertices are 384 contiguous
          // bytes; L2 merges the sectors).  Measured +2.4 % against staged float2 stores: the kernel is bound by
          // shared-memory bandwidth (UMMA operand reads + TMA writes), which the staging round trip competes for.
          float * o = outl + static_cast<size_t>((sb * SUBF + t) * fstride);
          if(sb * SUBF + t < nfv)
          {
            __stcs(o, ox);
            __stcs(o + 1, oy);
            __stcs(o + 2, oz);
          }
        }
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if(warp == 1) ptx::tmem_dealloc<TMEM_COLS>(tmem_base);
}

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
namespace
{
// GEMM 1 stages of 60 KB.  Three fit next to the six 6 KB transform slots (222 720 B), but measured slower than two
// (DESIGN.md 4.1)
constexpr int kStages = 2;

// The two joint windows of GEMM 2 (K = 16 each) for the skinning weights w (V, 24).  A vertex has at most a few
// non-zero weights and models number their vertices region by region, so most 128-vertex tiles touch a handful of
// joints; a tile whose joints all sit in one window needs one K step instead of two.  W0 holds 16 joints, W1 the 8
// others plus up to 8 joints of W0.  Every W0 is tried (C(24,16) = 735471, in increasing bit order); given W0, W1 takes
// the joints of the tiles that do not fit W0, largest tile first, while it stays within 16 joints.  The first W0 with
// the fewest vertices in tiles that fit neither window wins.  Only vertices < V count.
void choose_windows(const float * w, int V, int8_t (&slot_joint)[tc3::KJ], int8_t (&joint_slot)[kJoints],
                    std::vector<uint8_t> & mode)
{
  const int ntiles = (V + tc3::MV - 1) / tc3::MV;
  std::vector<uint32_t> tmask(ntiles, 0u);
  for(int v = 0; v < V; v++)
    for(int j = 0; j < kJoints; j++)
      if(w[static_cast<size_t>(v) * kJoints + j] != 0.f) tmask[v / tc3::MV] |= 1u << j;
  // distinct joint sets with their vertex counts, largest first (ties: first tile first)
  std::vector<std::pair<uint32_t, int>> sets;
  for(int t = 0; t < ntiles; t++)
  {
    const int nv = std::min(V, (t + 1) * tc3::MV) - t * tc3::MV;
    auto it = std::find_if(sets.begin(), sets.end(), [&](const std::pair<uint32_t, int> & q) { return q.first == tmask[t]; });
    if(it == sets.end())
      sets.emplace_back(tmask[t], nv);
    else
      it->second += nv;
  }
  std::stable_sort(sets.begin(), sets.end(), [](const std::pair<uint32_t, int> & a, const std::pair<uint32_t, int> & b) {
    return a.second > b.second;
  });
  const uint32_t all = (1u << kJoints) - 1;
  uint32_t best0 = 0, best1 = 0;
  long long best_cost = -1;
  for(uint32_t m0 = (1u << tc3::KW) - 1; m0 <= all;)
  {
    uint32_t m1 = all & ~m0;
    long long cost = 0;
    for(const auto & q : sets)
    {
      if((q.first & ~m0) == 0) continue;
      const uint32_t u = m1 | q.first;
      if(__builtin_popcount(u) <= tc3::KW)
        m1 = u;
      else
        cost += q.second;
    }
    if(best_cost < 0 || cost < best_cost) best_cost = cost, best0 = m0, best1 = m1;
    if(cost == 0) break;
    const uint32_t c = m0 & (~m0 + 1u), r = m0 + c; // next set of 16 bits (Gosper)
    m0 = (((r ^ m0) >> 2) / c) | r;
  }
  int n0 = 0, n1 = tc3::KW;
  for(int s = 0; s < tc3::KJ; s++) slot_joint[s] = -1;
  for(int j = 0; j < kJoints; j++)
  {
    if(best1 >> j & 1u) slot_joint[n1++] = static_cast<int8_t>(j);
    if(best0 >> j & 1u) slot_joint[n0++] = static_cast<int8_t>(j);
    joint_slot[j] = static_cast<int8_t>((best0 >> j & 1u) ? n0 - 1 : n1 - 1);
  }
  mode.resize(ntiles);
  for(int t = 0; t < ntiles; t++) mode[t] = (tmask[t] & ~best0) == 0 ? 0 : (tmask[t] & ~best1) == 0 ? 1 : 2;
}
} // namespace

namespace sb
{
size_t tc3_frame_operand_bytes(int64_t batch)
{
  const size_t bpad = align_up(static_cast<size_t>(batch), tc3::NF);
  return align_up(2 * bpad * tc3::KP * sizeof(__half)) + align_up(2 * bpad * kXformFloats * tc3::KJ * sizeof(__half));
}

// gate of the tcgen05 kernels (K2''' and lbs_tc_kernel): a CC 10.x device, the driver's tensor-map encoder and an even
// V >= 128.  Builds the stage images of the fp16 split basis and chooses the joint windows from the host weights
// (V, 24); called once from smplpp_model_create
int tc3_prepare_model(ModelDev & d, float basis_max_abs, const float * weights)
{
  d.tc3_ready = false;
  int dev = 0, major = 0;
  SB_CUDA(cudaGetDevice(&dev));
  SB_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  SB_CUDA(cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev));
  if(major != 10 || !encode_fn() || (d.V & 1) || d.V < tc3::MV || d.sm_count <= 0) return SMPLPP_OK;
  const int ntiles = (d.V + tc3::MV - 1) / tc3::MV;
  // largest power of two that keeps |basis| 2^e <= 1024: lo = x - hi stays a normal fp16 for all but tiny entries
  int e = 0;
  if(basis_max_abs > 0.f)
  {
    while(basis_max_abs * ldexpf(1.f, e + 1) <= 1024.f && e < 24) e++;
    while(basis_max_abs * ldexpf(1.f, e) > 1024.f && e > -24) e--;
  }
  d.tc3_basis_exp = e;
  const long long n = static_cast<long long>(ntiles) * 3 * tc3::MV * tc3::KP;
  SB_CUDA(cudaMalloc(&d.basis_img16, static_cast<size_t>(2) * n * sizeof(__half)));
  basis_image_f16_kernel<<<static_cast<unsigned>((n + 255) / 256), 256>>>(d.basis, d.V, ntiles, ldexpf(1.f, e),
                                                                         static_cast<uint8_t *>(d.basis_img16));
  SB_LAUNCHED();
  std::vector<uint8_t> mode;
  choose_windows(weights, d.V, d.tc3_slot_joint, d.tc3_joint_slot, mode);
  SB_CUDA(cudaMalloc(&d.tc3_tile_mode, mode.size()));
  SB_CUDA(cudaMemcpy(d.tc3_tile_mode, mode.data(), mode.size(), cudaMemcpyHostToDevice));
  SB_CUDA(cudaDeviceSynchronize());
  SB_CUDA(cudaFuncSetAttribute(blend_skin_tc3_kernel<kStages, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               tc3::Layout<kStages, 6>::SMEM_BYTES));
  d.tc3_tiles = ntiles;
  d.tc3_ready = true;
  return SMPLPP_OK;
}

void tc3_release_model(ModelDev & d)
{
  if(d.basis_img16) cudaFree(d.basis_img16);
  if(d.tc3_tile_mode) cudaFree(d.tc3_tile_mode);
  d.basis_img16 = nullptr;
  d.tc3_tile_mode = nullptr;
  d.tc3_ready = false;
}

// coef (B,224) and xforms (B,24,12) fp32 from K1; scratch: tc3_frame_operand_bytes(B)
int launch_blend_skin_tc3(const ModelDev & d, cudaStream_t st, int B, const float * coef, const float * xforms, void * scratch,
                          const float * theta, float * out, bool images_ready)
{
  if(!d.tc3_ready) return fail(SMPLPP_ERR_INVALID, "SMPL", "pipelined tcgen05 skinning variant is not available for this model");
  if(reinterpret_cast<uintptr_t>(out) & 7) return fail(SMPLPP_ERR_INVALID, "SMPL", "tcgen05 variants need 8-byte aligned vertices");
  if(reinterpret_cast<uintptr_t>(scratch) & 127) return fail(SMPLPP_ERR_INVALID, "SMPL", "tcgen05 variants need a 128-byte aligned workspace");
  const int Bpad = static_cast<int>(align_up(static_cast<size_t>(B), tc3::NF));
  uint8_t * img_b = static_cast<uint8_t *>(scratch);
  uint8_t * img_g = img_b + tc3::img_g_offset(Bpad);
  if(!images_ready)
  {
    const long long n = static_cast<long long>(Bpad) * (tc3::KP + kXformFloats * tc3::KJ) / 8; // 16-byte chunks
    frame_images3_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(coef, xforms, B, Bpad, img_b, img_g,
                                                                                  tc3::window_map(d));
    SB_LAUNCHED();
  }
  tc3::Params p;
  p.V = d.V;
  p.B = B;
  p.Bpad = Bpad;
  p.ntiles = d.tc3_tiles;
  p.nfb = Bpad / tc3::NF;
  p.nitems = p.ntiles * p.nfb;
  p.scale_p = ldexpf(1.f, -(d.tc3_basis_exp + tc3::COEF_EXP));
  p.scale_m = ldexpf(1.f, -(tc3::W_EXP + tc3::G_EXP));
  p.img_a = static_cast<const uint8_t *>(d.basis_img16);
  p.img_b = img_b;
  p.img_g = img_g;
  p.tile_mode = d.tc3_tile_mode;
  p.wmap = tc3::window_map(d);
  p.primary = 0;
  for(int j = 0; j < kJoints; j++) p.primary |= 1u << d.tc3_joint_slot[j];
  p.basis = d.basis;
  p.weights = d.weights_dense;
  p.wsum = d.lbs_wsum;
  p.theta = theta;
  p.out = out;
  const int grid = p.nitems < d.sm_count ? p.nitems : d.sm_count;
  blend_skin_tc3_kernel<kStages, 6><<<grid, tc3::THREADS, tc3::Layout<kStages, 6>::SMEM_BYTES, st>>>(p);
  SB_LAUNCHED();
  return SMPLPP_OK;
}
} // namespace sb
