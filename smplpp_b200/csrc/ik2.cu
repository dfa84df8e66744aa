// Fused MoSh / MoSh++ IK step on sm_100a: ONE kernel per iteration replaces the per-frame loop body of the reference's
// node/node.cpp:753-968 (forward on the task vertices, IkTask geometry src/IkTask.cpp:33-86, the Jacobian rows the
// reference harvests from Tensor::backward :823-873, fp64 normal equations :884-904, LLT / box QP :907-939, update
// :946-968) for F frames per CTA.
//
//   CTA = F "teams" of 128 threads (one team = one frame) + one TMA producer warp.
//   The teams walk the n tasks (markers) in lock step.  All a task needs from the model are the blend-basis rows of its
//   ~12 vertices (2688 B each): the producer streams them ONCE per CTA into a shared-memory ring (cp.async.bulk + mbarrier)
//   and all F frames consume them there - for the rest shape of the vertices AND for the pose-blend columns of the
//   Jacobian, which re-read those rows.  (The two-kernel predecessor re-read 1.7 MB of basis rows per FRAME from L2 and
//   wrote / re-read a 49 KB Jacobian per frame through HBM.)
//   The rows of J of one task live in shared memory just long enough to be accumulated into the frame's A = J'J (fp64,
//   4x4 tiles), so J never leaves the SM; the frame's team then factors A in place (tiled right-looking Cholesky) and
//   applies the step.
//
// Attachment topology comes as one self-contained TaskRec per task (tasks.cuh): shared by all frames (records of the task
// set, STAGED = true) or per (frame, task) after the projection step re-seated IkTask::faceIdx_ (node.cpp:993-1001;
// records built on the device by task_topo_kernel, basis rows read through L1 / L2, STAGED = false).
#include <algorithm>
#include <cmath>
#include <cstring>

#include <math_constants.h>

#include "common.cuh"
#include "forward.cuh"
#include "ik2.cuh"
#include "ik_math.cuh"
#include "tasks.cuh"
#include "tc_ptx.cuh"
#include "vposer.cuh"

using namespace sb;

namespace k2
{
constexpr int TEAM = 128;                      // threads per frame
constexpr int MAXF = 4;                        // frames per CTA
constexpr int PAIR_BYTES = 3 * kBlendK * 4;    // x | y | z basis rows of one vertex: 2688 B, contiguous in ModelDev::basis
constexpr int NBAR = 8;                        // tasks in flight in the ring
constexpr int SMEM_LIMIT = 227 * 1024;
} // namespace k2

// ------------------------------------------------------------------------------------------------------------
// shared-memory layout of one team (byte offsets from the team base), computed on the host
// ------------------------------------------------------------------------------------------------------------
struct Ik2Layout
{
  int theta, beta, coef, R, dR, Jt, G, tp, M, JS, dTg, dTp; // chain (floats)
  int A, bvec, misc;                                         // fp64: tiles, b, [esq, valid, bad, ok, ...]
  int rec;                                                   // the task's record (608 B)
  int tin, skin, pv, pr, sw, xw, sj, Au, itemN, cornN, ts, Dref, C4, CA4, ybuf, live, Q, Jrow, Jc; // per-task scratch
  int sx, sg, sd, sstate;                                    // solve temporaries (alias the per-task scratch)
  int team_bytes;
  int ring_off, ring_slots, bar_off, total;
};

struct Ik2Params
{
  ChainTopo topo;
  uint32_t anc_mask[kJoints];
  Ik2Layout L;
  // model
  const float * basis;
  const uint8_t * lbs_joint;
  const float * lbs_weight;
  const float * lbs_wsum;
  int Vpad, kmax;
  const float * joint_template;
  const float * joint_shape;
  // topology
  const TaskRec * recs;
  const TaskSkin * skins; // skinning rows of the records (kmax <= 4), else null: read from the model arrays
  long long rec_stride; // records per frame: 0 = shared by all frames
  int n, MP, MI, ML;
  // problem
  int B, F;
  int use_ring, beta_cols, phi_cols, vposer, enable_qp, skip_if_too_few, update_state, update_weights, schur;
  int theta_dim, thp, php, Dp, ldf, ld, nbt, ntile, dim_ref;
  float normal_offset, normal_task_weight, reg_theta, reg_phi, reg_beta, phi_limit, beta_limit, latent_reg, hand_reg;
  // per-frame state
  const float * theta75;  // (B, 75) assembled theta (== theta_state when !vposer)
  float * theta_state;    // (B, theta_dim)
  float * beta;
  long long beta_stride;
  float * vertex_weights; // (B, n, 3)
  const float * target_pos;
  const float * target_normal;
  const float * pos_task_weight;
  const float * vposer_jac; // (B, 63, 32)
  // outputs
  int * status;
  float * e_out;      // (B, 4n)
  float * j_out;      // (B, 4n, dim_ref) reference layout
  double * a_out;     // (B, dim_ref, dim_ref)
  double * b_out;     // (B, dim_ref)
  double * delta_out; // (B, dim_ref)
  float * dphi_out;   // (B, n, 2)
  double * a_ws;      // (B, ntiles * 16) copy of A for the active-set QP
  double * schur_out; // (B, 111)
  double * factor_ws; // (B, P)
  long long * dbg_cycles; // (32) phase timer of the debug build
};

// ------------------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------------------
// Phase timer of the task loop (debug builds only: -DSMPLPP_IK2_DBG): team 0 of CTA 0 accumulates the cycles between
// consecutive barriers of the task loop into p.dbg_cycles[phase].
#ifdef SMPLPP_IK2_DBG
#define IK2_STAMP(k)                                                                \
  do                                                                                \
  {                                                                                 \
    if(blockIdx.x == 0 && team == 0 && tt == 0 && p.dbg_cycles)                     \
    {                                                                               \
      const long long now = clock64();                                              \
      p.dbg_cycles[k] += now - dbg_last;                                            \
      dbg_last = now;                                                               \
    }                                                                               \
  } while(0)
#else
#define IK2_STAMP(k)
#endif
__device__ __forceinline__ void team_sync(int team)
{
  asm volatile("bar.sync %0, %1;" ::"r"(team + 1), "n"(k2::TEAM) : "memory");
}
__device__ __forceinline__ int tile_idx(int bi, int bj) // bi >= bj
{
  return bi * (bi + 1) / 2 + bj;
}
// The lower triangle of A lives in shared memory as 4x4 tiles in ELEMENT-MAJOR order: element e = 4 r + c of tile t sits at
// A[e * NT + t] (NT = number of tiles, odd).  Threads that own consecutive tiles then touch consecutive doubles; the
// tile-major order (16 contiguous doubles per tile) put all 32 lanes of a warp on the same bank.
// element (i, j), i >= j:
__device__ __forceinline__ double & Aat(double * A, int NT, int i, int j)
{
  return A[((i & 3) * 4 + (j & 3)) * NT + tile_idx(i >> 2, j >> 2)];
}
// u-th (row, column) of a lower triangle enumerated row by row
__device__ __forceinline__ void tri_coords(int u, int & i, int & j)
{
  i = static_cast<int>((sqrtf(8.f * static_cast<float>(u) + 1.f) - 1.f) * 0.5f);
  while((i + 1) * (i + 2) / 2 <= u) i++;
  while(i * (i + 1) / 2 > u) i--;
  j = u - i * (i + 1) / 2;
}

// Tiled right-looking Cholesky of the leading `npb` block pivots of the (nbt x nbt tiles) lower triangle, executed by one
// team.  With npb < nbt the trailing tiles are left holding the Schur complement.  *ok = 0 on a non-positive pivot
// (Eigen::LLT NumericalIssue, node.cpp:934-937).
__device__ void team_cholesky(double * A, int NT, int nbt, int npb, int tt, int team, volatile int * ok)
{
  for(int kb = 0; kb < npb; kb++)
  {
    const int tkk = tile_idx(kb, kb);
    if(tt == 0)
    {
      double l[4][4];
      bool good = true;
#pragma unroll
      for(int j = 0; j < 4; j++)
      {
        double d = A[(j * 4 + j) * NT + tkk];
#pragma unroll
        for(int k = 0; k < 4; k++)
          if(k < j) d -= l[j][k] * l[j][k];
        if(!(d > 0.0)) good = false;
        const double sd = sqrt(d);
        l[j][j] = sd;
        const double inv = 1.0 / sd;
#pragma unroll
        for(int i = 0; i < 4; i++)
          if(i > j)
          {
            double s = A[(i * 4 + j) * NT + tkk];
#pragma unroll
            for(int k = 0; k < 4; k++)
              if(k < j) s -= l[i][k] * l[j][k];
            l[i][j] = s * inv;
          }
      }
#pragma unroll
      for(int i = 0; i < 4; i++)
#pragma unroll
        for(int j = 0; j < 4; j++) A[(i * 4 + j) * NT + tkk] = j <= i ? l[i][j] : 0.0;
      if(!good) *ok = 0;
    }
    team_sync(team);
    if(!*ok) return;
    // panel: rows of the tiles below the pivot tile, X L_kk' = T  (one thread per row)
    {
      const double l00 = A[0 * NT + tkk], l10 = A[4 * NT + tkk], l11 = A[5 * NT + tkk], l20 = A[8 * NT + tkk],
                   l21 = A[9 * NT + tkk], l22 = A[10 * NT + tkk], l30 = A[12 * NT + tkk], l31 = A[13 * NT + tkk],
                   l32 = A[14 * NT + tkk], l33 = A[15 * NT + tkk];
      const double i00 = 1.0 / l00, i11 = 1.0 / l11, i22 = 1.0 / l22, i33 = 1.0 / l33;
      for(int u = tt; u < 4 * (nbt - kb - 1); u += k2::TEAM)
      {
        // thread = (row of the tile, tile): consecutive threads take the same row of consecutive tiles
        const int nt_below = nbt - kb - 1;
        const int r = u / nt_below, ti = u - r * nt_below;
        double * row = A + (r * 4) * NT + tile_idx(kb + 1 + ti, kb);
        const double x0 = row[0] * i00;
        const double x1 = (row[NT] - x0 * l10) * i11;
        const double x2 = (row[2 * NT] - x0 * l20 - x1 * l21) * i22;
        const double x3 = (row[3 * NT] - x0 * l30 - x1 * l31 - x2 * l32) * i33;
        row[0] = x0, row[NT] = x1, row[2 * NT] = x2, row[3 * NT] = x3;
      }
    }
    team_sync(team);
    // trailing update: T_ij -= T_ik T_jk'  for kb < j <= i
    {
      const int mrem = nbt - kb - 1;
      const int cnt = mrem * (mrem + 1) / 2;
      for(int u = tt; u < cnt; u += k2::TEAM)
      {
        int il, jl;
        tri_coords(u, il, jl);
        const int i = kb + 1 + il, j = kb + 1 + jl;
        const double * Ti = A + tile_idx(i, kb);
        const double * Tj = A + tile_idx(j, kb);
        double * T = A + tile_idx(i, j);
        double a[16], b[16];
#pragma unroll
        for(int e = 0; e < 16; e++) a[e] = Ti[e * NT], b[e] = Tj[e * NT];
#pragma unroll
        for(int r = 0; r < 4; r++)
#pragma unroll
          for(int c = 0; c < 4; c++)
          {
            double s = T[(r * 4 + c) * NT];
#pragma unroll
            for(int k = 0; k < 4; k++) s = fma(-a[r * 4 + k], b[c * 4 + k], s);
            T[(r * 4 + c) * NT] = s;
          }
      }
    }
    team_sync(team);
  }
}

// x <- L^-T L^-1 x on the leading n x n block (n a multiple of 4); executed by warp 0 of the team, result in x.
// Blocked by the 4x4 tiles: every lane solves the diagonal tile redundantly in registers (no exchange inside a block),
// then the lanes update the remaining rows; one warp barrier per block instead of two per unknown.
__device__ void warp_tiled_solve(double * A, int NT, int n, double * x, int tt)
{
  if(tt >= 32) return;
  const int nb = n >> 2;
  for(int kb = 0; kb < nb; kb++)
  {
    const double * Tk = A + tile_idx(kb, kb);
    const double x0 = x[4 * kb] / Tk[0];
    const double x1 = (x[4 * kb + 1] - Tk[4 * NT] * x0) / Tk[5 * NT];
    const double x2 = (x[4 * kb + 2] - Tk[8 * NT] * x0 - Tk[9 * NT] * x1) / Tk[10 * NT];
    const double x3 = (x[4 * kb + 3] - Tk[12 * NT] * x0 - Tk[13 * NT] * x1 - Tk[14 * NT] * x2) / Tk[15 * NT];
    __syncwarp();
    if(tt == 0) x[4 * kb] = x0, x[4 * kb + 1] = x1, x[4 * kb + 2] = x2, x[4 * kb + 3] = x3;
    for(int i = 4 * (kb + 1) + tt; i < n; i += 32)
    {
      const double * row = A + ((i & 3) * 4) * NT + tile_idx(i >> 2, kb);
      x[i] -= row[0] * x0 + row[NT] * x1 + row[2 * NT] * x2 + row[3 * NT] * x3;
    }
    __syncwarp();
  }
  for(int kb = nb - 1; kb >= 0; kb--)
  {
    const double * Tk = A + tile_idx(kb, kb);
    const double x3 = x[4 * kb + 3] / Tk[15 * NT];
    const double x2 = (x[4 * kb + 2] - Tk[14 * NT] * x3) / Tk[10 * NT];
    const double x1 = (x[4 * kb + 1] - Tk[9 * NT] * x2 - Tk[13 * NT] * x3) / Tk[5 * NT];
    const double x0 = (x[4 * kb] - Tk[4 * NT] * x1 - Tk[8 * NT] * x2 - Tk[12 * NT] * x3) / Tk[0];
    __syncwarp();
    if(tt == 0) x[4 * kb] = x0, x[4 * kb + 1] = x1, x[4 * kb + 2] = x2, x[4 * kb + 3] = x3;
    for(int i = tt; i < 4 * kb; i += 32)
    {
      // L(4 kb + c, i): tile (kb, i >> 2), element (c, i & 3)
      const double * col = A + (i & 3) * NT + tile_idx(kb, i >> 2);
      x[i] -= col[0] * x0 + col[4 * NT] * x1 + col[8 * NT] * x2 + col[12 * NT] * x3;
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------------------
// per-frame attachment records on the device: one warp per (frame, task)
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) task_topo_kernel(long long total, const int32_t * __restrict__ face_idx, int F,
                                                        const int32_t * __restrict__ faces, const int32_t * __restrict__ adj_offset,
                                                        const int32_t * __restrict__ adj_faces,
                                                        const uint32_t * __restrict__ vert_jmask, TaskRec * __restrict__ out,
                                                        TaskSkin * __restrict__ skins, const uint8_t * __restrict__ lbs_joint,
                                                        const float * __restrict__ lbs_weight, const float * __restrict__ lbs_wsum,
                                                        int Vpad, int kmax)
{
  __shared__ TaskRec s_rec[4];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long id = static_cast<long long>(blockIdx.x) * 4 + warp;
  if(id >= total) return;
  TaskRec & r = s_rec[warp];
  for(int i = lane; i < static_cast<int>(sizeof(TaskRec) / 4); i += 32) reinterpret_cast<uint32_t *>(&r)[i] = 0u;
  __syncwarp();
  const int f = face_idx[id];
  bool bad = f < 0 || f >= F;
  int np = 0, ni = 0;
  if(!bad)
  {
    if(lane < 3) r.gv[lane] = faces[3 * f + lane];
    np = 3;
    __syncwarp();
    for(int c = 0; c < 3 && !bad; c++)
    {
      const int v = r.gv[c];
      const int s0 = adj_offset[v], s1 = adj_offset[v + 1];
      int cnt = 0;
      for(int k = s0; k < s1; k++)
      {
        if(ni >= kRecItems)
        {
          bad = true;
          break;
        }
        const int g = adj_faces[k];
        for(int s = 0; s < 3; s++)
        {
          const int u = faces[3 * g + s];
          // pair-local id of u: search the list (two entries per lane), append when new
          const bool hit0 = lane < np && r.gv[lane] == u;
          const bool hit1 = lane + 32 < np && r.gv[lane + 32] == u;
          const unsigned m0 = __ballot_sync(0xffffffffu, hit0), m1 = __ballot_sync(0xffffffffu, hit1);
          int q;
          if(m0)
            q = __ffs(m0) - 1;
          else if(m1)
            q = 32 + __ffs(m1) - 1;
          else
          {
            if(np >= kRecPairs)
            {
              bad = true;
              break;
            }
            q = np++;
            if(lane == 0) r.gv[q] = u;
          }
          if(lane == 0) r.item[ni][s] = static_cast<uint8_t>(q);
          __syncwarp();
        }
        if(bad) break;
        if(lane == 0) r.item[ni][3] = static_cast<uint8_t>(c);
        ni++, cnt++;
      }
      if(lane == 0) r.nic[c] = static_cast<uint8_t>(cnt);
    }
  }
  __syncwarp();
  if(!bad)
  {
    // references of every pair, in item order (fixed summation order of the normal derivatives)
    if(lane == 0)
    {
      int off = 0;
      for(int q = 0; q < np; q++)
      {
        r.ref_off[q] = static_cast<uint8_t>(off);
        for(int it = 0; it < ni; it++)
          for(int s = 0; s < 3; s++)
            if(r.item[it][s] == q) r.refs[off++] = static_cast<uint8_t>(it * 4 + s);
      }
      r.ref_off[np] = static_cast<uint8_t>(off);
    }
    uint32_t m_all = 0, m_corner = 0;
    for(int q = lane; q < np; q += 32)
    {
      const uint32_t vm = vert_jmask[r.gv[q]];
      m_all |= vm;
      if(q < 3) m_corner |= vm;
    }
    for(int o = 16; o > 0; o >>= 1)
    {
      m_all |= __shfl_xor_sync(0xffffffffu, m_all, o);
      m_corner |= __shfl_xor_sync(0xffffffffu, m_corner, o);
    }
    if(lane == 0) r.jmask = m_all, r.jmask_corner = m_corner, r.np = static_cast<uint8_t>(np), r.ni = static_cast<uint8_t>(ni);
  }
  if(lane == 0) r.face = bad ? -1 : f;
  __syncwarp();
  uint4 * dst = reinterpret_cast<uint4 *>(out + id);
  const uint4 * src = reinterpret_cast<const uint4 *>(&r);
  for(int i = lane; i < static_cast<int>(sizeof(TaskRec) / 16); i += 32) dst[i] = src[i];
  if(skins)
  {
    TaskSkin & sk = skins[id];
    const int npp = bad ? 0 : np;
    for(int i = lane; i < kRecPairs * 4; i += 32)
    {
      const int q = i >> 2, sl = i & 3;
      const bool on = q < npp && sl < kmax;
      const int gv = on ? r.gv[q] : 0;
      sk.w[q][sl] = on ? lbs_weight[static_cast<size_t>(sl) * Vpad + gv] : 0.f;
      sk.j[q][sl] = on ? lbs_joint[static_cast<size_t>(sl) * Vpad + gv] : 0;
    }
    for(int q = lane; q < kRecPairs; q += 32) sk.ws[q] = q < npp ? lbs_wsum[r.gv[q]] : 1.f;
  }
}

// ------------------------------------------------------------------------------------------------------------
// the fused step
// ------------------------------------------------------------------------------------------------------------
template<int ROWS, bool STAGED>
__global__ void __launch_bounds__(k2::MAXF * k2::TEAM + 32, 1) ik_fused_kernel(const Ik2Params p)
{
  using namespace k2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const Ik2Layout & L = p.L;
  const int tid = threadIdx.x;
  const int F = p.F;
  const int n = p.n;
  uint64_t * bar_full = reinterpret_cast<uint64_t *>(smem_raw + L.bar_off);
  uint64_t * bar_done = bar_full + NBAR;
  unsigned char * ring = smem_raw + L.ring_off;
  const int R = L.ring_slots;
  if(STAGED)
  {
    if(tid == 0)
    {
      for(int i = 0; i < NBAR; i++)
      {
        ptx::mbar_init(bar_full + i, 1);
        ptx::mbar_init(bar_done + i, static_cast<uint32_t>(F * (TEAM / 32)));
      }
      ptx::fence_barrier_init();
    }
    __syncthreads();
    if(tid >= F * TEAM)
    {
      // ---- producer warp: basis rows of the pairs of task m -> ring, up to NBAR tasks / R slots ahead of the consumers ----
      if((tid & 31) == 0)
      {
        // pair-granular: the byte count of a task is armed up front, its copies go out as ring slots come free, so the
        // ring is always full and the next task's first rows are in flight while the current one is still being read
        int ring_pos = 0, free_slots = R, oldest = 0;
        auto release_oldest = [&]() {
          ptx::mbar_wait(bar_done + (oldest % NBAR), static_cast<uint32_t>((oldest / NBAR) & 1));
          free_slots += p.use_ring ? p.recs[oldest].np : 3;
          oldest++;
        };
        for(int m = 0; m < n; m++)
        {
          const TaskRec * rec = p.recs + m;
          const int npe = p.use_ring ? rec->np : 3;
          while(m - oldest >= NBAR) release_oldest();
          uint64_t * full = bar_full + (m % NBAR);
          ptx::mbar_expect_tx(full, static_cast<uint32_t>(npe * PAIR_BYTES));
          for(int q = 0; q < npe; q++)
          {
            while(free_slots < 1) release_oldest();
            ptx::bulk_load_1d(ring + static_cast<size_t>(ring_pos) * PAIR_BYTES,
                              p.basis + static_cast<size_t>(rec->gv[q]) * (3 * kBlendK), PAIR_BYTES, full);
            ring_pos = ring_pos + 1 < R ? ring_pos + 1 : 0;
            free_slots--;
          }
        }
      }
      return;
    }
  }
  // Roles inside a team are rotated by one warp per team: hardware warp w of every team sits on SM sub-partition w % 4,
  // and the thin phases (one thread, three threads, one warp) would otherwise all land on sub-partition 0.
  const int team = tid / TEAM;
  const int tt = ((tid % TEAM) + 32 * team) % TEAM, tw = tt >> 5, lane = tt & 31;
  const long long f_raw = static_cast<long long>(blockIdx.x) * F + team;
  const bool live_frame = f_raw < p.B; // a padding team of the last CTA repeats the last frame and writes nothing
  const long long f = live_frame ? f_raw : p.B - 1;
  unsigned char * base = smem_raw + static_cast<size_t>(team) * L.team_bytes;
  float * s_theta = reinterpret_cast<float *>(base + L.theta);
  float * s_beta = reinterpret_cast<float *>(base + L.beta);
  float * s_coef = reinterpret_cast<float *>(base + L.coef);
  float * s_R = reinterpret_cast<float *>(base + L.R);
  float * s_dR = reinterpret_cast<float *>(base + L.dR);
  float * s_Jt = reinterpret_cast<float *>(base + L.Jt);
  float * s_G = reinterpret_cast<float *>(base + L.G);
  float * s_tp = reinterpret_cast<float *>(base + L.tp);
  float * s_M = reinterpret_cast<float *>(base + L.M);
  float * s_JS = reinterpret_cast<float *>(base + L.JS);
  float * s_dTg = reinterpret_cast<float *>(base + L.dTg);
  float * s_dTp = reinterpret_cast<float *>(base + L.dTp);
  double * s_A = reinterpret_cast<double *>(base + L.A);
  double * s_b = reinterpret_cast<double *>(base + L.bvec);
  double * s_misc = reinterpret_cast<double *>(base + L.misc); // [0] esq  [1] valid  [2] bad  [3] ok  [4] flag  [5] iter  [6] atmin
  float * s_pv = reinterpret_cast<float *>(base + L.pv);
  float * s_pr = reinterpret_cast<float *>(base + L.pr);
  float * s_sw = reinterpret_cast<float *>(base + L.sw);
  float * s_xw = reinterpret_cast<float *>(base + L.xw);
  uint8_t * s_sj = reinterpret_cast<uint8_t *>(base + L.sj);
  float * s_Au = reinterpret_cast<float *>(base + L.Au);
  float * s_itemN = reinterpret_cast<float *>(base + L.itemN);
  float * s_cornN = reinterpret_cast<float *>(base + L.cornN);
  float * s_ts = reinterpret_cast<float *>(base + L.ts);
  float * s_Dref = reinterpret_cast<float *>(base + L.Dref);
  float * s_C4 = reinterpret_cast<float *>(base + L.C4);
  float * s_CA4 = reinterpret_cast<float *>(base + L.CA4);
  float * s_y = reinterpret_cast<float *>(base + L.ybuf);
  uint8_t * s_live = reinterpret_cast<uint8_t *>(base + L.live);
  float * s_Q = reinterpret_cast<float *>(base + L.Q);
  float * s_Jrow = reinterpret_cast<float *>(base + L.Jrow);
  float * s_Jc = reinterpret_cast<float *>(base + L.Jc);
  float * s_tin = reinterpret_cast<float *>(base + L.tin);
  const int kmax = p.kmax, ML = p.ML;
  const int ldf = p.ldf, ld = p.ld;
  const int phi_off_f = 76;             // phi columns of the theta-space row
  const int beta_off_f = 76 + p.php;    // beta columns of the theta-space row
  const int NT = p.ntile; // tiles of the (augmented) lower triangle, padded to an odd count

  // ---- prologue: state, rotations and their derivatives, joints, chain ----
  for(int i = tt; i < 75; i += TEAM) s_theta[i] = p.theta75[static_cast<size_t>(f) * 75 + i];
  if(tt < kShapeDim) s_beta[tt] = p.beta[static_cast<size_t>(f) * p.beta_stride + tt];
  for(int i = tt; i < NT * 16; i += TEAM) s_A[i] = 0.0;
  for(int i = tt; i < p.Dp + 4; i += TEAM) s_b[i] = 0.0;
  team_sync(team);
  if(tt < kJoints) chain_joint(tt, s_theta, s_beta, p.joint_template, p.joint_shape, p.beta_cols, s_R, s_dR, s_Jt, s_JS);
  team_sync(team);
  // blend coefficients of the frame: pose feature vec(R_1..R_23) - vec(I) | beta | 0 ...  The template column (217) is
  // NOT part of the dot product: the ~1 m template is added last, to the fully reduced sum of the mm-sized blend terms
  // (one rounding at the 1 m scale, as in the forward kernels; task normals amplify vertex noise by 1 / edge length)
  for(int i = tt; i < kBlendK; i += TEAM)
  {
    float v = 0.f;
    if(i < kPoseDim)
    {
      const int e = i % 9;
      v = s_R[9 * (i / 9 + 1) + e] - ((e == 0 || e == 4 || e == 8) ? 1.f : 0.f);
    }
    else if(i < kPoseDim + kShapeDim)
      v = s_beta[i - kPoseDim];
    s_coef[i] = v;
  }
  if(tt < 32) chain_globals_warp(tt, p.topo, s_R, s_Jt, s_G, s_tp);
  team_sync(team);
  if(tt < 72) chain_dM(tt, p.topo, s_dR, s_G, s_M);
  // d tg_j / d beta and d t'_j / d beta (3 x 10 per joint)
  if(p.beta_cols)
  {
    for(int d = 0; d <= p.topo.max_depth; d++)
    {
      for(int u = tt; u < kJoints * kShapeDim; u += TEAM)
      {
        const int j = u / kShapeDim, i = u % kShapeDim;
        if(p.topo.depth[j] == d) chain_dtg_dbeta(j, i, p.topo.parent[j], s_G, s_JS, s_dTg);
      }
      team_sync(team);
    }
    for(int u = tt; u < kJoints * kShapeDim; u += TEAM) chain_dtp_dbeta(u / kShapeDim, u % kShapeDim, s_G, s_JS, s_dTg, s_dTp);
  }
  team_sync(team);

  // per-task inputs of the frame (attachment weights, target, marker weight, target normal): fetched once, coalesced,
  // instead of by one thread per task with the full global latency on the critical path of every task
  for(int i = tt; i < 3 * n; i += TEAM)
  {
    s_tin[i] = p.vertex_weights[static_cast<size_t>(f) * 3 * n + i];
    s_tin[3 * n + i] = p.target_pos[static_cast<size_t>(f) * 3 * n + i];
    if(ROWS == 4) s_tin[7 * n + i] = p.target_normal ? p.target_normal[static_cast<size_t>(f) * 3 * n + i] : (i % 3 == 2 ? 1.f : 0.f);
  }
  for(int i = tt; i < n; i += TEAM) s_tin[6 * n + i] = p.pos_task_weight ? p.pos_task_weight[static_cast<size_t>(f) * n + i] : 1.f;
  team_sync(team);
  // thread 0 of the team carries the frame's scalars through the task loop
  double esq = 0.0;
  int valid = 0, bad = 0;
  int ring_pos = 0;
  const f3 trans = mk3(s_theta[0], s_theta[1], s_theta[2]);
  const float * Jv = p.vposer ? p.vposer_jac + static_cast<size_t>(f) * 63 * 32 : nullptr;
  const TaskRec * grec = p.recs + static_cast<size_t>(f) * p.rec_stride;

  // tiles of A = J'J owned by this thread (two at most are kept in registers; larger problems recompute the coordinates)
  const int nb_acc = p.Dp >> 2;
  const int ntiles_acc = nb_acc * (nb_acc + 1) / 2;
  int my_bi[2] = {0, 0}, my_bj[2] = {0, 0};
#pragma unroll
  for(int s2 = 0; s2 < 2; s2++)
    if(tt + s2 * TEAM < ntiles_acc) tri_coords(tt + s2 * TEAM, my_bi[s2], my_bj[s2]);

  // the record of task m lives in buffer m & 1; the next one is fetched while the current task is being accumulated
  const TaskSkin * gskin = p.skins ? p.skins + static_cast<size_t>(f) * p.rec_stride : nullptr;
  const int skin_bytes = static_cast<int>(sizeof(TaskSkin));
  if(tt < static_cast<int>(sizeof(TaskRec) / 16))
    reinterpret_cast<uint4 *>(base + L.rec)[tt] = __ldg(reinterpret_cast<const uint4 *>(grec) + tt);
  if(gskin && tt >= 32 && tt - 32 < skin_bytes / 16)
    reinterpret_cast<uint4 *>(base + L.skin)[tt - 32] = __ldg(reinterpret_cast<const uint4 *>(gskin) + (tt - 32));
  team_sync(team);

#ifdef SMPLPP_IK2_DBG
  long long dbg_last = clock64();
#endif
  for(int m = 0; m < n; m++)
  {
    const TaskRec * s_rec = reinterpret_cast<const TaskRec *>(base + L.rec);
    // ---- empty J rows (the previous task's rows were consumed before its closing barrier) ----
    for(int i = tt; i < 4 * ldf; i += TEAM) s_Jrow[i] = 0.f;
    const bool rec_ok = s_rec->face >= 0;
    const int npe = rec_ok ? (p.use_ring ? s_rec->np : 3) : 0;
    const int nie = rec_ok && p.use_ring ? s_rec->ni : 0;
    const size_t fm = static_cast<size_t>(f) * n + m;
    // ---- rest shape of the task's vertices: basis row . coefficients (warp per pair, lanes over the 224 columns) ----
    const unsigned char * ring_base = nullptr;
    if(STAGED)
    {
      if(lane == 0) ptx::mbar_wait(bar_full + (m % NBAR), static_cast<uint32_t>((m / NBAR) & 1));
      __syncwarp();
      ring_base = ring;
    }
    for(int q = tw; q < npe; q += TEAM / 32)
    {
      const float * P;
      if(STAGED)
      {
        const int slot = ring_pos + q < R ? ring_pos + q : ring_pos + q - R;
        P = reinterpret_cast<const float *>(ring_base + static_cast<size_t>(slot) * PAIR_BYTES);
      }
      else
        P = p.basis + static_cast<size_t>(s_rec->gv[q]) * (3 * kBlendK);
      float ax = 0.f, ay = 0.f, az = 0.f;
#pragma unroll
      for(int i = 0; i < kBlendK / 32; i++)
      {
        const int k = lane + 32 * i;
        const float c = s_coef[k];
        ax = fmaf(STAGED ? P[k] : __ldg(P + k), c, ax);
        ay = fmaf(STAGED ? P[kBlendK + k] : __ldg(P + kBlendK + k), c, ay);
        az = fmaf(STAGED ? P[2 * kBlendK + k] : __ldg(P + 2 * kBlendK + k), c, az);
      }
#pragma unroll
      for(int o = 16; o > 0; o >>= 1)
      {
        ax += __shfl_xor_sync(0xffffffffu, ax, o);
        ay += __shfl_xor_sync(0xffffffffu, ay, o);
        az += __shfl_xor_sync(0xffffffffu, az, o);
      }
      if(lane == 0)
      {
        constexpr int kT = kPoseDim + kShapeDim; // template column
        s_pr[3 * q] = ax + (STAGED ? P[kT] : __ldg(P + kT));
        s_pr[3 * q + 1] = ay + (STAGED ? P[kBlendK + kT] : __ldg(P + kBlendK + kT));
        s_pr[3 * q + 2] = az + (STAGED ? P[2 * kBlendK + kT] : __ldg(P + 2 * kBlendK + kT));
      }
    }
    team_sync(team);
    IK2_STAMP(0);
    // ---- skinning, one thread per vertex: normalised weights, w_j x_uj (vertex carried by bone j, no root translation),
    //      the posed vertex in the reference's order of operations (LinearBlendSkinning.cpp:445-483: M = sum_j W_j G'_j
    //      with the raw weights, h = M [rest; 1], vertex = h / sum_j W_j + trans -- the task normals amplify any rounding
    //      difference in the vertices by 1 / edge length) and A_u = sum_j w_j Rg_j (rotation part of the skinning matrix);
    //      the last warp lists the live joints of the task (the joint must be an ancestor of a vertex of the task) ----
    const uint32_t jm = rec_ok ? (p.use_ring ? s_rec->jmask : s_rec->jmask_corner) : 0u;
    const int nlive = min(__popc(jm), ML);
    if(tt >= 96 && tt - 96 < nlive) s_live[tt - 96] = static_cast<uint8_t>(__fns(jm, 0, tt - 96 + 1));
    if(tt < npe)
    {
      const int gv = s_rec->gv[tt];
      const TaskSkin * s_skin = reinterpret_cast<const TaskSkin *>(base + L.skin);
      const float ws = gskin ? s_skin->ws[tt] : __ldg(p.lbs_wsum + gv);
      const f3 ru = ld3(s_pr + 3 * tt);
      float Au[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      float Mr[12] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for(int sl = 0; sl < kmax; sl++)
      {
        const int i = tt * kmax + sl;
        const float wr = gskin ? s_skin->w[tt][sl] : __ldg(p.lbs_weight + static_cast<size_t>(sl) * p.Vpad + gv);
        const int j = gskin ? s_skin->j[tt][sl] : __ldg(p.lbs_joint + static_cast<size_t>(sl) * p.Vpad + gv);
        const float wj = wr / ws;
        s_sw[i] = wj;
        s_sj[i] = static_cast<uint8_t>(j);
        const float * G = s_G + 12 * j;
        const f3 x = skin_term(G, s_tp + 3 * j, 1, ru, wj);
        s_xw[3 * i] = x.x, s_xw[3 * i + 1] = x.y, s_xw[3 * i + 2] = x.z;
#pragma unroll
        for(int r = 0; r < 3; r++)
        {
#pragma unroll
          for(int c = 0; c < 3; c++)
          {
            Au[3 * r + c] = fmaf(wj, G[4 * r + c], Au[3 * r + c]);
            Mr[4 * r + c] = fmaf(wr, G[4 * r + c], Mr[4 * r + c]);
          }
          Mr[4 * r + 3] = fmaf(wr, s_tp[3 * j + r], Mr[4 * r + 3]);
        }
      }
      f3 v; // homo2cart divides (LinearBlendSkinning.cpp:538-553)
      v.x = (Mr[0] * ru.x + Mr[1] * ru.y + Mr[2] * ru.z + Mr[3]) / ws + trans.x;
      v.y = (Mr[4] * ru.x + Mr[5] * ru.y + Mr[6] * ru.z + Mr[7]) / ws + trans.y;
      v.z = (Mr[8] * ru.x + Mr[9] * ru.y + Mr[10] * ru.z + Mr[11]) / ws + trans.z;
      s_pv[3 * tt] = v.x, s_pv[3 * tt + 1] = v.y, s_pv[3 * tt + 2] = v.z;
#pragma unroll
      for(int e = 0; e < 9; e++) s_Au[9 * tt + e] = Au[e];
    }
    team_sync(team);
    IK2_STAMP(1);
    // ---- y_uk = sum_{j in desc*(k)} w_j (x_uj - tg_k) for the live joints: warps 1..3, while warp 0 does the normals ----
    if(tt >= 32)
      for(int u = tt - 32; u < npe * nlive; u += TEAM - 32)
      {
        const int q = u / nlive, li = u - q * nlive;
        const int k = s_live[li];
        const f3 tgk = mk3(s_G[12 * k + 3], s_G[12 * k + 7], s_G[12 * k + 11]);
        f3 y = mk3(0.f, 0.f, 0.f);
        for(int sl = 0; sl < kmax; sl++)
        {
          const int i = q * kmax + sl;
          const float wj = s_sw[i];
          if(wj != 0.f && ((p.anc_mask[s_sj[i]] >> k) & 1u)) y = y + (ld3(s_xw + 3 * i) - wj * tgk);
        }
        float * yo = s_y + 3 * (q * ML + li);
        yo[0] = y.x, yo[1] = y.y, yo[2] = y.z;
      }
    // ---- face normals of the ring items, vertex normals of the corners (SMPL::calcNormal / calcVertexNormal) ----
    if(p.use_ring && tt < 32)
    {
      for(int it0 = tt; it0 < nie; it0 += 32)
      {
        const uint8_t * it = s_rec->item[it0];
        float inv;
        const f3 nn = face_normal(ld3(s_pv + 3 * it[0]), ld3(s_pv + 3 * it[1]), ld3(s_pv + 3 * it[2]), inv);
        s_itemN[4 * it0] = nn.x, s_itemN[4 * it0 + 1] = nn.y, s_itemN[4 * it0 + 2] = nn.z, s_itemN[4 * it0 + 3] = inv;
      }
      __syncwarp(); // items, corners and the task are chained inside warp 0
      if(tt < 3 && rec_ok)
      {
        int s0 = 0;
        for(int c = 0; c < tt; c++) s0 += s_rec->nic[c];
        float inv;
        const f3 nn = corner_normal(s0, s0 + s_rec->nic[tt], [&](int it) { return ld3(s_itemN + 4 * it); }, inv);
        s_cornN[4 * tt] = nn.x, s_cornN[4 * tt + 1] = nn.y, s_cornN[4 * tt + 2] = nn.z, s_cornN[4 * tt + 3] = inv;
      }
      __syncwarp();
    }
    // ---- the task: actual position, re-weighting (node.cpp:803-804), residual (:807-820), phi columns ----
    if(tt == 0)
    {
      f3 v[3], nc[3];
      for(int c = 0; c < 3; c++)
      {
        v[c] = rec_ok ? ld3(s_pv + 3 * c) : mk3(0.f, 0.f, 0.f);
        nc[c] = p.use_ring ? ld3(s_cornN + 4 * c) : mk3(0.f, 0.f, 0.f);
      }
      // reweight_task, task_residual, store_task_scratch, phi_frame / phi_column (ik_math.cuh) written inline: through the
      // helpers ptxas spills 4-12 more bytes in this kernel
      const float w[3] = {s_tin[3 * m], s_tin[3 * m + 1], s_tin[3 * m + 2]};
      f3 pos = w[0] * v[0] + w[1] * v[1] + w[2] * v[2];
      float inv_s = 0.f;
      if(p.use_ring && p.normal_offset > 0.f)
        pos = pos + p.normal_offset * normalize_inv(w[0] * nc[0] + w[1] * nc[1] + w[2] * nc[2], inv_s);
      float wn[3];
      triangle_weights(pos, v[0], v[1], v[2], wn);
      if(p.update_weights && live_frame)
        p.vertex_weights[3 * fm] = wn[0], p.vertex_weights[3 * fm + 1] = wn[1], p.vertex_weights[3 * fm + 2] = wn[2];
      f3 nh = mk3(0.f, 0.f, 0.f);
      if(p.use_ring) nh = normalize_inv(wn[0] * nc[0] + wn[1] * nc[1] + wn[2] * nc[2], inv_s);
      f3 pn = wn[0] * v[0] + wn[1] * v[1] + wn[2] * v[2];
      if(p.normal_offset > 0.f) pn = pn + p.normal_offset * nh;
      const float posw = s_tin[6 * n + m];
      const f3 tgt = ld3(s_tin + 3 * n + 3 * m);
      const f3 nt = ROWS == 4 ? ld3(s_tin + 7 * n + 3 * m) : mk3(0.f, 0.f, 1.f);
      float e[4] = {posw * (pn.x - tgt.x), posw * (pn.y - tgt.y), posw * (pn.z - tgt.z),
                    p.normal_task_weight > 0.f ? p.normal_task_weight * (dot3(nh, nt) + 1.f) : 0.f};
      if(!rec_ok) e[0] = e[1] = e[2] = e[3] = CUDART_NAN_F; // attachment outside the record limits: numerical-issue status
      if(p.e_out && live_frame)
      {
        float * eo = p.e_out + static_cast<size_t>(f) * 4 * n + 4 * m;
        eo[0] = e[0], eo[1] = e[1], eo[2] = e[2], eo[3] = e[3];
      }
      if(!(isfinite(e[0]) && isfinite(e[1]) && isfinite(e[2]) && isfinite(e[3]))) bad = 1;
      if(posw > 0.f) valid++;
#pragma unroll
      for(int r = 0; r < 4; r++) esq += static_cast<double>(e[r]) * static_cast<double>(e[r]);
      float * ts = s_ts;
      ts[0] = wn[0], ts[1] = wn[1], ts[2] = wn[2];
      ts[3] = nh.x, ts[4] = nh.y, ts[5] = nh.z, ts[6] = inv_s, ts[7] = posw;
      ts[8] = nt.x, ts[9] = nt.y, ts[10] = nt.z;
      ts[12] = e[0], ts[13] = e[1], ts[14] = e[2], ts[15] = e[3];
      if(p.phi_cols)
      {
        // d w' / d pos (pos = detached actual position + tangents phi, IkTask.cpp:49-57), tangents (:33-47)
        const f3 r0 = cross3(v[1] - pos, v[2] - pos), r1 = cross3(v[2] - pos, v[0] - pos), r2 = cross3(v[0] - pos, v[1] - pos);
        const float a0 = norm3(r0), a1 = norm3(r1), a2 = norm3(r2), S = a0 + a1 + a2;
        const f3 g0 = cross3((1.f / a0) * r0, v[2] - v[1]), g1 = cross3((1.f / a1) * r1, v[0] - v[2]),
                 g2 = cross3((1.f / a2) * r2, v[1] - v[0]);
        const f3 gs = g0 + g1 + g2;
        const f3 dw[3] = {(1.f / S) * (g0 - wn[0] * gs), (1.f / S) * (g1 - wn[1] * gs), (1.f / S) * (g2 - wn[2] * gs)};
        const f3 t1 = v[1] - v[0];
        const f3 nrm = cross3(t1, v[2] - v[0]);
        const f3 t2 = cross3(nrm, t1);
        float dummy;
        const f3 tang[2] = {normalize_inv(t1, dummy), normalize_inv(t2, dummy)};
        for(int k = 0; k < 2; k++)
        {
          const float dwk[3] = {dot3(dw[0], tang[k]), dot3(dw[1], tang[k]), dot3(dw[2], tang[k])};
          f3 dp = dwk[0] * v[0] + dwk[1] * v[1] + dwk[2] * v[2];
          f3 dn = mk3(0.f, 0.f, 0.f);
          if(p.use_ring) dn = proj_apply(nh, inv_s, dwk[0] * nc[0] + dwk[1] * nc[1] + dwk[2] * nc[2]);
          if(p.normal_offset > 0.f) dp = dp + p.normal_offset * dn;
          const int col = phi_off_f + 2 * m + k;
          s_Jrow[0 * ldf + col] = posw * dp.x;
          s_Jrow[1 * ldf + col] = posw * dp.y;
          s_Jrow[2 * ldf + col] = posw * dp.z;
          s_Jrow[3 * ldf + col] = p.normal_task_weight > 0.f ? p.normal_task_weight * dot3(nt, dn) : 0.f;
        }
      }
    }
    team_sync(team);
    IK2_STAMP(2);
    // ---- d(normal) / d(vertex): one thread per (item, slot) reference, then a fixed-order sum per pair ----
    if(p.use_ring)
    {
      if(tt < 3 * nie)
      {
        const int it = tt / 3, slot = tt - 3 * it;
        const uint8_t * iv = s_rec->item[it];
        const int c = iv[3];
        const float wg = 1.f / static_cast<float>(s_rec->nic[c]);
        const float scale = s_ts[c] * wg;
        const f3 nh = mk3(s_ts[3], s_ts[4], s_ts[5]);
        const float inv_s = s_ts[6];
        f3 ax[3];
        ref_edge_cross(ld3(s_pv + 3 * iv[0]), ld3(s_pv + 3 * iv[1]), ld3(s_pv + 3 * iv[2]), slot, ax);
        const f3 ng = ld3(s_itemN + 4 * it), nci = ld3(s_cornN + 4 * c);
        const float inv_g = s_itemN[4 * it + 3], inv_q = s_cornN[4 * c + 3];
        float * D = s_Dref + 9 * tt;
#pragma unroll
        for(int cc = 0; cc < 3; cc++)
        {
          const f3 y = proj_apply(nh, inv_s, proj_apply(nci, inv_q, proj_apply(ng, inv_g, ax[cc])));
          D[cc] = scale * y.x, D[3 + cc] = scale * y.y, D[6 + cc] = scale * y.z;
        }
      }
      team_sync(team);
    IK2_STAMP(3);
    }
    // ---- C4 = d(residual rows) / d(vertex) (4 x 3) per pair ----
    if(tt < npe)
    {
      float D[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if(p.use_ring)
      {
        for(int rf = s_rec->ref_off[tt]; rf < s_rec->ref_off[tt + 1]; rf++)
        {
          const int code = s_rec->refs[rf];
          const float * Dr = s_Dref + 9 * ((code >> 2) * 3 + (code & 3));
#pragma unroll
          for(int e = 0; e < 9; e++) D[e] += Dr[e];
        }
      }
      float * C = s_C4 + 12 * tt;
      c4_block<ROWS>(s_ts, tt, D, p.normal_offset, p.normal_task_weight, C);
      // CA4 = C4 . A_u (the pose-blend columns contract it with the basis rows)
      const float * Au = s_Au + 9 * tt;
      float * CA = s_CA4 + 12 * tt;
#pragma unroll
      for(int r = 0; r < 4; r++)
#pragma unroll
        for(int c = 0; c < 3; c++) CA[3 * r + c] = C[3 * r] * Au[c] + C[3 * r + 1] * Au[3 + c] + C[3 * r + 2] * Au[6 + c];
    }
    team_sync(team);
    IK2_STAMP(4);
    // ---- translation columns (last warp); kinematic-chain columns: sum_u C4_u M_kc y_uk  (thread = (live joint, row)) ----
    if(tt >= 96 && tt - 96 < 3 * ROWS)
    {
      const int r = (tt - 96) / 3, c = (tt - 96) - 3 * r;
      float acc = 0.f;
      for(int q = 0; q < npe; q++) acc += s_C4[12 * q + 3 * r + c];
      s_Jrow[r * ldf + c] = acc;
    }
    for(int u = tt; u < nlive * ROWS; u += TEAM)
    {
      const int li = u / ROWS, r = u - li * ROWS;
      const int k = s_live[li];
      float W[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for(int q = 0; q < npe; q++)
      {
        const float * C = s_C4 + 12 * q + 3 * r;
        const float * y = s_y + 3 * (q * ML + li);
        const float c0 = C[0], c1 = C[1], c2 = C[2], y0 = y[0], y1 = y[1], y2 = y[2];
        W[0] = fmaf(c0, y0, W[0]), W[1] = fmaf(c0, y1, W[1]), W[2] = fmaf(c0, y2, W[2]);
        W[3] = fmaf(c1, y0, W[3]), W[4] = fmaf(c1, y1, W[4]), W[5] = fmaf(c1, y2, W[5]);
        W[6] = fmaf(c2, y0, W[6]), W[7] = fmaf(c2, y1, W[7]), W[8] = fmaf(c2, y2, W[8]);
      }
#pragma unroll
      for(int c = 0; c < 3; c++)
      {
        const float * Mk = s_M + 9 * (3 * k + c);
        float acc = 0.f;
#pragma unroll
        for(int e = 0; e < 9; e++) acc = fmaf(Mk[e], W[e], acc);
        s_Jrow[r * ldf + 3 + 3 * k + c] = acc;
      }
    }
    // ---- beta columns, rigid part: sum_u C4_u sum_j w_j d t'_j / d beta_i  (thread = (beta, row)) ----
    if(p.beta_cols)
    {
      for(int u = tt; u < kShapeDim * ROWS; u += TEAM)
      {
        const int ib = u / ROWS, r = u - ib * ROWS;
        float out = 0.f;
        for(int q = 0; q < npe; q++)
        {
          f3 y = mk3(0.f, 0.f, 0.f);
          for(int sl = 0; sl < kmax; sl++)
          {
            const int i = q * kmax + sl;
            const float wj = s_sw[i];
            const int j = s_sj[i];
            if(wj != 0.f)
              y = y + wj * mk3(s_dTp[(3 * j) * kShapeDim + ib], s_dTp[(3 * j + 1) * kShapeDim + ib], s_dTp[(3 * j + 2) * kShapeDim + ib]);
          }
          const float * C = s_C4 + 12 * q + 3 * r;
          out += C[0] * y.x + C[1] * y.y + C[2] * y.z;
        }
        s_Jrow[r * ldf + beta_off_f + ib] = out;
      }
    }
    team_sync(team);
    IK2_STAMP(5);
    // ---- pose-blend (and shape-blend) columns, step 1: Q = sum_u CA4_u P_u (ROWS x 224); lane owns two columns ----
    {
      const int col = 2 * (32 * tw + lane);
      if(col < kBlendK)
      {
        float qa[ROWS], qb[ROWS];
#pragma unroll
        for(int r = 0; r < ROWS; r++) qa[r] = qb[r] = 0.f;
        for(int q = 0; q < npe; q++)
        {
          float2 px, py, pz;
          if(STAGED)
          {
            const int slot = ring_pos + q < R ? ring_pos + q : ring_pos + q - R;
            const float * P = reinterpret_cast<const float *>(ring_base + static_cast<size_t>(slot) * PAIR_BYTES) + col;
            px = *reinterpret_cast<const float2 *>(P);
            py = *reinterpret_cast<const float2 *>(P + kBlendK);
            pz = *reinterpret_cast<const float2 *>(P + 2 * kBlendK);
          }
          else
          {
            const float * P = p.basis + static_cast<size_t>(s_rec->gv[q]) * (3 * kBlendK) + col;
            px = __ldg(reinterpret_cast<const float2 *>(P));
            py = __ldg(reinterpret_cast<const float2 *>(P + kBlendK));
            pz = __ldg(reinterpret_cast<const float2 *>(P + 2 * kBlendK));
          }
          const float4 * C4 = reinterpret_cast<const float4 *>(s_CA4 + 12 * q);
          const float4 c0 = C4[0], c1 = C4[1], c2 = C4[2];
          const float C[12] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w, c2.x, c2.y, c2.z, c2.w};
#pragma unroll
          for(int r = 0; r < ROWS; r++)
          {
            qa[r] = fmaf(C[3 * r], px.x, fmaf(C[3 * r + 1], py.x, fmaf(C[3 * r + 2], pz.x, qa[r])));
            qb[r] = fmaf(C[3 * r], px.y, fmaf(C[3 * r + 1], py.y, fmaf(C[3 * r + 2], pz.y, qb[r])));
          }
        }
#pragma unroll
        for(int r = 0; r < ROWS; r++) *reinterpret_cast<float2 *>(s_Q + r * kBlendK + col) = make_float2(qa[r], qb[r]);
      }
      if(STAGED)
      {
        __syncwarp();
        if(lane == 0) ptx::mbar_arrive(bar_done + (m % NBAR)); // this warp is done with the task's ring slots
        ring_pos = ring_pos + npe < R ? ring_pos + npe : ring_pos + npe - R;
      }
    }
    team_sync(team);
    IK2_STAMP(6);
    // ---- step 2: J[r][3 + 3k + c] += sum_e Q[r][9(k-1)+e] dvec(R_k)/dtheta_kc [e];  beta columns += Q[r][207 + i] ----
    for(int u = tt; u < 69 * ROWS; u += TEAM)
    {
      const int r = u / 69, kc = u - 69 * r;
      const int k = kc / 3 + 1, c = kc - 3 * (k - 1);
      const float * Qr = s_Q + r * kBlendK + 9 * (k - 1);
      const float * dv = s_dR + 27 * k + 9 * c;
      float acc = 0.f;
#pragma unroll
      for(int e = 0; e < 9; e++) acc = fmaf(Qr[e], dv[e], acc);
      s_Jrow[r * ldf + 3 + 3 * k + c] += acc;
    }
    if(p.beta_cols)
      for(int u = tt; u < kShapeDim * ROWS; u += TEAM)
      {
        const int ib = u / ROWS, r = u - ib * ROWS;
        s_Jrow[r * ldf + beta_off_f + ib] += s_Q[r * kBlendK + kPoseDim + ib];
      }
    team_sync(team);
    IK2_STAMP(7);
    // ---- VPoser: contract the 63 body columns with d(axis-angle)/d(latent) (node.cpp:761-772) ----
    const float * Jsrc = s_Jrow;
    if(p.vposer)
    {
      for(int u = tt; u < ROWS * 32; u += TEAM)
      {
        const int r = u >> 5, t = u & 31;
        const float * jr = s_Jrow + r * ldf + 6;
        float acc = 0.f;
#pragma unroll 7
        for(int q = 0; q < 63; q++) acc = fmaf(jr[q], __ldg(Jv + q * 32 + t), acc);
        s_Jc[r * ld + 6 + t] = acc;
      }
      const int extra = p.php + (p.beta_cols ? 12 : 0);
      for(int u = tt; u < ROWS * (12 + extra); u += TEAM)
      {
        const int r = u / (12 + extra), c = u - r * (12 + extra);
        int src, dst;
        if(c < 6)
          src = c, dst = c;
        else if(c < 12)
          src = 63 + c, dst = 32 + c;
        else
          src = 76 + (c - 12), dst = 44 + (c - 12);
        s_Jc[r * ld + dst] = s_Jrow[r * ldf + src];
      }
      Jsrc = s_Jc;
      team_sync(team);
    IK2_STAMP(8);
    }
    // ---- the task's rows in the reference layout (the "Jacobian getter") ----
    if(p.j_out && live_frame)
    {
      float * jo = p.j_out + (static_cast<size_t>(f) * 4 * n + 4 * m) * p.dim_ref;
      for(int u = tt; u < 4 * p.dim_ref; u += TEAM)
      {
        const int r = u / p.dim_ref, c = u - r * p.dim_ref;
        float v = 0.f;
        if(r < ROWS)
        {
          if(c < p.theta_dim)
            v = Jsrc[r * ld + c];
          else if(c < p.theta_dim + 2 * n)
            v = p.phi_cols ? Jsrc[r * ld + p.thp + (c - p.theta_dim)] : 0.f;
          else if(p.beta_cols)
            v = Jsrc[r * ld + p.thp + p.php + (c - p.theta_dim - 2 * n)];
        }
        jo[u] = v;
      }
    }
    // ---- A += J'J (fp64, 4x4 tiles of the lower triangle), b += J'e; next task's record ----
    {
      if(m + 1 < n && tt < static_cast<int>(sizeof(TaskRec) / 16))
        reinterpret_cast<uint4 *>(base + L.rec)[tt] = __ldg(reinterpret_cast<const uint4 *>(grec + m + 1) + tt);
      if(m + 1 < n && gskin && tt >= 48 && tt - 48 < skin_bytes / 16)
        reinterpret_cast<uint4 *>(base + L.skin)[tt - 48] = __ldg(reinterpret_cast<const uint4 *>(gskin + m + 1) + (tt - 48));
      auto accum_tile = [&](int tl, int bi, int bj) {
        double * T = s_A + tl;
        double acc[16];
#pragma unroll
        for(int e = 0; e < 16; e++) acc[e] = T[e * NT];
#pragma unroll
        for(int r = 0; r < ROWS; r++)
        {
          const float4 ja = *reinterpret_cast<const float4 *>(Jsrc + r * ld + 4 * bi);
          const float4 jb = *reinterpret_cast<const float4 *>(Jsrc + r * ld + 4 * bj);
          const double a4[4] = {ja.x, ja.y, ja.z, ja.w};
          const double b4[4] = {jb.x, jb.y, jb.z, jb.w};
#pragma unroll
          for(int a = 0; a < 4; a++)
#pragma unroll
            for(int b = 0; b < 4; b++) acc[4 * a + b] = fma(a4[a], b4[b], acc[4 * a + b]);
        }
#pragma unroll
        for(int e = 0; e < 16; e++) T[e * NT] = acc[e];
      };
      if(tt < ntiles_acc) accum_tile(tt, my_bi[0], my_bj[0]);
      if(tt + TEAM < ntiles_acc) accum_tile(tt + TEAM, my_bi[1], my_bj[1]);
      for(int tl = tt + 2 * TEAM; tl < ntiles_acc; tl += TEAM)
      {
        int bi, bj;
        tri_coords(tl, bi, bj);
        accum_tile(tl, bi, bj);
      }
      for(int c = tt; c < p.Dp; c += TEAM)
      {
        double acc = 0.0;
#pragma unroll
        for(int r = 0; r < ROWS; r++) acc = fma(static_cast<double>(Jsrc[r * ld + c]), static_cast<double>(s_ts[12 + r]), acc);
        s_b[c] += acc;
      }
    }
    team_sync(team);
    IK2_STAMP(9);
  }

  IK2_STAMP(30);
  // =========================================================================================================
  // normal equations complete: damping, prior, solve, update  (node.cpp:887-968)
  // =========================================================================================================
  if(tt == 0) s_misc[0] = esq, s_misc[1] = valid, s_misc[2] = bad, s_misc[3] = 1.0;
  team_sync(team);
    IK2_STAMP(10);
  esq = s_misc[0];
  valid = static_cast<int>(s_misc[1]);
  bad = static_cast<int>(s_misc[2]);
  volatile int * s_ok = reinterpret_cast<volatile int *>(s_misc + 7);
  volatile int * s_flag = s_ok + 1;
  if(tt == 0) s_ok[0] = 1, s_flag[0] = 0;
  const bool too_few = p.skip_if_too_few && valid < n / 2; // node.cpp:785
  const int Dp = p.Dp, thp = p.thp, php = p.php;
  const int beta_off = thp + php;
  const int nb = Dp >> 2;
  // category of a compact position: 0 theta, 1 phi, 2 beta, -1 padding
  auto category = [&](int i) -> int {
    if(i < p.theta_dim) return 0;
    if(i < thp) return -1;
    if(i < thp + p.phi_cols) return 1;
    if(i < beta_off) return -1;
    if(i < beta_off + p.beta_cols) return 2;
    return -1;
  };
  for(int i = tt; i < Dp; i += TEAM)
  {
    const int cat = category(i);
    double add;
    if(cat < 0)
      add = (p.schur && i >= beta_off) ? 0.0 : 1.0; // padding unknown: identity row (never a pivot inside the beta block of the Schur stage)
    else
    {
      const double reg = cat == 0 ? p.reg_theta : (cat == 1 ? p.reg_phi : p.reg_beta);
      add = reg + esq;
      if(p.schur && cat == 2) add = 0.0; // the beta block is damped once, globally, in the apply step
      if(p.vposer && cat == 0)
      {
        const double w = i < 6 ? 0.0 : (i >= p.theta_dim - 6 ? p.hand_reg : p.latent_reg);
        add += w;
        s_b[i] += w * static_cast<double>(p.theta_state[static_cast<size_t>(f) * p.theta_dim + i]);
      }
    }
    Aat(s_A, NT, i, i) += add;
  }
  team_sync(team);
  // compact position -> column of the reference layout [theta | phi (2n) | beta]
  auto ref_col = [&](int i) -> int {
    const int cat = category(i);
    if(cat == 0) return i;
    if(cat == 1) return p.theta_dim + (i - thp);
    if(cat == 2) return p.theta_dim + 2 * n + (i - beta_off);
    return -1;
  };
  if((p.a_out || p.b_out) && live_frame)
  {
    if(p.a_out)
    {
      double * Ao = p.a_out + static_cast<size_t>(f) * p.dim_ref * p.dim_ref;
      for(int i = tt; i < p.dim_ref * p.dim_ref; i += TEAM) Ao[i] = 0.0;
      team_sync(team);
      for(int u = tt; u < Dp * (Dp + 1) / 2; u += TEAM)
      {
        int r, c;
        tri_coords(u, r, c);
        const int rr = ref_col(r), cc = ref_col(c);
        if(rr < 0 || cc < 0) continue;
        const double v = Aat(s_A, NT, r, c);
        Ao[rr * p.dim_ref + cc] = v;
        Ao[cc * p.dim_ref + rr] = v;
      }
      if(!p.phi_cols)
        for(int i = tt; i < 2 * n; i += TEAM)
          Ao[(p.theta_dim + i) * p.dim_ref + p.theta_dim + i] = static_cast<double>(p.reg_phi) + esq;
    }
    if(p.b_out)
    {
      double * bo = p.b_out + static_cast<size_t>(f) * p.dim_ref;
      for(int i = tt; i < p.dim_ref; i += TEAM) bo[i] = 0.0;
      team_sync(team);
      for(int i = tt; i < Dp; i += TEAM)
      {
        const int c = ref_col(i);
        if(c >= 0) bo[c] = s_b[i];
      }
    }
    team_sync(team);
  }
  double * x = reinterpret_cast<double *>(base + L.sx);
  double * g = reinterpret_cast<double *>(base + L.sg);
  double * dstep = reinterpret_cast<double *>(base + L.sd);
  int * state = reinterpret_cast<int *>(base + L.sstate);

  if(p.schur)
  {
    // ---- shared-beta stage: partial Cholesky with b appended as an extra row, so that the elimination also produces
    //      y0 = L^-1 b_f and r = b_beta - Y' y0 ----
    for(int i = tt; i < Dp; i += TEAM) Aat(s_A, NT, Dp, i) = s_b[i];
    team_sync(team);
    const int npiv = beta_off; // thp (phi is off in this stage)
    team_cholesky(s_A, NT, p.nbt, npiv >> 2, tt, team, s_ok);
    const bool good = s_ok[0] && !bad && !too_few;
    if(live_frame)
    {
      double * out = p.schur_out + static_cast<size_t>(f) * 111;
      for(int i = tt; i < 111; i += TEAM)
      {
        double v = 0.0;
        if(good)
        {
          if(i < 100)
          {
            const int r = i / 10, c = i % 10;
            v = r >= c ? Aat(s_A, NT, beta_off + r, beta_off + c) : Aat(s_A, NT, beta_off + c, beta_off + r);
          }
          else if(i < 110)
            v = Aat(s_A, NT, Dp, beta_off + (i - 100));
          else
            v = esq;
        }
        out[i] = v;
      }
      // factor rows for the apply step, in the packed layout of shared_beta_apply_kernel (padding unknowns dropped):
      // L_ff (theta_dim), Y' rows (10 x theta_dim), y0 (theta_dim)
      const int td = p.theta_dim;
      const int P = td * (td + 1) / 2 + (p.beta_cols + 1) * td;
      double * fw = p.factor_ws + static_cast<size_t>(f) * P;
      const int nff = td * (td + 1) / 2;
      for(int u = tt; u < nff; u += TEAM)
      {
        int r, c;
        tri_coords(u, r, c);
        fw[u] = Aat(s_A, NT, r, c);
      }
      for(int u = tt; u < (p.beta_cols + 1) * td; u += TEAM)
      {
        const int r = u / td, c = u - r * td;
        fw[nff + u] = r < p.beta_cols ? Aat(s_A, NT, beta_off + r, c) : Aat(s_A, NT, Dp, c);
      }
      if(tt == 0) p.status[f] = too_few ? 1 : ((bad || !s_ok[0]) ? 2 : 0);
    }
    return;
  }

  // ---- bounds: which variables can be bound-active (node.cpp:911-929) ----
  const bool qp = p.enable_qp && (p.phi_cols > 0 || p.beta_cols > 0) && p.a_ws != nullptr;
  int status = 0;
  if(!qp)
  {
    team_cholesky(s_A, NT, nb, nb, tt, team, s_ok);
    for(int i = tt; i < Dp; i += TEAM) x[i] = -s_b[i];
    team_sync(team);
    if(s_ok[0]) warp_tiled_solve(s_A, NT, Dp, x, tt);
    team_sync(team);
    if(!s_ok[0]) status = 2;
  }
  else
  {
    // primal active-set on min 1/2 x'Ax + b'x, lo <= x <= hi (same iteration as the oracle's solve_box_qp)
    const int ntiles = nb * (nb + 1) / 2;
    double * A0 = p.a_ws + static_cast<size_t>(f_raw < p.B ? f_raw : 0) * NT * 16;
    volatile int * s_iter = s_flag + 1;
    volatile int * s_atmin = s_flag + 2;
    if(live_frame)
      for(int i = tt; i < NT * 16; i += TEAM) A0[i] = s_A[i];
    for(int i = tt; i < Dp; i += TEAM)
    {
      x[i] = 0.0;
      state[i] = category(i) < 0 ? 2 : 0; // padding unknowns stay pinned at 0
    }
    if(tt == 0) s_iter[0] = 0, s_atmin[0] = 0;
    team_sync(team);
    auto lim = [&](int i) -> double {
      const int cat = category(i);
      if(cat == 1) return static_cast<double>(p.phi_limit);
      if(cat == 2) return static_cast<double>(p.beta_limit);
      return INFINITY;
    };
    // a padding team has no A0 slot of its own: it re-reads the last frame's copy, which that frame's team may still be
    // writing - harmless, because nothing it computes is stored
    const double * Aref = live_frame ? A0 : p.a_ws + static_cast<size_t>(p.B - 1) * NT * 16;
    const int max_iter = 20 * Dp + 50;
    while(true)
    {
      for(int i = tt; i < Dp; i += TEAM)
      {
        double acc = s_b[i];
        for(int k = 0; k < Dp; k++) acc = fma(i >= k ? Aref[((i & 3) * 4 + (k & 3)) * NT + tile_idx(i >> 2, k >> 2)]
                                                     : Aref[((k & 3) * 4 + (i & 3)) * NT + tile_idx(k >> 2, i >> 2)],
                                              x[k], acc);
        g[i] = acc;
      }
      // masked copy: fixed variables become identity rows / columns
      for(int tl = tt; tl < ntiles; tl += TEAM)
      {
        int bi, bj;
        tri_coords(tl, bi, bj);
#pragma unroll
        for(int e = 0; e < 16; e++)
        {
          const int r = 4 * bi + (e >> 2), c = 4 * bj + (e & 3);
          const bool fixed = state[r] != 0 || state[c] != 0;
          s_A[e * NT + tl] = fixed ? (r == c ? 1.0 : 0.0) : Aref[e * NT + tl];
        }
      }
      team_sync(team);
      team_cholesky(s_A, NT, nb, nb, tt, team, s_ok);
      if(!s_ok[0])
      {
        status = 2;
        break;
      }
      for(int i = tt; i < Dp; i += TEAM) dstep[i] = state[i] != 0 ? 0.0 : -g[i];
      team_sync(team);
      warp_tiled_solve(s_A, NT, Dp, dstep, tt);
      team_sync(team);
      if(tt == 0)
      {
        double dmax = 0.0, xmax = 1.0;
        for(int i = 0; i < Dp; i++)
        {
          dmax = fmax(dmax, fabs(dstep[i]));
          xmax = fmax(xmax, fabs(x[i]));
        }
        int flag = 0;
        // s_atmin: the previous step was a full, unblocked Newton step, so x already minimises the objective on the
        // current face; the multiplier test follows directly (the re-solved step is rounding noise)
        if(s_atmin[0] || dmax <= 1e-14 * xmax)
        {
          int worst = -1;
          double worst_val = 1e-12;
          for(int i = 0; i < Dp; i++)
          {
            const double viol = state[i] == -1 ? -g[i] : (state[i] == 1 ? g[i] : 0.0);
            if(viol > worst_val) worst_val = viol, worst = i;
          }
          if(worst < 0)
            flag = 1; // optimal
          else
            state[worst] = 0;
          s_atmin[0] = 0;
        }
        else
        {
          double alpha = 1.0;
          int block = -1, side = 0;
          for(int i = 0; i < Dp; i++)
          {
            if(state[i] != 0) continue;
            const double l = lim(i);
            if(!isfinite(l)) continue;
            if(dstep[i] > 0.0)
            {
              const double a = (l - x[i]) / dstep[i];
              if(a < alpha) alpha = a, block = i, side = 1;
            }
            else if(dstep[i] < 0.0)
            {
              const double a = (-l - x[i]) / dstep[i];
              if(a < alpha) alpha = a, block = i, side = -1;
            }
          }
          for(int i = 0; i < Dp; i++)
            if(state[i] == 0) x[i] += alpha * dstep[i];
          s_atmin[0] = block < 0;
          if(block >= 0)
          {
            x[block] = side > 0 ? lim(block) : -lim(block);
            state[block] = lim(block) == 0.0 ? 2 : side;
          }
        }
        s_iter[0] = s_iter[0] + 1;
        if(s_iter[0] >= max_iter && !flag) flag = 2;
        s_flag[0] = flag;
      }
      team_sync(team);
      if(s_flag[0] == 1) break;
      if(s_flag[0] == 2)
      {
        status = 3;
        break;
      }
    }
    team_sync(team);
  }
  IK2_STAMP(31);
  if(bad) status = 2;
  if(status == 0 && too_few) status = 1;
  if(!live_frame) return;
  // ---- outputs + update (node.cpp:946-968) ----
  if(p.delta_out)
  {
    double * dout = p.delta_out + static_cast<size_t>(f) * p.dim_ref;
    for(int i = tt; i < p.dim_ref; i += TEAM) dout[i] = 0.0;
    team_sync(team);
    for(int i = tt; i < Dp; i += TEAM)
    {
      const int c = ref_col(i);
      if(c >= 0) dout[c] = status == 2 ? 0.0 : x[i];
    }
  }
  if(p.dphi_out)
    for(int i = tt; i < 2 * n; i += TEAM)
      p.dphi_out[static_cast<size_t>(f) * 2 * n + i] = (p.phi_cols && status != 2) ? static_cast<float>(x[thp + i]) : 0.f;
  if(p.update_state && status == 0)
  {
    for(int i = tt; i < p.theta_dim; i += TEAM)
      p.theta_state[static_cast<size_t>(f) * p.theta_dim + i] += static_cast<float>(x[i]);
    if(p.beta_cols && p.beta)
      for(int i = tt; i < p.beta_cols; i += TEAM)
        p.beta[static_cast<size_t>(f) * p.beta_stride + i] += static_cast<float>(x[beta_off + i]);
  }
  if(tt == 0) p.status[f] = status;
}

// ------------------------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------------------------
namespace sb
{
std::atomic<int> g_ik_variant{0};

int build_task_rec_host(const smplpp_model * model, int64_t face, TaskRec & r)
{
  std::memset(&r, 0, sizeof(r));
  const auto & faces = model->h_faces;
  const auto & aoff = model->h_adj_offset;
  const auto & afaces = model->h_adj_faces;
  int np = 3, ni = 0;
  for(int c = 0; c < 3; c++) r.gv[c] = faces[3 * face + c];
  for(int c = 0; c < 3; c++)
  {
    const int v = r.gv[c];
    int cnt = 0;
    for(int k = aoff[v]; k < aoff[v + 1]; k++)
    {
      if(ni >= kRecItems) return -1;
      const int g = afaces[k];
      for(int s = 0; s < 3; s++)
      {
        const int u = faces[3 * g + s];
        int q = -1;
        for(int i = 0; i < np; i++)
          if(r.gv[i] == u)
          {
            q = i;
            break;
          }
        if(q < 0)
        {
          if(np >= kRecPairs) return -1;
          q = np++;
          r.gv[q] = u;
        }
        r.item[ni][s] = static_cast<uint8_t>(q);
      }
      r.item[ni][3] = static_cast<uint8_t>(c);
      ni++, cnt++;
    }
    r.nic[c] = static_cast<uint8_t>(cnt);
  }
  int off = 0;
  for(int q = 0; q < np; q++)
  {
    r.ref_off[q] = static_cast<uint8_t>(off);
    for(int it = 0; it < ni; it++)
      for(int s = 0; s < 3; s++)
        if(r.item[it][s] == q) r.refs[off++] = static_cast<uint8_t>(it * 4 + s);
  }
  r.ref_off[np] = static_cast<uint8_t>(off);
  for(int q = 0; q < np; q++)
  {
    r.jmask |= model->h_vert_jmask[r.gv[q]];
    if(q < 3) r.jmask_corner |= model->h_vert_jmask[r.gv[q]];
  }
  r.face = static_cast<int32_t>(face);
  r.np = static_cast<uint8_t>(np);
  r.ni = static_cast<uint8_t>(ni);
  return 0;
}

void build_task_skin_host(const smplpp_model * model, const TaskRec & rec, TaskSkin & sk)
{
  std::memset(&sk, 0, sizeof(sk));
  for(int q = 0; q < kRecPairs; q++) sk.ws[q] = 1.f;
  for(int q = 0; q < rec.np; q++)
  {
    const int v = rec.gv[q];
    int k = 0;
    float sum = 0.f;
    for(int j = 0; j < kJoints; j++)
    {
      const float w = model->h_weights[static_cast<size_t>(v) * kJoints + j];
      sum += w; // joint order, as lbs_wsum
      if(w != 0.f && k < 4)
      {
        sk.w[q][k] = w;
        sk.j[q][k] = static_cast<uint8_t>(j);
        k++;
      }
    }
    sk.ws[q] = sum;
  }
}

size_t ik2_skin_bytes(int64_t batch, int n)
{
  return static_cast<size_t>(batch) * n * sizeof(TaskSkin);
}

int launch_task_topo(const ModelDev & d, cudaStream_t st, long long total, const int32_t * face_idx, TaskRec * out, TaskSkin * skins)
{
  task_topo_kernel<<<static_cast<unsigned>((total + 3) / 4), 128, 0, st>>>(total, face_idx, d.F, d.faces, d.adj_offset, d.adj_faces,
                                                                         d.vert_jmask, out, d.kmax <= 4 ? skins : nullptr,
                                                                         d.lbs_joint, d.lbs_weight, d.lbs_wsum, d.Vpad, d.kmax);
  SB_LAUNCHED();
  return SMPLPP_OK;
}

namespace
{
inline int up16(int v)
{
  return (v + 15) / 16 * 16;
}

// shared-memory plan: per-team arrays, then the ring and its barriers.  Returns false when not even one team fits.
bool plan_smem(Ik2Params & p, int rows, bool staged, int want_slots)
{
  Ik2Layout & L = p.L;
  int off = 0;
  auto takef = [&](int floats) {
    const int o = off;
    off += up16(floats * 4);
    return o;
  };
  L.theta = takef(76), L.beta = takef(12), L.coef = takef(kBlendK), L.R = takef(216), L.dR = takef(648), L.Jt = takef(72);
  L.G = takef(288), L.tp = takef(72), L.M = takef(648);
  L.JS = L.dTg = L.dTp = 0;
  if(p.beta_cols) L.JS = takef(720), L.dTg = takef(720), L.dTp = takef(720);
  p.ntile = (p.nbt * (p.nbt + 1) / 2) | 1; // odd: the 16 element planes of the tile storage start on different banks
  L.A = off, off += p.ntile * 16 * 8;
  L.bvec = off, off += up16((p.Dp + 4) * 8);
  L.misc = off, off += 128;
  L.tin = takef((rows == 4 ? 10 : 7) * p.n);
  const int scratch0 = off;
  L.rec = off, off += up16(static_cast<int>(sizeof(TaskRec)));
  L.skin = off, off += p.skins ? static_cast<int>(sizeof(TaskSkin)) : 0;
  const int MP = p.MP, MI = p.MI, ML = p.ML, kmax = p.kmax;
  // theta, beta, R and Jt (1504 B) are only read by the prologue: the small per-task arrays reuse that space when they fit
  {
    int dead = L.theta;
    const int dead_end = L.coef; // theta | beta
    auto take_dead = [&](int bytes, int & field) {
      if(dead + up16(bytes) <= dead_end)
        field = dead, dead += up16(bytes);
      else
        field = off, off += up16(bytes);
    };
    take_dead(16 * 4, L.ts);
    take_dead(12 * 4, L.cornN);
    take_dead(MP * kmax, L.sj);
  }
  L.pv = takef(3 * MP), L.pr = takef(3 * MP), L.sw = takef(MP * kmax), L.xw = takef(3 * MP * kmax);
  L.Au = takef(9 * MP), L.itemN = takef(4 * std::max(MI, 1));
  // d(normal)/d(vertex) contributions and Q are live in disjoint phases of a task
  L.Dref = L.Q = takef(std::max(27 * std::max(MI, 1), rows * kBlendK));
  L.ybuf = takef(3 * MP * ML);
  L.C4 = takef(12 * MP), L.CA4 = takef(12 * MP);
  L.live = off, off += up16(ML);
  L.Jrow = takef(4 * p.ldf);
  L.Jc = p.vposer ? takef(4 * p.ld) : L.Jrow;
  // solve temporaries alias the per-task scratch
  int so = scratch0;
  L.sx = so, so += up16(p.Dp * 8);
  L.sg = so, so += up16(p.Dp * 8);
  L.sd = so, so += up16(p.Dp * 8);
  L.sstate = so, so += up16(p.Dp * 4);
  off = std::max(off, so);
  L.team_bytes = up16(off);
  const int bar_bytes = 2 * k2::NBAR * 8;
  int F = k2::MAXF;
  for(; F >= 1; F--)
  {
    int ring = 0;
    if(staged)
    {
      const int room = k2::SMEM_LIMIT - F * L.team_bytes - bar_bytes - 16;
      if(room < p.MP * k2::PAIR_BYTES) continue;
      ring = std::min(room / k2::PAIR_BYTES, want_slots);
    }
    else if(F * L.team_bytes > k2::SMEM_LIMIT)
      continue;
    p.F = F;
    L.ring_off = F * L.team_bytes;
    L.ring_slots = ring;
    L.bar_off = L.ring_off + ring * k2::PAIR_BYTES;
    L.bar_off = (L.bar_off + 15) / 16 * 16;
    L.total = L.bar_off + bar_bytes;
    return true;
  }
  return false;
}
} // namespace

size_t ik2_rec_bytes(int64_t batch, int n)
{
  return static_cast<size_t>(batch) * n * sizeof(TaskRec);
}

size_t ik2_qp_ws_doubles(const Ik2Dims & d)
{
  const int nb = d.Dp / 4;
  return static_cast<size_t>((nb * (nb + 1) / 2) | 1) * 16;
}

Ik2Dims ik2_dims(int n, bool vposer, bool phi, bool beta)
{
  Ik2Dims d{};
  d.theta_dim = vposer ? 44 : 75;
  d.thp = (d.theta_dim + 3) / 4 * 4;
  d.phi_cols = phi ? 2 * n : 0;
  d.php = (d.phi_cols + 3) / 4 * 4;
  d.beta_cols = beta ? kShapeDim : 0;
  d.Dp = d.thp + d.php + (beta ? 12 : 0);
  d.ldf = 76 + d.php + (beta ? 12 : 0);
  d.ld = vposer ? d.Dp : d.ldf;
  return d;
}

int launch_ik_fused(const Ik2Call & c)
{
  const smplpp_ik_options * o = c.opt;
  const ModelDev & md = c.model->d;
  const smplpp_tasks * t = c.tasks;
  Ik2Params p{};
  p.topo = make_topo(md);
  for(int j = 0; j < kJoints; j++)
  {
    uint32_t m = 0;
    for(int k = j; k >= 0; k = md.parent[k]) m |= 1u << k;
    p.anc_mask[j] = m;
  }
  p.basis = md.basis, p.lbs_joint = md.lbs_joint, p.lbs_weight = md.lbs_weight, p.lbs_wsum = md.lbs_wsum;
  p.Vpad = md.Vpad, p.kmax = md.kmax;
  p.joint_template = md.joint_template, p.joint_shape = md.joint_shape;
  const bool per_frame = c.frame_recs != nullptr;
  p.recs = per_frame ? c.frame_recs : t->recs;
  p.skins = md.kmax <= 4 ? (per_frame ? c.frame_skins : t->skins) : nullptr;
  p.rec_stride = per_frame ? t->d.n : 0;
  p.n = t->d.n;
  const bool vposer = o->enable_vposer != 0;
  const bool phi = !c.schur && o->enable_phi && o->phi_limit > 0.f;
  const bool beta = c.schur || o->optimize_beta;
  const Ik2Dims dm = ik2_dims(p.n, vposer, phi, beta);
  p.use_ring = (o->normal_offset > 0.f || o->normal_task_weight > 0.f) ? 1 : 0;
  // per-frame records can hold any attachment of the mesh: size the scratch for the record limits
  p.MP = per_frame ? (p.use_ring ? kRecPairs : 3) : (p.use_ring ? t->maxPairs : 3);
  p.MI = per_frame ? (p.use_ring ? kRecItems : 0) : (p.use_ring ? t->maxItems : 0);
  p.ML = per_frame ? kJoints : t->maxLive;
  p.B = c.B;
  p.beta_cols = dm.beta_cols, p.phi_cols = dm.phi_cols, p.vposer = vposer ? 1 : 0;
  p.enable_qp = o->enable_qp, p.skip_if_too_few = o->skip_if_too_few, p.update_state = o->update_state;
  p.update_weights = 1;
  p.schur = c.schur ? 1 : 0;
  p.theta_dim = dm.theta_dim, p.thp = dm.thp, p.php = dm.php, p.Dp = dm.Dp, p.ldf = dm.ldf, p.ld = dm.ld;
  p.nbt = dm.Dp / 4 + (c.schur ? 1 : 0);
  p.dim_ref = dm.theta_dim + 2 * p.n + (o->optimize_beta ? kShapeDim : 0);
  p.normal_offset = o->normal_offset, p.normal_task_weight = o->normal_task_weight;
  p.reg_theta = o->delta_theta_reg, p.reg_phi = o->delta_phi_reg, p.reg_beta = o->delta_beta_reg;
  p.phi_limit = o->phi_limit, p.beta_limit = o->delta_beta_limit;
  p.latent_reg = o->vposer_latent_reg, p.hand_reg = o->vposer_hand_reg;
  p.theta75 = c.theta75, p.theta_state = c.theta_state, p.beta = c.beta, p.beta_stride = c.beta_stride;
  p.vertex_weights = c.vertex_weights, p.target_pos = c.target_pos, p.target_normal = c.target_normal;
  p.pos_task_weight = c.pos_task_weight, p.vposer_jac = c.vjac;
  p.status = c.status, p.e_out = c.e_out, p.j_out = c.j_out, p.a_out = c.a_out, p.b_out = c.b_out, p.delta_out = c.delta_out;
  p.dphi_out = c.dphi_out, p.a_ws = c.a_ws, p.schur_out = c.schur_out, p.factor_ws = c.factor_ws;
  p.dbg_cycles = nullptr;
#ifdef SMPLPP_IK2_DBG
  {
    static long long * dbg = nullptr;
    if(!dbg)
    {
      cudaMalloc(&dbg, 32 * sizeof(long long));
      cudaMemset(dbg, 0, 32 * sizeof(long long));
    }
    long long h[32];
    cudaMemcpy(h, dbg, sizeof(h), cudaMemcpyDeviceToHost);
    long long tot = 0;
    for(int i = 0; i < 32; i++) tot += h[i];
    if(tot > 0)
    {
      fprintf(stderr, "ik2 phase cycles (previous launch, team 0 of CTA 0):");
      for(int i = 0; i < 32; i++)
        if(h[i]) fprintf(stderr, " [%d] %lld", i, h[i]);
      fprintf(stderr, " total %lld\n", tot);
    }
    cudaMemset(dbg, 0, 32 * sizeof(long long));
    p.dbg_cycles = dbg;
  }
#endif
  const int rows = o->normal_task_weight > 0.f ? 4 : 3;
  const bool staged = !per_frame;
  if(!plan_smem(p, rows, staged, 3 * p.MP))
    return fail(SMPLPP_ERR_INVALID, "IkTask", "IK problem too large for one team per frame (shared memory)");
  const int threads = p.F * k2::TEAM + (staged ? 32 : 0);
  const int grid = (c.B + p.F - 1) / p.F;
#define SB_IK2(R, S)                                                                                                  \
  do                                                                                                                  \
  {                                                                                                                   \
    SB_CUDA(cudaFuncSetAttribute(ik_fused_kernel<R, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, p.L.total));      \
    ik_fused_kernel<R, S><<<grid, threads, p.L.total, c.st>>>(p);                                                      \
  } while(0)
  if(rows == 4 && staged)
    SB_IK2(4, true);
  else if(rows == 4)
    SB_IK2(4, false);
  else if(staged)
    SB_IK2(3, true);
  else
    SB_IK2(3, false);
#undef SB_IK2
  SB_LAUNCHED();
  return SMPLPP_OK;
}
} // namespace sb
