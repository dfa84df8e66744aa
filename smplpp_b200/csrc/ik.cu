// MoSh / MoSh++ IK step on sm_100a: batched replacement of the per-frame loop body of the reference's
// node/node.cpp:753-968 and of smplpp::IkTask (src/IkTask.cpp).
//
//   sparse forward      K1 (pose chain) + K2 (fused blend + skinning) on the compact rows of the task vertices
//   ik_jacobian_kernel  one CTA per frame: chain derivatives, task geometry (normals, re-weighting :803-804,
//                       residual :807-820) and the ANALYTIC Jacobian that the reference obtains row by row
//                       from Tensor::backward (:823-873)                                  -> e, J (fp32)
//   ik_solve_kernel     one CTA per frame: A = J'J, b = J'e in fp64 + damping + VPoser prior (:884-904),
//                       Cholesky / box-constrained active-set QP (:907-939), update (:946-968)
//   shared-beta stage   partial Cholesky (Schur complement onto the 10 betas), deterministic reduction,
//                       10-dim box QP, back-substitution (SURVEY §8e)
#include <algorithm>
#include <cmath>
#include <map>

#include "common.cuh"
#include "forward.cuh"
#include "ik2.cuh"
#include "ik_math.cuh"
#include "ik_solve.cuh"
#include "tasks.cuh"
#include "vposer.cuh"

using namespace sb;

// ------------------------------------------------------------------------------------------------------------
// standalone helpers of the API
// ------------------------------------------------------------------------------------------------------------
__global__ void triangle_weights_kernel(long long n, const float * __restrict__ pos, const float * __restrict__ tri,
                                        float * __restrict__ w)
{
  long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if(i >= n) return;
  float out[3];
  triangle_weights(ld3(pos + 3 * i), ld3(tri + 9 * i), ld3(tri + 9 * i + 3), ld3(tri + 9 * i + 6), out);
  w[3 * i] = out[0], w[3 * i + 1] = out[1], w[3 * i + 2] = out[2];
}

// IkTask::calcActualPos / calcActualNormal (src/IkTask.cpp:59-86) on a full vertex buffer: thread per (frame, task)
// face_idx: (n) int64 shared by all frames, or face_idx32 (B, n) int32 per frame (IkTask::faceIdx_ after the re-seating of
// node.cpp:993-1001).  dphi (B, n, 2), nullable: the point moves by tangents * phi (IkTask::calcTangents, IkTask.cpp:33-47;
// node.cpp:955-958).
__global__ void task_positions_kernel(const int32_t * __restrict__ faces, const int32_t * __restrict__ adj_offset,
                                      const int32_t * __restrict__ adj_faces, int V, int B, int n,
                                      const long long * __restrict__ face_idx, const int32_t * __restrict__ face_idx32,
                                      const float * __restrict__ verts, const float * __restrict__ weights, float offset,
                                      const float * __restrict__ dphi, float * __restrict__ pos_out, float * __restrict__ nrm_out)
{
  long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if(i >= static_cast<long long>(B) * n) return;
  int b = static_cast<int>(i / n), m = static_cast<int>(i % n);
  const float * vb = verts + static_cast<size_t>(b) * V * 3;
  const int f = face_idx32 ? face_idx32[i] : static_cast<int>(face_idx[m]);
  const float * w = weights + i * 3;
  f3 p = mk3(0.f, 0.f, 0.f), s = mk3(0.f, 0.f, 0.f);
  const bool need_n = offset > 0.f || nrm_out != nullptr;
  for(int c = 0; c < 3; c++)
  {
    int v = faces[3 * f + c];
    p = p + w[c] * ld3(vb + 3 * v);
    if(need_n)
    {
      int s0 = adj_offset[v], s1 = adj_offset[v + 1];
      float wg = 1.f / static_cast<float>(s1 - s0);
      f3 q = mk3(0.f, 0.f, 0.f);
      for(int k = s0; k < s1; k++)
      {
        int g = adj_faces[k];
        f3 a = ld3(vb + 3 * faces[3 * g]), bq = ld3(vb + 3 * faces[3 * g + 1]), cq = ld3(vb + 3 * faces[3 * g + 2]);
        float inv;
        q = q + wg * normalize_inv(cross3(bq - a, cq - a), inv);
      }
      float inv;
      s = s + w[c] * normalize_inv(q, inv);
    }
  }
  if(need_n)
  {
    float inv;
    f3 nh = normalize_inv(s, inv);
    if(offset > 0.f) p = p + offset * nh;
    if(nrm_out) nrm_out[3 * i] = nh.x, nrm_out[3 * i + 1] = nh.y, nrm_out[3 * i + 2] = nh.z;
  }
  if(dphi)
  {
    const f3 v0 = ld3(vb + 3 * faces[3 * f]), v1 = ld3(vb + 3 * faces[3 * f + 1]), v2 = ld3(vb + 3 * faces[3 * f + 2]);
    const f3 t1 = v1 - v0;
    const f3 t2 = cross3(cross3(t1, v2 - v0), t1);
    float inv;
    p = p + dphi[2 * i] * normalize_inv(t1, inv) + dphi[2 * i + 1] * normalize_inv(t2, inv);
  }
  pos_out[3 * i] = p.x, pos_out[3 * i + 1] = p.y, pos_out[3 * i + 2] = p.z;
}

// IkTask::calcTangents (src/IkTask.cpp:33-47): t1 = normalize(v1 - v0), t2 = normalize(((v1 - v0) x (v2 - v0)) x (v1 - v0));
// out (B, n, 3, 2) like IkTask::tangents_ (columns are the two tangents)
__global__ void task_tangents_kernel(const int32_t * __restrict__ faces, int V, int B, int n,
                                     const long long * __restrict__ face_idx, const int32_t * __restrict__ face_idx32,
                                     const float * __restrict__ verts, float * __restrict__ out)
{
  long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if(i >= static_cast<long long>(B) * n) return;
  const int b = static_cast<int>(i / n), m = static_cast<int>(i % n);
  const float * vb = verts + static_cast<size_t>(b) * V * 3;
  const int f = face_idx32 ? face_idx32[i] : static_cast<int>(face_idx[m]);
  const f3 v0 = ld3(vb + 3 * faces[3 * f]), v1 = ld3(vb + 3 * faces[3 * f + 1]), v2 = ld3(vb + 3 * faces[3 * f + 2]);
  const f3 t1r = v1 - v0;
  const f3 t2r = cross3(cross3(t1r, v2 - v0), t1r);
  float inv;
  const f3 t1 = normalize_inv(t1r, inv), t2 = normalize_inv(t2r, inv);
  float * o = out + 6 * i;
  o[0] = t1.x, o[1] = t2.x, o[2] = t1.y, o[3] = t2.y, o[4] = t1.z, o[5] = t2.z;
}

// VPoser state (B,44) -> theta rows 0,1 and 23,24 (node.cpp:761-772); rows 2..22 are written by the decoder
__global__ void theta_assemble_kernel(int B, const float * __restrict__ state, float * __restrict__ theta)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= B * 12) return;
  int b = i / 12, k = i % 12;
  theta[static_cast<size_t>(b) * 75 + (k < 6 ? k : 63 + k)] = state[static_cast<size_t>(b) * 44 + (k < 6 ? k : 32 + k)];
}

// ------------------------------------------------------------------------------------------------------------
// C1: per-frame residual + analytic Jacobian
// ------------------------------------------------------------------------------------------------------------
namespace c1
{
constexpr int THREADS = 256;    // FFMA pose-blend phase inside the kernel (125 registers)
constexpr int THREADS_TC = 384; // pose-blend columns left to ik_poseblend_tc_kernel (80 registers)
constexpr int TS = 16; // floats of per-task scratch
}

struct IkJacParams
{
  ChainTopo topo;
  uint32_t anc_mask[kJoints]; // bit k set when k is j or an ancestor of j
  TasksDev t;
  const float * joint_template;
  const float * joint_shape;
  int B;
  int use_ring;   // normals needed (normal_offset > 0 or normal task)
  int beta_cols;  // 10 or 0
  int phi_cols;   // 2n or 0
  int vposer;     // contract the 63 body columns with the decoder Jacobian
  int update_weights;
  float normal_offset, normal_task_weight;
  const float * theta;  // (B, 75) assembled theta
  const float * beta;   // (B, 10) stride beta_stride
  long long beta_stride;
  const float * verts;  // (B, nUse, 3) sparse forward output
  const float * rest;   // (B, nUse, 3)
  int nUse;
  float * vertex_weights;       // (B, n, 3) in/out
  const float * target_pos;     // (B, n, 3)
  const float * target_normal;  // (B, n, 3) or null
  const float * pos_task_weight; // (B, n) or null
  const float * vposer_jac;     // (B, 63, 32) or null
  float * e_out;   // (B, 4n)
  float * jfull;   // (B, 4n, ldfull) theta-space Jacobian [75 | phi | beta]; == jout when !vposer
  int ldfull;
  float * jout;    // (B, 4n, ld) compact Jacobian [thetaDim | phi | beta]
  int ld;
  int * frame_info; // (B, 2): valid marker count, non-finite flag
  // pose-blend columns on tensor cores (ik_poseblend_tc_kernel): this kernel then skips P5d (and P5e) and leaves
  // CA4 = d(residual rows) / d(rest vertex) and d vec(R_k) / d theta_k of every frame behind
  float * ca_out;        // (B, ca_stride): per task [4 row slots][32 * K-blocks], k = 3 * pair + axis; null: FFMA phase here
  const int * ca_slot_off; // (n + 1) first K-block of every task
  int ca_stride;
  float * dr_out;        // (B, 23, 28): s_dR of joints 1..23, rows padded to 16 bytes
};

// TC: the pose-blend columns are left to ik_poseblend_tc_kernel (P5d / P5e are not even compiled in: 125 -> fewer registers)
template<int ROWS, bool TC>
__global__ void __launch_bounds__(TC ? c1::THREADS_TC : c1::THREADS, 2) ik_jacobian_kernel(const IkJacParams p)
{
  using c1::TS;
  constexpr int THREADS = TC ? c1::THREADS_TC : c1::THREADS;
  extern __shared__ __align__(16) float sm[];
  const int tid = threadIdx.x;
  const int f = blockIdx.x;
  const TasksDev & t = p.t;
  const int n = t.n;
  // ---- shared memory carve-up ----
  float * s_theta = sm;                  // 76
  float * s_beta = s_theta + 76;         // 12
  float * s_R = s_beta + 12;             // 24*9
  float * s_dR = s_R + 216;              // 24*27
  float * s_Jt = s_dR + 648;             // 24*3
  float * s_G = s_Jt + 72;               // 24*12  [Rg | tg]
  float * s_tp = s_G + 288;              // 24*3   t' = tg - Rg Jt
  float * s_M = s_tp + 72;               // 72*9
  float * s_JS = s_M + 648;              // 24*30 (beta only)
  float * s_dTg = s_JS + (p.beta_cols ? 720 : 0);
  float * s_dTp = s_dTg + (p.beta_cols ? 720 : 0);
  float * s_C4 = s_dTp + (p.beta_cols ? 720 : 0);                // nPairs*12, 16-byte aligned (read as float4 in P5d)
  float * s_verts = s_C4 + 12 * t.nPairs;
  float * s_rest = s_verts + 3 * p.nUse;
  float * s_itemN = s_rest + 3 * p.nUse;                   // nItems*4
  float * s_cornN = s_itemN + (p.use_ring ? 4 * t.nItems : 0); // 3n*4
  float * s_task = s_cornN + (p.use_ring ? 12 * n : 0);        // n*TS
  float * s_sw = s_task + TS * n;                              // nUse*kmax   normalised skinning weights w_j / sum w
  float * s_xw = s_sw + p.nUse * t.kmax;                       // nUse*kmax*3 wn_j * x_uj (vertex carried by bone j)
  uint8_t * s_sj = reinterpret_cast<uint8_t *>(s_xw + 3 * p.nUse * t.kmax); // nUse*kmax joint ids
  // compact list of the (task, joint) pairs whose joint moves the task (P5b), 2-byte aligned after s_sj
  uint16_t * s_act = reinterpret_cast<uint16_t *>(s_sj + ((p.nUse * t.kmax + 1) & ~1));
  __shared__ int s_valid, s_bad, s_nact;

  if(tid == 0) s_valid = 0, s_bad = 0, s_nact = 0;
  for(int i = tid; i < 75; i += THREADS) s_theta[i] = p.theta[static_cast<size_t>(f) * 75 + i];
  if(tid < kShapeDim) s_beta[tid] = p.beta[static_cast<size_t>(f) * p.beta_stride + tid];
  {
    const float * gr = p.rest + static_cast<size_t>(f) * p.nUse * 3;
    for(int i = tid; i < 3 * p.nUse; i += THREADS) s_rest[i] = gr[i];
    for(int i = tid; i < p.nUse * t.kmax; i += THREADS)
    {
      s_sw[i] = t.sw_norm[i]; // W[u, slot] / sum_j W[u, j], [u][slot] like the shared-memory copy
      s_sj[i] = t.sj_flat[i];
    }
  }
  __syncthreads();

  // ---- P1: rotations, their derivatives, joints ----
  if(tid < kJoints)
  {
    const int j = tid;
    rodrigues_grad(s_theta[3 + 3 * j], s_theta[4 + 3 * j], s_theta[5 + 3 * j], s_R + 9 * j, s_dR + 27 * j);
#pragma unroll
    for(int k = 0; k < 3; k++)
    {
      float acc = p.joint_template[3 * j + k];
#pragma unroll
      for(int i = 0; i < kShapeDim; i++)
      {
        float js = p.joint_shape[(3 * j + k) * kShapeDim + i];
        acc = fmaf(js, s_beta[i], acc);
        if(p.beta_cols) s_JS[(3 * j + k) * kShapeDim + i] = js;
      }
      s_Jt[3 * j + k] = acc;
    }
  }
  __syncthreads();
  // ---- P2a: global transforms level by level (warp 0) ----
  if(tid < 32)
  {
    const int j = tid;
    const int parent = j < kJoints ? p.topo.parent[j] : -1;
    const int depth = j < kJoints ? p.topo.depth[j] : -1;
    for(int d = 0; d <= p.topo.max_depth; d++)
    {
      if(depth == d)
      {
        const float * R = s_R + 9 * j;
        float * G = s_G + 12 * j;
        if(parent < 0)
        {
          for(int r = 0; r < 3; r++)
          {
            G[4 * r] = R[3 * r], G[4 * r + 1] = R[3 * r + 1], G[4 * r + 2] = R[3 * r + 2];
            G[4 * r + 3] = s_Jt[3 * j + r];
          }
        }
        else
        {
          const float * P = s_G + 12 * parent;
          float tl[3] = {s_Jt[3 * j] - s_Jt[3 * parent], s_Jt[3 * j + 1] - s_Jt[3 * parent + 1],
                         s_Jt[3 * j + 2] - s_Jt[3 * parent + 2]};
          for(int r = 0; r < 3; r++)
          {
            float p0 = P[4 * r], p1 = P[4 * r + 1], p2 = P[4 * r + 2], p3 = P[4 * r + 3];
            for(int c = 0; c < 3; c++) G[4 * r + c] = p0 * R[c] + p1 * R[3 + c] + p2 * R[6 + c];
            G[4 * r + 3] = p0 * tl[0] + p1 * tl[1] + p2 * tl[2] + p3;
          }
        }
      }
      __syncwarp();
    }
    if(j < kJoints)
    {
      const float * G = s_G + 12 * j;
      for(int r = 0; r < 3; r++)
        s_tp[3 * j + r] = G[4 * r + 3] - (G[4 * r] * s_Jt[3 * j] + G[4 * r + 1] * s_Jt[3 * j + 1] + G[4 * r + 2] * s_Jt[3 * j + 2]);
    }
  }
  __syncthreads();
  // ---- skinning of the task vertices (LinearBlendSkinning.cpp:445-553 on the ~480 rows the tasks touch): the terms
  //      wn_j x_uj = (W[u,j] / sum W) (Rg_j rest_u + t'_j) are what the chain columns need anyway (P5b), their sum over
  //      the influences plus the root translation is the posed vertex - no skinning launch, no vertex round trip ----
  for(int u = tid; u < p.nUse; u += THREADS)
  {
    const f3 ru = ld3(s_rest + 3 * u);
    f3 v = mk3(s_theta[0], s_theta[1], s_theta[2]);
    f3 acc = mk3(0.f, 0.f, 0.f);
    for(int sl = 0; sl < t.kmax; sl++)
    {
      const int i = u * t.kmax + sl;
      const int j = s_sj[i];
      const float wj = s_sw[i];
      const float * G = s_G + 12 * j;
      const f3 x = mk3(wj * (G[0] * ru.x + G[1] * ru.y + G[2] * ru.z + s_tp[3 * j]),
                       wj * (G[4] * ru.x + G[5] * ru.y + G[6] * ru.z + s_tp[3 * j + 1]),
                       wj * (G[8] * ru.x + G[9] * ru.y + G[10] * ru.z + s_tp[3 * j + 2]));
      s_xw[3 * i] = x.x, s_xw[3 * i + 1] = x.y, s_xw[3 * i + 2] = x.z;
      acc = acc + x;
    }
    v = v + acc;
    s_verts[3 * u] = v.x, s_verts[3 * u + 1] = v.y, s_verts[3 * u + 2] = v.z;
  }
  // ---- P2b: M_kc = Rg_parent(k) dR_kc Rg_k^T  (d x_j / d theta_kc = M_kc (x_j - tg_k)) ----
  if(tid < 72)
  {
    const int k = tid / 3;
    const float * A = s_dR + 9 * tid;
    const float * Rk = s_G + 12 * k;
    const int parent = p.topo.parent[k];
    float T[9];
    if(parent < 0)
    {
      for(int e = 0; e < 9; e++) T[e] = A[e];
    }
    else
    {
      const float * P = s_G + 12 * parent;
      for(int a = 0; a < 3; a++)
        for(int e = 0; e < 3; e++) T[3 * a + e] = P[4 * a] * A[e] + P[4 * a + 1] * A[3 + e] + P[4 * a + 2] * A[6 + e];
    }
    for(int a = 0; a < 3; a++)
      for(int b = 0; b < 3; b++)
        s_M[9 * tid + 3 * a + b] = T[3 * a] * Rk[4 * b] + T[3 * a + 1] * Rk[4 * b + 1] + T[3 * a + 2] * Rk[4 * b + 2];
  }
  // ---- P2c: d tg_j / d beta and d t'_j / d beta (3x10 per joint).  One warp per beta component, lane = joint: the walk down
  //      the tree needs only warp barriers (it was a block barrier per level: a dozen of them with 240 busy threads) ----
  if(p.beta_cols)
  {
    const int j = tid & 31;
    const bool on = j < kJoints;
    const int parent = on ? p.topo.parent[j] : -1;
    const int depth = on ? p.topo.depth[j] : -1;
    for(int i = tid >> 5; i < kShapeDim; i += THREADS / 32)
    {
      for(int d = 0; d <= p.topo.max_depth; d++)
      {
        if(on && depth == d)
        {
          if(parent < 0)
          {
            for(int r = 0; r < 3; r++) s_dTg[(3 * j + r) * kShapeDim + i] = s_JS[(3 * j + r) * kShapeDim + i];
          }
          else
          {
            const float * P = s_G + 12 * parent;
            float dl[3];
            for(int r = 0; r < 3; r++) dl[r] = s_JS[(3 * j + r) * kShapeDim + i] - s_JS[(3 * parent + r) * kShapeDim + i];
            for(int r = 0; r < 3; r++)
              s_dTg[(3 * j + r) * kShapeDim + i] =
                  s_dTg[(3 * parent + r) * kShapeDim + i] + P[4 * r] * dl[0] + P[4 * r + 1] * dl[1] + P[4 * r + 2] * dl[2];
          }
        }
        __syncwarp();
      }
      if(on)
      {
        const float * G = s_G + 12 * j;
        float js[3] = {s_JS[(3 * j) * kShapeDim + i], s_JS[(3 * j + 1) * kShapeDim + i], s_JS[(3 * j + 2) * kShapeDim + i]};
        for(int r = 0; r < 3; r++)
          s_dTp[(3 * j + r) * kShapeDim + i] =
              s_dTg[(3 * j + r) * kShapeDim + i] - (G[4 * r] * js[0] + G[4 * r + 1] * js[1] + G[4 * r + 2] * js[2]);
      }
    }
  }
  __syncthreads(); // posed vertices complete
  // ---- P4 / G1: face normals of the ring items ----
  if(p.use_ring)
  {
    for(int it = tid; it < t.nItems; it += THREADS)
    {
      f3 v0 = ld3(s_verts + 3 * t.item_verts[3 * it]), v1 = ld3(s_verts + 3 * t.item_verts[3 * it + 1]),
         v2 = ld3(s_verts + 3 * t.item_verts[3 * it + 2]);
      float inv;
      f3 nn = normalize_inv(cross3(v1 - v0, v2 - v0), inv);
      s_itemN[4 * it] = nn.x, s_itemN[4 * it + 1] = nn.y, s_itemN[4 * it + 2] = nn.z, s_itemN[4 * it + 3] = inv;
    }
  }
  __syncthreads();
  // ---- G2: vertex normals of the corners (SMPL::calcVertexNormal) ----
  if(p.use_ring)
  {
    for(int ci = tid; ci < 3 * n; ci += THREADS)
    {
      int s0 = t.item_off[ci], s1 = t.item_off[ci + 1];
      float wg = 1.f / static_cast<float>(s1 - s0);
      f3 q = mk3(0.f, 0.f, 0.f);
      for(int it = s0; it < s1; it++) q = q + wg * ld3(s_itemN + 4 * it);
      float inv;
      f3 nn = normalize_inv(q, inv);
      s_cornN[4 * ci] = nn.x, s_cornN[4 * ci + 1] = nn.y, s_cornN[4 * ci + 2] = nn.z, s_cornN[4 * ci + 3] = inv;
    }
  }
  __syncthreads();
  // ---- G3: per task: actual position, re-weighting (node.cpp:803-804), residual (:807-820), phi columns ----
  float * Jf = p.jfull + static_cast<size_t>(f) * 4 * n * p.ldfull;
  for(int m = tid; m < n; m += THREADS)
  {
    const size_t fm = static_cast<size_t>(f) * n + m;
    f3 v[3], nc[3];
    for(int c = 0; c < 3; c++)
    {
      v[c] = ld3(s_verts + 3 * t.corner[3 * m + c]);
      nc[c] = p.use_ring ? ld3(s_cornN + 4 * (3 * m + c)) : mk3(0.f, 0.f, 0.f);
    }
    float w[3] = {p.vertex_weights[3 * fm], p.vertex_weights[3 * fm + 1], p.vertex_weights[3 * fm + 2]};
    f3 pos = w[0] * v[0] + w[1] * v[1] + w[2] * v[2];
    float inv_s = 0.f;
    if(p.use_ring && p.normal_offset > 0.f)
      pos = pos + p.normal_offset * normalize_inv(w[0] * nc[0] + w[1] * nc[1] + w[2] * nc[2], inv_s);
    float wn[3];
    triangle_weights(pos, v[0], v[1], v[2], wn);
    if(p.update_weights)
      p.vertex_weights[3 * fm] = wn[0], p.vertex_weights[3 * fm + 1] = wn[1], p.vertex_weights[3 * fm + 2] = wn[2];
    f3 nh = mk3(0.f, 0.f, 0.f);
    if(p.use_ring) nh = normalize_inv(wn[0] * nc[0] + wn[1] * nc[1] + wn[2] * nc[2], inv_s);
    f3 pn = wn[0] * v[0] + wn[1] * v[1] + wn[2] * v[2];
    if(p.normal_offset > 0.f) pn = pn + p.normal_offset * nh;
    const float posw = p.pos_task_weight ? p.pos_task_weight[fm] : 1.f;
    f3 tgt = ld3(p.target_pos + 3 * fm);
    f3 nt = p.target_normal ? ld3(p.target_normal + 3 * fm) : mk3(0.f, 0.f, 1.f);
    float e[4] = {posw * (pn.x - tgt.x), posw * (pn.y - tgt.y), posw * (pn.z - tgt.z),
                  p.normal_task_weight > 0.f ? p.normal_task_weight * (dot3(nh, nt) + 1.f) : 0.f};
    float * eo = p.e_out + static_cast<size_t>(f) * 4 * n + 4 * m;
    eo[0] = e[0], eo[1] = e[1], eo[2] = e[2], eo[3] = e[3];
    if(!(isfinite(e[0]) && isfinite(e[1]) && isfinite(e[2]) && isfinite(e[3]))) atomicOr(&s_bad, 1);
    if(posw > 0.f) atomicAdd(&s_valid, 1);
    float * ts = s_task + TS * m;
    ts[0] = wn[0], ts[1] = wn[1], ts[2] = wn[2];
    ts[3] = nh.x, ts[4] = nh.y, ts[5] = nh.z, ts[6] = inv_s, ts[7] = posw;
    ts[8] = nt.x, ts[9] = nt.y, ts[10] = nt.z;
    if(p.phi_cols)
    {
      // d w' / d pos (pos = detached actual position + tangents phi, IkTask.cpp:49-57), tangents (:33-47)
      f3 r0 = cross3(v[1] - pos, v[2] - pos), r1 = cross3(v[2] - pos, v[0] - pos), r2 = cross3(v[0] - pos, v[1] - pos);
      float a0 = norm3(r0), a1 = norm3(r1), a2 = norm3(r2), S = a0 + a1 + a2;
      f3 g0 = cross3((1.f / a0) * r0, v[2] - v[1]), g1 = cross3((1.f / a1) * r1, v[0] - v[2]),
         g2 = cross3((1.f / a2) * r2, v[1] - v[0]);
      f3 gs = g0 + g1 + g2;
      f3 dw[3] = {(1.f / S) * (g0 - wn[0] * gs), (1.f / S) * (g1 - wn[1] * gs), (1.f / S) * (g2 - wn[2] * gs)};
      f3 t1 = v[1] - v[0];
      f3 nrm = cross3(t1, v[2] - v[0]);
      f3 t2 = cross3(nrm, t1);
      float dummy;
      f3 tang[2] = {normalize_inv(t1, dummy), normalize_inv(t2, dummy)};
      for(int k = 0; k < 2; k++)
      {
        float dwk[3] = {dot3(dw[0], tang[k]), dot3(dw[1], tang[k]), dot3(dw[2], tang[k])};
        f3 dp = dwk[0] * v[0] + dwk[1] * v[1] + dwk[2] * v[2];
        f3 dn = mk3(0.f, 0.f, 0.f);
        if(p.use_ring) dn = proj_apply(nh, inv_s, dwk[0] * nc[0] + dwk[1] * nc[1] + dwk[2] * nc[2]);
        if(p.normal_offset > 0.f) dp = dp + p.normal_offset * dn;
        const int col = 75 + 2 * m + k;
        Jf[(4 * m + 0) * p.ldfull + col] = posw * dp.x;
        Jf[(4 * m + 1) * p.ldfull + col] = posw * dp.y;
        Jf[(4 * m + 2) * p.ldfull + col] = posw * dp.z;
        Jf[(4 * m + 3) * p.ldfull + col] = p.normal_task_weight > 0.f ? p.normal_task_weight * dot3(nt, dn) : 0.f;
      }
    }
  }
  // zero the phi columns of the other tasks' rows (J.middleCols(thetaDim, phiDim).setZero(), node.cpp:792)
  if(p.phi_cols)
  {
    for(int i = tid; i < 4 * n * p.phi_cols; i += THREADS)
    {
      int row = i / p.phi_cols, c = i % p.phi_cols;
      if(c / 2 != row / 4) Jf[row * p.ldfull + 75 + c] = 0.f;
    }
  }
  __syncthreads();
  // ---- G4: per (task, vertex) pair: C4 = d(residual rows) / d(vertex)  (ROWS x 3); also wn_j * x_uj ----
  // pairs in the order of decreasing reference count (pair_order): the lanes of a warp then run the same number of trips
  // (a corner is referenced by ~12 ring faces, a ring-only vertex by ~3: in pair order a warp ran at 1/3 efficiency)
  for(int ip0 = 0, round = 0; ip0 < t.nPairs; ip0 += THREADS, round++)
  {
    // odd rounds run backwards: the warp that had the heaviest vertices of one round gets the lightest of the next
    const int ip = ip0 + ((round & 1) ? THREADS - 1 - tid : tid);
    if(ip >= t.nPairs) continue;
    const int pr = t.pair_order[ip];
    const int m = t.pair_task[pr];
    const int q = pr - t.pair_off[m];
    float * C = s_C4 + 12 * pr;
    if(!p.use_ring && q >= 3)
    {
#pragma unroll
      for(int e = 0; e < 12; e++) C[e] = 0.f;
      continue;
    }
    const float * ts = s_task + TS * m;
    float D[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if(p.use_ring)
    {
      // d nh / d v = sum over the corners c, over the ring faces g of c that contain v:
      //   (w_c / deg_c) P(nh) P(n_c) P(n_g) [a]x      (P(n) x = (x - n (n.x)) / |unnormalised n|, a = the opposite edge)
      // the references of a pair are ordered by face and the faces by corner: P(n_g) [a]x is summed per corner first, the
      // two outer projections are applied once per (pair, corner)
      const f3 nh = mk3(ts[3], ts[4], ts[5]);
      const float inv_s = ts[6];
      int rf = t.pair_ref_off[pr];
      const int rf_end = t.pair_ref_off[pr + 1];
      int c = 0;
      while(rf < rf_end)
      {
        int it = t.pair_refs[rf] >> 2;
        while(it >= t.item_off[3 * m + c + 1]) c++;
        const int ci = 3 * m + c;
        const int it_end = t.item_off[ci + 1];
        f3 S[3] = {mk3(0.f, 0.f, 0.f), mk3(0.f, 0.f, 0.f), mk3(0.f, 0.f, 0.f)};
        do
        {
          const int slot = t.pair_refs[rf] & 3;
          f3 v0 = ld3(s_verts + 3 * t.item_verts[3 * it]), v1 = ld3(s_verts + 3 * t.item_verts[3 * it + 1]),
             v2 = ld3(s_verts + 3 * t.item_verts[3 * it + 2]);
          f3 e1 = v1 - v0, e2 = v2 - v0;
          f3 a = slot == 0 ? (e2 - e1) : (slot == 1 ? mk3(-e2.x, -e2.y, -e2.z) : e1);
          const f3 ng = ld3(s_itemN + 4 * it);
          const float inv_g = s_itemN[4 * it + 3];
          const f3 ax[3] = {mk3(0.f, a.z, -a.y), mk3(-a.z, 0.f, a.x), mk3(a.y, -a.x, 0.f)}; // a x e_c
#pragma unroll
          for(int cc = 0; cc < 3; cc++) S[cc] = S[cc] + proj_apply(ng, inv_g, ax[cc]);
          rf++;
          if(rf < rf_end) it = t.pair_refs[rf] >> 2;
        } while(rf < rf_end && it < it_end);
        const float scale = ts[c] / static_cast<float>(it_end - t.item_off[ci]);
        const f3 nci = ld3(s_cornN + 4 * ci);
        const float inv_q = s_cornN[4 * ci + 3];
#pragma unroll
        for(int cc = 0; cc < 3; cc++)
        {
          f3 y = proj_apply(nh, inv_s, proj_apply(nci, inv_q, S[cc]));
          D[cc] += scale * y.x, D[3 + cc] += scale * y.y, D[6 + cc] += scale * y.z;
        }
      }
    }
    const float posw = ts[7];
    const float wc = q < 3 ? ts[q] : 0.f; // pairs 0..2 of a task are its corners 0..2
#pragma unroll
    for(int r = 0; r < 3; r++)
#pragma unroll
      for(int c = 0; c < 3; c++) C[3 * r + c] = posw * (((r == c) ? wc : 0.f) + p.normal_offset * D[3 * r + c]);
    if(ROWS == 4)
    {
      const float nw = p.normal_task_weight;
#pragma unroll
      for(int c = 0; c < 3; c++) C[9 + c] = nw * (ts[8] * D[c] + ts[9] * D[3 + c] + ts[10] * D[6 + c]);
    }
    else
    {
      C[9] = C[10] = C[11] = 0.f;
    }
  }
  __syncthreads();
  if(tid == 0)
  {
    p.frame_info[2 * f] = s_valid;
    p.frame_info[2 * f + 1] = s_bad;
  }
  // ---- P5a: translation columns (d vert / d trans = I) and zero rows of inactive row slots ----
  for(int i = tid; i < n * 4 * 3; i += THREADS)
  {
    const int m = i / 12, r = (i / 3) % 4, c = i % 3;
    float acc = 0.f;
    if(r < ROWS)
    {
      const int p0 = t.pair_off[m];
      const int np = p.use_ring ? t.pair_off[m + 1] - p0 : 3;
      for(int q = 0; q < np; q++) acc += s_C4[12 * (p0 + q) + 3 * r + c];
    }
    Jf[(4 * m + r) * p.ldfull + c] = acc;
  }
  // ---- P5b: kinematic-chain columns: sum_u C4_u M_kc y_uk,  y_uk = sum_{j in desc*(k)} wn_j (x_uj - tg_k) ----
  // Only ~1/3 of the (task, joint) pairs are live (the joint must be an ancestor of a vertex of the task): they are
  // compacted first, so that the heavy loop below runs with full warps; the dead entries are zero-filled here.
  for(int i = tid; i < n * kJoints; i += THREADS)
  {
    const int m = i / kJoints, k = i % kJoints;
    const uint32_t mask = p.use_ring ? t.task_joint_mask[m] : t.task_joint_mask_corner[m];
    if((mask >> k) & 1u)
      s_act[atomicAdd(&s_nact, 1)] = static_cast<uint16_t>(i);
    else
    {
#pragma unroll
      for(int r = 0; r < 4; r++)
#pragma unroll
        for(int c = 0; c < 3; c++) Jf[(4 * m + r) * p.ldfull + 3 + 3 * k + c] = 0.f;
    }
  }
  __syncthreads();
  // two neighbouring lanes share a live (task, joint) pair: each sums half of the task's vertices (everything up to the
  // entries of J is linear in the per-vertex terms), the even lane adds the odd lane's result and stores.  330 live pairs
  // are 1.3 rounds of 256 threads; 660 half items are 2.6 rounds of half the length.
  const int nact2 = 2 * s_nact;
  for(int ia0 = 0; ia0 < nact2; ia0 += THREADS)
  {
    const int ia = ia0 + tid;
    const bool on = ia < nact2;
    const int half = ia & 1;
    const int i = s_act[on ? ia >> 1 : 0];
    const int m = i / kJoints, k = i % kJoints;
    float out[4][3];
#pragma unroll
    for(int r = 0; r < 4; r++) out[r][0] = out[r][1] = out[r][2] = 0.f;
    {
      float W[ROWS][9];
#pragma unroll
      for(int r = 0; r < ROWS; r++)
#pragma unroll
        for(int e = 0; e < 9; e++) W[r][e] = 0.f;
      const int p0 = t.pair_off[m];
      const int np = p.use_ring ? t.pair_off[m + 1] - p0 : 3;
      const f3 tgk = mk3(s_G[12 * k + 3], s_G[12 * k + 7], s_G[12 * k + 11]);
      const int q0 = on ? (half ? (np + 1) >> 1 : 0) : 0, q1 = on ? (half ? np : (np + 1) >> 1) : 0;
      for(int q = q0; q < q1; q++)
      {
        const int u = t.pair_vert[p0 + q];
        f3 y = mk3(0.f, 0.f, 0.f);
        for(int sl = 0; sl < t.kmax; sl++)
        {
          const int i = u * t.kmax + sl;
          const float wj = s_sw[i];
          if(wj != 0.f && ((p.anc_mask[s_sj[i]] >> k) & 1u)) y = y + (ld3(s_xw + 3 * i) - wj * tgk);
        }
        const float * C = s_C4 + 12 * (p0 + q);
#pragma unroll
        for(int r = 0; r < ROWS; r++)
#pragma unroll
          for(int a = 0; a < 3; a++)
          {
            W[r][3 * a] = fmaf(C[3 * r + a], y.x, W[r][3 * a]);
            W[r][3 * a + 1] = fmaf(C[3 * r + a], y.y, W[r][3 * a + 1]);
            W[r][3 * a + 2] = fmaf(C[3 * r + a], y.z, W[r][3 * a + 2]);
          }
      }
#pragma unroll
      for(int c = 0; c < 3; c++)
      {
        const float * M = s_M + 9 * (3 * k + c);
#pragma unroll
        for(int r = 0; r < ROWS; r++)
        {
          float acc = 0.f;
#pragma unroll
          for(int e = 0; e < 9; e++) acc = fmaf(M[e], W[r][e], acc);
          out[r][c] = acc;
        }
      }
    }
#pragma unroll
    for(int r = 0; r < 4; r++)
#pragma unroll
      for(int c = 0; c < 3; c++)
      {
        out[r][c] += __shfl_xor_sync(0xffffffffu, out[r][c], 1);
        if(on && !half) Jf[(4 * m + r) * p.ldfull + 3 + 3 * k + c] = out[r][c];
      }
  }
  // ---- P5c: beta columns, rigid part: sum_u C4_u sum_j wn_j d t'_j / d beta_i.  Four lanes per (task, beta component),
  //      each sums a quarter of the task's vertices (410 items were 1.07 rounds of 384 threads, the second nearly empty) ----
  if(p.beta_cols)
  {
    const int bcol = 75 + p.phi_cols;
    const int nitem4 = 4 * n * kShapeDim;
    for(int i0 = 0; i0 < nitem4; i0 += THREADS)
    {
      const int i4 = i0 + tid;
      const bool on = i4 < nitem4;
      const int part = i4 & 3, item = on ? i4 >> 2 : 0;
      const int m = item / kShapeDim, ib = item % kShapeDim;
      float out[4] = {0.f, 0.f, 0.f, 0.f};
      const int p0 = t.pair_off[m];
      const int np = p.use_ring ? t.pair_off[m + 1] - p0 : 3;
      const int q0 = on ? part * np / 4 : 0, q1 = on ? (part + 1) * np / 4 : 0;
      for(int q = q0; q < q1; q++)
      {
        const int u = t.pair_vert[p0 + q];
        f3 y = mk3(0.f, 0.f, 0.f);
        for(int sl = 0; sl < t.kmax; sl++)
        {
          const int i = u * t.kmax + sl;
          const float wj = s_sw[i];
          const int j = s_sj[i];
          if(wj != 0.f)
            y = y + wj * mk3(s_dTp[(3 * j) * kShapeDim + ib], s_dTp[(3 * j + 1) * kShapeDim + ib],
                             s_dTp[(3 * j + 2) * kShapeDim + ib]);
        }
        const float * C = s_C4 + 12 * (p0 + q);
#pragma unroll
        for(int r = 0; r < ROWS; r++) out[r] += C[3 * r] * y.x + C[3 * r + 1] * y.y + C[3 * r + 2] * y.z;
      }
#pragma unroll
      for(int r = 0; r < 4; r++)
      {
        out[r] += __shfl_xor_sync(0xffffffffu, out[r], 1);
        out[r] += __shfl_xor_sync(0xffffffffu, out[r], 2);
        if(on && part == 0) Jf[(4 * m + r) * p.ldfull + bcol + ib] = out[r];
      }
    }
  }
  __syncthreads();
  // ---- CA4 = C4 . A_u in place, A_u = sum_j wn_j Rg_j (the rotation part of the skinning matrix) ----
  for(int pr = tid; pr < t.nPairs; pr += THREADS)
  {
    if(!p.use_ring && pr - t.pair_off[t.pair_task[pr]] >= 3) continue; // ring-only vertices are not loaded
    const int u = t.pair_vert[pr];
    float A[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for(int sl = 0; sl < t.kmax; sl++)
    {
      const float wj = s_sw[u * t.kmax + sl];
      const float * G = s_G + 12 * s_sj[u * t.kmax + sl];
#pragma unroll
      for(int r = 0; r < 3; r++)
#pragma unroll
        for(int c = 0; c < 3; c++) A[3 * r + c] = fmaf(wj, G[4 * r + c], A[3 * r + c]);
    }
    float * C = s_C4 + 12 * pr;
    float out[12];
#pragma unroll
    for(int r = 0; r < 4; r++)
#pragma unroll
      for(int c = 0; c < 3; c++) out[3 * r + c] = C[3 * r] * A[c] + C[3 * r + 1] * A[3 + c] + C[3 * r + 2] * A[6 + c];
#pragma unroll
    for(int e = 0; e < 12; e++) C[e] = out[e];
    if constexpr(TC)
    {
      const int m = t.pair_task[pr], q = pr - t.pair_off[m];
      const int s0 = p.ca_slot_off[m], kp = 32 * (p.ca_slot_off[m + 1] - s0);
      float * dst = p.ca_out + static_cast<size_t>(f) * p.ca_stride + static_cast<size_t>(s0) * 128 + 3 * q;
#pragma unroll
      for(int r = 0; r < ROWS; r++)
#pragma unroll
        for(int a = 0; a < 3; a++) dst[r * kp + a] = out[3 * r + a];
    }
  }
  if constexpr(TC)
  {
    float * dst = p.dr_out + static_cast<size_t>(f) * 644; // [23 joints][28]: 27 entries + one pad (16-byte rows)
    for(int i = tid; i < 644; i += THREADS)
    {
      const int k = i / 28, e = i - 28 * k;
      dst[i] = e < 27 ? s_dR[27 * (k + 1) + e] : 0.f;
    }
    return; // P5d / P5e run as kernels of their own
  }
  else
  {
  __syncthreads();
  // ---- P5d: pose-blend (and shape-blend) columns: Q_m = sum_u CA4_u P_u (ROWS x 218), J += Q_m dvec(R_k)/dtheta.
  //      One warp per task; lanes 0..27 own EIGHT CONSECUTIVE basis columns each (8 x 28 = 224) of the K-major x / y / z
  //      rows of a vertex: a pair costs 6 16-byte loads + 3 broadcast loads for 24 * ROWS FMAs, and exactly the 2688
  //      bytes of the three rows cross L2 (the (x, y, z, 0) float4-per-column layout moved 3584; at 16384 frames this
  //      phase runs at the L2 -> SM bandwidth, so bytes are time).  The version before gave a lane two scattered columns:
  //      18 FMAs per pair and a segmented 4-level shuffle reduction per (row, axis) that cost as much as the contraction.
  //      The 9 columns of a joint always span exactly two neighbouring lanes: every lane forms the partial sums of the two
  //      joints its columns touch, the lane holding a joint's first column adds its right neighbour's piece (one shuffle
  //      per value) - a fixed order, so results stay bitwise reproducible. ----
  {
    const int warp = tid >> 5, lane = tid & 31;
    const int bcol = 75 + p.phi_cols;
    const int c_first = 8 * lane;                      // first owned column (lanes 28..31 own none)
    const bool has_cols = c_first < kBlendK;
    // slot A: the joint of the first column; slot B: the next joint, which the lane reaches into
    const int kA = c_first < kPoseDim ? c_first / 9 + 1 : 0;
    const int endA = 9 * kA;                           // first column behind joint kA
    // the joint this lane completes: the one whose first column lies in [c_first, c_first + 8)
    int kOwn = 0;
    if(c_first < kPoseDim)
    {
      const int kk = (c_first + 8) / 9 + 1;            // first joint starting at or after c_first
      if(9 * (kk - 1) < c_first + 8 && kk < kJoints) kOwn = kk;
    }
    const bool ownIsA = kOwn != 0 && kOwn == kA;       // the joint starts exactly at the lane's first column
    // derivative entries of the owned columns: dv[i][c] = d vec(R_k)[e] / d theta_kc
    float dv[8][3];
#pragma unroll
    for(int i = 0; i < 8; i++)
    {
      const int d = c_first + i;
      const bool on = d < kPoseDim;
      const int k = on ? d / 9 + 1 : 1, e = on ? d % 9 : 0;
#pragma unroll
      for(int c = 0; c < 3; c++) dv[i][c] = on ? s_dR[27 * k + 9 * c + e] : 0.f;
    }
    for(int m = warp; m < n; m += THREADS / 32)
    {
      float qacc[ROWS][8];
#pragma unroll
      for(int r = 0; r < ROWS; r++)
#pragma unroll
        for(int i = 0; i < 8; i++) qacc[r][i] = 0.f;
      const int p0 = t.pair_off[m];
      const int np = p.use_ring ? t.pair_off[m + 1] - p0 : 3;
      const uint32_t jmask = p.use_ring ? t.task_joint_mask[m] : t.task_joint_mask_corner[m];
      // the rigid part of the owned joint was written by P5b: fetch it now, the round trip overlaps the contraction
      float jprev[ROWS][3];
      if(kOwn)
      {
        const bool live = (jmask >> kOwn) & 1u;
#pragma unroll
        for(int r = 0; r < ROWS; r++)
#pragma unroll
          for(int c = 0; c < 3; c++) jprev[r][c] = live ? Jf[(4 * m + r) * p.ldfull + 3 + 3 * kOwn + c] : 0.f;
      }
      if(has_cols)
        for(int q = 0; q < np; q++)
        {
          const float * row = t.basis + static_cast<size_t>(3 * t.pair_vert[p0 + q]) * kBlendK + c_first;
          const float4 x0 = __ldg(reinterpret_cast<const float4 *>(row)), x1 = __ldg(reinterpret_cast<const float4 *>(row + 4));
          const float4 y0 = __ldg(reinterpret_cast<const float4 *>(row + kBlendK)), y1 = __ldg(reinterpret_cast<const float4 *>(row + kBlendK + 4));
          const float4 z0 = __ldg(reinterpret_cast<const float4 *>(row + 2 * kBlendK)), z1 = __ldg(reinterpret_cast<const float4 *>(row + 2 * kBlendK + 4));
          const float bx[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
          const float by[8] = {y0.x, y0.y, y0.z, y0.w, y1.x, y1.y, y1.z, y1.w};
          const float bz[8] = {z0.x, z0.y, z0.z, z0.w, z1.x, z1.y, z1.z, z1.w};
          const float4 * C4 = reinterpret_cast<const float4 *>(s_C4 + 12 * (p0 + q));
          const float4 c0 = C4[0], c1 = C4[1], c2 = C4[2];
          const float C[12] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w, c2.x, c2.y, c2.z, c2.w};
#pragma unroll
          for(int r = 0; r < ROWS; r++)
#pragma unroll
            for(int i = 0; i < 8; i++)
              qacc[r][i] = fmaf(C[3 * r], bx[i], fmaf(C[3 * r + 1], by[i], fmaf(C[3 * r + 2], bz[i], qacc[r][i])));
        }
      // partial sums of the two touched joints over the owned columns, combined with the right neighbour's slot A
#pragma unroll
      for(int r = 0; r < ROWS; r++)
#pragma unroll
        for(int c = 0; c < 3; c++)
        {
          float sa = 0.f, sb2 = 0.f;
#pragma unroll
          for(int i = 0; i < 8; i++)
          {
            const float v = qacc[r][i] * dv[i][c]; // dv = 0 on columns that are no pose feature
            if(c_first + i < endA)
              sa += v;
            else
              sb2 += v;
          }
          const float n1 = __shfl_down_sync(0xffffffffu, sa, 1);
          if(kOwn) Jf[(4 * m + r) * p.ldfull + 3 + 3 * kOwn + c] = jprev[r][c] + ((ownIsA ? sa : sb2) + n1);
        }
      // shape-blend columns 207..216 -> beta columns
      if(p.beta_cols)
      {
#pragma unroll
        for(int i = 0; i < 8; i++)
        {
          const int ib = c_first + i - kPoseDim;
          if(ib >= 0 && ib < kShapeDim)
          {
#pragma unroll
            for(int r = 0; r < ROWS; r++) Jf[(4 * m + r) * p.ldfull + bcol + ib] += qacc[r][i];
          }
        }
      }
    }
  }
  // ---- P5e: VPoser: contract the 63 body columns with d(axis-angle)/d(latent) (node.cpp:761-772) ----
  if(p.vposer)
  {
    __syncthreads();
    float * Jo = p.jout + static_cast<size_t>(f) * 4 * n * p.ld;
    const float * Jv = p.vposer_jac + static_cast<size_t>(f) * 63 * 32;
    const int extra = p.phi_cols + p.beta_cols;
    // thread = (task m, latent column tt): the decoder Jacobian entry is loaded once for the task's ROWS rows
    for(int i = tid; i < n * 32; i += THREADS)
    {
      const int m = i >> 5, tt = i & 31;
      const float * jr = Jf + (4 * m) * p.ldfull + 6;
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 7
      for(int q = 0; q < 63; q++)
      {
        const float v = __ldg(Jv + q * 32 + tt);
#pragma unroll
        for(int r = 0; r < ROWS; r++) acc[r] = fmaf(jr[r * p.ldfull + q], v, acc[r]);
      }
#pragma unroll
      for(int r = 0; r < 4; r++) Jo[(4 * m + r) * p.ld + 6 + tt] = acc[r];
    }
    for(int i = tid; i < 4 * n * (12 + extra); i += THREADS)
    {
      const int row = i / (12 + extra), c = i % (12 + extra);
      int src, dst;
      if(c < 6)
        src = c, dst = c;
      else if(c < 12)
        src = 63 + c, dst = 32 + c;
      else
        src = 75 + (c - 12), dst = 44 + (c - 12);
      Jo[row * p.ld + dst] = Jf[row * p.ldfull + src];
    }
  }
  } // !TC
}

// P5e of ik_jacobian_kernel as a kernel of its own (the pose-blend columns are added by ik_poseblend_tc_kernel between
// the two): contract the 63 body columns with d(axis-angle)/d(latent) (node.cpp:761-772), one CTA per frame.
// The frame's decoder Jacobian (63 x 32) and the body columns of its live rows sit in shared memory; warp = 16 rows, lane =
// latent column: per four body columns a lane reads 4 decoder entries and, as broadcasts, one float4 per row for 64 FMAs
// (the first version re-read both operands from L1 for every task: 0.88 ms per 16384 frames, now 0.3).
template<int ROWS>
__global__ void __launch_bounds__(256) ik_vposer_contract_kernel(int n, int extra, const float * __restrict__ jfull, int ldfull,
                                                                 const float * __restrict__ vposer_jac, float * __restrict__ jout,
                                                                 int ld)
{
  extern __shared__ __align__(16) float s_vc[];
  float * s_jv = s_vc;            // [64][32]: row 63 is zero
  float * s_j = s_vc + 64 * 32;   // [128][64]: body columns of up to 128 live rows, column 63 is zero
  const int tid = threadIdx.x, f = blockIdx.x, warp = tid >> 5, lane = tid & 31;
  const float * Jf = jfull + static_cast<size_t>(f) * 4 * n * ldfull;
  float * Jo = jout + static_cast<size_t>(f) * 4 * n * ld;
  const float * Jv = vposer_jac + static_cast<size_t>(f) * 63 * 32;
  const int nlive = n * ROWS;
  for(int i = tid; i < 64 * 32; i += 256) s_jv[i] = i < 63 * 32 ? __ldg(Jv + i) : 0.f;
  auto grow = [&](int l) { return 4 * (l / ROWS) + l % ROWS; }; // global row of live row l
  for(int l0 = 0; l0 < nlive; l0 += 128)
  {
    const int cnt = min(128, nlive - l0);
    __syncthreads(); // previous pass consumed
    for(int i = tid; i < 128 * 64; i += 256)
    {
      const int rl = i >> 6, q = i & 63;
      s_j[i] = (rl < cnt && q < 63) ? Jf[grow(l0 + rl) * ldfull + 6 + q] : 0.f;
    }
    __syncthreads();
    float acc[16];
#pragma unroll
    for(int r = 0; r < 16; r++) acc[r] = 0.f;
    const float4 * rows = reinterpret_cast<const float4 *>(s_j + warp * 16 * 64);
#pragma unroll 4
    for(int q4 = 0; q4 < 16; q4++)
    {
      const float v0 = s_jv[(4 * q4) * 32 + lane], v1 = s_jv[(4 * q4 + 1) * 32 + lane], v2 = s_jv[(4 * q4 + 2) * 32 + lane],
                  v3 = s_jv[(4 * q4 + 3) * 32 + lane];
#pragma unroll
      for(int r = 0; r < 16; r++)
      {
        const float4 a = rows[r * 16 + q4];
        acc[r] = fmaf(a.x, v0, fmaf(a.y, v1, fmaf(a.z, v2, fmaf(a.w, v3, acc[r]))));
      }
    }
#pragma unroll
    for(int r = 0; r < 16; r++)
    {
      const int rl = warp * 16 + r;
      if(rl < cnt) Jo[grow(l0 + rl) * ld + 6 + lane] = acc[r];
    }
  }
  // the other columns of the live rows: [trans | root] and the hands move, phi / beta columns follow
  for(int i = tid; i < nlive * (12 + extra); i += 256)
  {
    const int row = grow(i / (12 + extra)), c = i % (12 + extra);
    int src, dst;
    if(c < 6)
      src = c, dst = c;
    else if(c < 12)
      src = 63 + c, dst = 32 + c;
    else
      src = 75 + (c - 12), dst = 44 + (c - 12);
    Jo[row * ld + dst] = Jf[row * ldfull + src];
  }
  // row slots that carry no residual stay zero
  if(ROWS < 4)
    for(int i = tid; i < n * ld; i += 256) Jo[(4 * (i / ld) + 3) * ld + i % ld] = 0.f;
}

// ------------------------------------------------------------------------------------------------------------
// C2: per-frame normal equations (fp64) + Cholesky / box QP + update
// ------------------------------------------------------------------------------------------------------------
namespace c2
{
constexpr int THREADS = 256;
}


__device__ __forceinline__ int tri_idx(int i, int j) // i >= j
{
  return i * (i + 1) / 2 + j;
}

// Right-looking Cholesky of the leading `npiv` pivots of the packed lower-triangular (N x N) matrix in shared
// memory.  Returns false (in *ok) on a non-positive pivot (Eigen::LLT NumericalIssue, node.cpp:934-937).
// With npiv < N the trailing block is left holding the Schur complement.
// `col` (N doubles of shared memory) receives the scaled pivot column, so the trailing update reads it with unit
// stride; rows of the trailing triangle go to warps round-robin, lanes along the row.  (The first version mapped a
// flat element index to (row, column) with a double-precision sqrt per element and pivot: 65 % of the kernel's
// instructions, ncu source page of r01e.)
__device__ void block_cholesky(double * L, double * col, int N, int npiv, int tid, int nthreads, int * ok)
{
  const int warp = tid >> 5, lane = tid & 31, nwarps = nthreads >> 5;
  // two block barriers per pivot: the next pivot's diagonal is also published in col[N] by the thread that updates it,
  // so every thread can read it without racing the scaling step that overwrites L[j][j]
  __syncthreads();
  if(tid == 0) col[N] = L[0];
  __syncthreads();
  for(int j = 0; j < npiv; j++)
  {
    const double d = col[N];
    if(!(d > 0.0))
    {
      if(tid == 0) *ok = 0;
      __syncthreads();
      return;
    }
    const double inv = 1.0 / sqrt(d);
    for(int i = j + tid; i < N; i += nthreads)
    {
      const double v = i == j ? sqrt(d) : L[tri_idx(i, j)] * inv;
      L[tri_idx(i, j)] = v;
      col[i] = v;
    }
    __syncthreads();
    // trailing update: L[i][k] -= L[i][j] L[k][j] for j < k <= i
    for(int i = j + 1 + warp; i < N; i += nwarps)
    {
      const double lij = col[i];
      double * row = L + tri_idx(i, 0);
      for(int k = j + 1 + lane; k <= i; k += 32)
      {
        const double v = row[k] - lij * col[k];
        row[k] = v;
        if(i == j + 1 && k == j + 1) col[N] = v; // the next pivot
      }
    }
    __syncthreads();
  }
}

// x <- L^-T L^-1 x for the leading n x n block, executed by warp 0 (other threads idle); result in x.  Four unknowns per
// step: every lane solves the 4x4 diagonal block redundantly in registers, then the lanes update the other rows.
__device__ void warp_chol_solve(const double * L, int n, double * x, int tid)
{
  if(tid >= 32) return;
  for(int k0 = 0; k0 < n; k0 += 4)
  {
    const int bs = min(4, n - k0);
    double xs[4] = {0.0, 0.0, 0.0, 0.0};
    for(int c = 0; c < bs; c++)
    {
      double v = x[k0 + c];
      for(int k = 0; k < c; k++) v -= L[tri_idx(k0 + c, k0 + k)] * xs[k];
      xs[c] = v / L[tri_idx(k0 + c, k0 + c)];
    }
    __syncwarp();
    if(tid == 0)
      for(int c = 0; c < bs; c++) x[k0 + c] = xs[c];
    for(int i = k0 + bs + tid; i < n; i += 32)
    {
      const double * row = L + tri_idx(i, k0);
      double v = x[i];
      for(int c = 0; c < bs; c++) v -= row[c] * xs[c];
      x[i] = v;
    }
    __syncwarp();
  }
  const int last = (n - 1) / 4 * 4;
  for(int k0 = last; k0 >= 0; k0 -= 4)
  {
    const int bs = min(4, n - k0);
    double xs[4] = {0.0, 0.0, 0.0, 0.0};
    for(int c = bs - 1; c >= 0; c--)
    {
      double v = x[k0 + c];
      for(int k = c + 1; k < bs; k++) v -= L[tri_idx(k0 + k, k0 + c)] * xs[k];
      xs[c] = v / L[tri_idx(k0 + c, k0 + c)];
    }
    __syncwarp();
    if(tid == 0)
      for(int c = 0; c < bs; c++) x[k0 + c] = xs[c];
    for(int i = tid; i < k0; i += 32)
    {
      double v = x[i];
      for(int c = 0; c < bs; c++) v -= L[tri_idx(k0 + c, i)] * xs[c];
      x[i] = v;
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(c2::THREADS, 4) ik_solve_kernel(const IkSolveParams p)
{
  const int THREADS = blockDim.x; // chosen by the host from the number of 4x4 tiles of A (<= c2::THREADS)
  extern __shared__ __align__(16) double smd[];
  const int tid = threadIdx.x;
  const int f = blockIdx.x;
  const int D = p.D;
  const int NT = D * (D + 1) / 2;
  double * L = smd;            // packed lower, NT
  double * bvec = L + NT;      // D
  double * x = bvec + D;       // D
  double * g = x + D;          // D
  double * dstep = g + D;      // D
  double * colbuf = dstep + D; // D + 2: pivot column of block_cholesky (+ the next pivot at [N], N <= D + 1)
  int * state = reinterpret_cast<int *>(colbuf + D + 2); // D: 0 free, -1 at lower, +1 at upper, 2 pinned
  __shared__ double s_esq;
  __shared__ int s_ok, s_flag, s_iter, s_atmin;
  __shared__ double s_red[c2::THREADS / 32];

  const int rows = 4 * p.n;
  const float * J = p.J + static_cast<size_t>(f) * rows * p.ld;
  const float * e = p.e + static_cast<size_t>(f) * rows;
  const int valid = p.frame_info[2 * f], bad = p.frame_info[2 * f + 1];
  const bool too_few = p.skip_if_too_few && valid < p.n / 2; // node.cpp:785
  if(tid == 0) s_ok = 1;

  // ---- ||e||^2 ----
  {
    double acc = 0.0;
    for(int r = tid; r < rows; r += THREADS) acc += static_cast<double>(e[r]) * static_cast<double>(e[r]);
    for(int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if((tid & 31) == 0) s_red[tid >> 5] = acc;
    __syncthreads();
    if(tid == 0)
    {
      double s = 0.0;
      for(int w = 0; w < THREADS / 32; w++) s += s_red[w];
      s_esq = s;
    }
  }
  // ---- A = J'J in 4x4 tiles of the lower triangle and b = J'e; fp32 entries widened exactly, fp64 accumulation.
  //      The rows of one task (rows_per_task x ld floats) are staged in shared memory, double buffered: the global loads
  //      of task m+1 are coalesced, issued by the first threads and in flight while task m is consumed (every thread
  //      fetching its own two float4 per row from L1 / L2 was 25 % long-scoreboard stalls, and b = J'e another serial
  //      pass over the rows). ----
  {
    const int nb = (D + 3) / 4;
    const int ntiles = nb * (nb + 1) / 2;
    const int rpt = p.rows_per_task;
    const int ld4 = p.ld >> 2;                                   // float4 per row (ld is a multiple of 4)
    float4 * s_rows = reinterpret_cast<float4 *>(reinterpret_cast<char *>(smd) + p.rows_off); // [2][4][ld4]
    const int per_task = rpt * ld4;
    auto fetch = [&](int m, int i) -> float4 { // float4 i of the staged rows of task m
      const int q = i / ld4, c4 = i - q * ld4;
      return __ldg(reinterpret_cast<const float4 *>(J + static_cast<size_t>(4 * m + q) * p.ld) + c4);
    };
    double accb = 0.0;
    for(int tl0 = 0; tl0 < ntiles; tl0 += THREADS)
    {
      const int tl = tl0 + tid;
      const bool valid = tl < ntiles;
      int bi = 0, bj = 0;
      if(valid)
      {
        bi = static_cast<int>((sqrt(8.0 * tl + 1.0) - 1.0) * 0.5);
        while((bi + 1) * (bi + 2) / 2 <= tl) bi++;
        while(bi * (bi + 1) / 2 > tl) bi--;
        bj = tl - bi * (bi + 1) / 2;
      }
      double acc[4][4];
#pragma unroll
      for(int a = 0; a < 4; a++)
#pragma unroll
        for(int b = 0; b < 4; b++) acc[a][b] = 0.0;
      __syncthreads(); // the previous pass is done with both buffers
      for(int i = tid; i < per_task; i += THREADS) s_rows[(i / ld4) * ld4 + (i % ld4)] = fetch(0, i);
      __syncthreads();
      for(int m = 0; m < p.n; m++)
      {
        const int buf = m & 1;
        // next task: global -> registers now, registers -> shared memory after this task's arithmetic
        float4 nxt[2];
        const bool more = m + 1 < p.n;
#pragma unroll
        for(int u = 0; u < 2; u++)
          if(more && tid + u * THREADS < per_task) nxt[u] = fetch(m + 1, tid + u * THREADS);
        const float4 * rows = s_rows + buf * 4 * ld4;
        if(valid)
        {
#pragma unroll
          for(int q = 0; q < 4; q++)
            if(q < rpt)
            {
              const float4 ja = rows[q * ld4 + bi], jb = rows[q * ld4 + bj];
              const double a4[4] = {ja.x, ja.y, ja.z, ja.w};
              const double b4[4] = {jb.x, jb.y, jb.z, jb.w};
#pragma unroll
              for(int a = 0; a < 4; a++)
#pragma unroll
                for(int b = 0; b < 4; b++) acc[a][b] = fma(a4[a], b4[b], acc[a][b]);
            }
        }
        if(tl0 == 0 && tid < D)
        {
          const float * rf = reinterpret_cast<const float *>(rows);
#pragma unroll
          for(int q = 0; q < 4; q++)
            if(q < rpt) accb = fma(static_cast<double>(rf[q * p.ld + tid]), static_cast<double>(e[4 * m + q]), accb);
        }
#pragma unroll
        for(int u = 0; u < 2; u++)
          if(more && tid + u * THREADS < per_task)
          {
            const int i = tid + u * THREADS;
            s_rows[(buf ^ 1) * 4 * ld4 + (i / ld4) * ld4 + (i % ld4)] = nxt[u];
          }
        __syncthreads();
      }
      if(valid)
      {
#pragma unroll
        for(int a = 0; a < 4; a++)
#pragma unroll
          for(int b = 0; b < 4; b++)
          {
            const int i = 4 * bi + a, j = 4 * bj + b;
            if(i < D && j <= i) L[tri_idx(i, j)] = acc[a][b];
          }
      }
    }
    // D may exceed the block size only for the largest problems: the remaining entries of b the plain way
    if(tid < D) bvec[tid] = accb;
    for(int i = tid + THREADS; i < D; i += THREADS)
    {
      double acc = 0.0;
      for(int r = 0; r < rows; r++)
        if((r & 3) < rpt) acc = fma(static_cast<double>(J[static_cast<size_t>(r) * p.ld + i]), static_cast<double>(e[r]), acc);
      bvec[i] = acc;
    }
  }
  __syncthreads();
  // ---- damping (node.cpp:887-893) and the VPoser prior (:895-904) ----
  const int npiv = p.schur ? D - p.beta_cols : D;
  for(int i = tid; i < D; i += THREADS)
  {
    double reg = i < p.theta_dim ? p.reg_theta : (i < p.theta_dim + p.phi_cols ? p.reg_phi : p.reg_beta);
    double add = reg + s_esq;
    if(p.schur && i >= npiv) add = 0.0; // the beta block is damped once, globally, in the apply step
    if(p.vposer && i < p.theta_dim)
    {
      const double w = i < 6 ? 0.0 : (i >= p.theta_dim - 6 ? p.hand_reg : p.latent_reg);
      add += w;
      bvec[i] += w * static_cast<double>(p.theta_state[static_cast<size_t>(f) * p.theta_dim + i]);
    }
    L[tri_idx(i, i)] += add;
  }
  __syncthreads();
  // ---- optional outputs in the reference layout ----
  if(p.a_out || p.b_out)
  {
    auto ref_col = [&](int c) {
      if(c < p.theta_dim) return c;
      if(c < p.theta_dim + p.phi_cols) return c;              // phi columns sit right after theta in both layouts
      return p.theta_dim + 2 * p.n + (c - p.theta_dim - p.phi_cols);
    };
    if(p.a_out)
    {
      double * A = p.a_out + static_cast<size_t>(f) * p.dim_ref * p.dim_ref;
      for(int i = tid; i < p.dim_ref * p.dim_ref; i += THREADS) A[i] = 0.0;
      __syncthreads();
      for(int i = tid; i < NT; i += THREADS)
      {
        int r = static_cast<int>((sqrt(8.0 * i + 1.0) - 1.0) * 0.5);
        while((r + 1) * (r + 2) / 2 <= i) r++;
        while(r * (r + 1) / 2 > i) r--;
        const int c = i - r * (r + 1) / 2;
        A[ref_col(r) * p.dim_ref + ref_col(c)] = L[i];
        A[ref_col(c) * p.dim_ref + ref_col(r)] = L[i];
      }
      if(!p.phi_cols)
        for(int i = tid; i < 2 * p.n; i += THREADS)
          A[(p.theta_dim + i) * p.dim_ref + p.theta_dim + i] = static_cast<double>(p.reg_phi) + s_esq;
    }
    if(p.b_out)
    {
      double * bo = p.b_out + static_cast<size_t>(f) * p.dim_ref;
      for(int i = tid; i < p.dim_ref; i += THREADS) bo[i] = 0.0;
      __syncthreads();
      for(int i = tid; i < D; i += THREADS) bo[ref_col(i)] = bvec[i];
    }
    __syncthreads();
  }

  if(p.schur)
  {
    // ---- shared-beta stage: augmented partial Cholesky.  Append b as an extra row so that the elimination
    //      also produces y0 = L^-1 b_f and r = b_beta - Y' y0 (see DESIGN.md) ----
    // layout: rows 0..D-1 of the packed matrix, then row D = [b' | 0]
    double * aug = L + NT; // row D of the packed (D+1)x(D+1) matrix aliases bvec/x (D + 1 entries fit: bvec,x are 2D)
    // bvec already sits at L + NT .. L + NT + D - 1 = packed row D, columns 0..D-1; set the corner
    if(tid == 0) aug[D] = 0.0;
    __syncthreads();
    block_cholesky(L, colbuf, D + 1, npiv, tid, THREADS, &s_ok);
    double * out = p.schur_out + static_cast<size_t>(f) * 111;
    const bool good = s_ok && !bad && !too_few;
    for(int i = tid; i < 111; i += THREADS)
    {
      double v = 0.0;
      if(good)
      {
        if(i < 100)
        {
          const int r = i / 10, c = i % 10;
          v = r >= c ? L[tri_idx(npiv + r, npiv + c)] : L[tri_idx(npiv + c, npiv + r)];
        }
        else if(i < 110)
          v = L[tri_idx(D, npiv + (i - 100))];
        else
          v = s_esq;
      }
      out[i] = v;
    }
    // keep the factor rows for the apply step: L_ff (packed npiv), Y' rows (10 x npiv), y0 (npiv)
    const int P = npiv * (npiv + 1) / 2 + (p.beta_cols + 1) * npiv;
    double * fw = p.factor_ws + static_cast<size_t>(f) * P;
    const int nff = npiv * (npiv + 1) / 2;
    for(int i = tid; i < nff; i += THREADS) fw[i] = L[i];
    for(int i = tid; i < (p.beta_cols + 1) * npiv; i += THREADS)
    {
      const int r = i / npiv, c = i % npiv;
      fw[nff + i] = L[tri_idx(npiv + r, c)];
    }
    if(tid == 0) p.status[f] = too_few ? 1 : ((bad || !s_ok) ? 2 : 0);
    return;
  }

  // ---- bounds: which variables can be bound-active (node.cpp:911-929) ----
  const bool phi_bounded = p.phi_cols > 0;
  const bool beta_bounded = p.beta_cols > 0;
  const bool qp = p.enable_qp && (phi_bounded || beta_bounded) && p.a_ws != nullptr;
  int status = 0;
  if(!qp)
  {
    // plain LLT: delta = -A^-1 b
    block_cholesky(L, colbuf, D, D, tid, THREADS, &s_ok);
    for(int i = tid; i < D; i += THREADS) x[i] = -bvec[i];
    __syncthreads();
    if(s_ok) warp_chol_solve(L, D, x, tid);
    __syncthreads();
    if(!s_ok) status = 2;
  }
  else
  {
    // primal active-set on min 1/2 x'Ax + b'x, lo <= x <= hi (same iteration as the oracle's solve_box_qp)
    double * A0 = p.a_ws + static_cast<size_t>(f) * NT;
    for(int i = tid; i < NT; i += THREADS) A0[i] = L[i];
    for(int i = tid; i < D; i += THREADS)
    {
      x[i] = 0.0;
      state[i] = 0;
    }
    if(tid == 0) s_flag = 0, s_iter = 0, s_atmin = 0;
    __syncthreads();
    auto lim = [&](int i) -> double {
      if(i < p.theta_dim) return INFINITY;
      if(i < p.theta_dim + p.phi_cols) return static_cast<double>(p.phi_limit);
      return static_cast<double>(p.beta_limit);
    };
    const int max_iter = 20 * D + 50;
    while(true)
    {
      // g = A0 x + b
      for(int i = tid; i < D; i += THREADS)
      {
        double acc = bvec[i];
        for(int k = 0; k < D; k++) acc = fma(i >= k ? A0[tri_idx(i, k)] : A0[tri_idx(k, i)], x[k], acc);
        g[i] = acc;
      }
      // masked copy: fixed variables become identity rows/columns
      for(int i = tid; i < NT; i += THREADS)
      {
        int r = static_cast<int>((sqrt(8.0 * i + 1.0) - 1.0) * 0.5);
        while((r + 1) * (r + 2) / 2 <= i) r++;
        while(r * (r + 1) / 2 > i) r--;
        const int c = i - r * (r + 1) / 2;
        const bool fixed = state[r] != 0 || state[c] != 0;
        L[i] = fixed ? (r == c ? 1.0 : 0.0) : A0[i];
      }
      __syncthreads();
      block_cholesky(L, colbuf, D, D, tid, THREADS, &s_ok);
      if(!s_ok)
      {
        status = 2;
        break;
      }
      for(int i = tid; i < D; i += THREADS) dstep[i] = state[i] != 0 ? 0.0 : -g[i];
      __syncthreads();
      warp_chol_solve(L, D, dstep, tid);
      __syncthreads();
      if(tid == 0)
      {
        double dmax = 0.0, xmax = 1.0;
        for(int i = 0; i < D; i++)
        {
          dmax = fmax(dmax, fabs(dstep[i]));
          xmax = fmax(xmax, fabs(x[i]));
        }
        int flag = 0;
        // s_atmin: the previous step was a full, unblocked Newton step, so x already minimises the objective on the
        // current face; the re-solved step is rounding noise (not necessarily below the threshold when A is
        // ill-conditioned near convergence) and the multiplier test follows directly
        if(s_atmin || dmax <= 1e-14 * xmax)
        {
          int worst = -1;
          double worst_val = 1e-12;
          for(int i = 0; i < D; i++)
          {
            double viol = state[i] == -1 ? -g[i] : (state[i] == 1 ? g[i] : 0.0);
            if(viol > worst_val) worst_val = viol, worst = i;
          }
          if(worst < 0)
            flag = 1; // optimal
          else
            state[worst] = 0;
          s_atmin = 0;
        }
        else
        {
          double alpha = 1.0;
          int block = -1, side = 0;
          for(int i = 0; i < D; i++)
          {
            if(state[i] != 0) continue;
            const double l = lim(i);
            if(!isfinite(l)) continue;
            if(dstep[i] > 0.0)
            {
              double a = (l - x[i]) / dstep[i];
              if(a < alpha) alpha = a, block = i, side = 1;
            }
            else if(dstep[i] < 0.0)
            {
              double a = (-l - x[i]) / dstep[i];
              if(a < alpha) alpha = a, block = i, side = -1;
            }
          }
          for(int i = 0; i < D; i++)
            if(state[i] == 0) x[i] += alpha * dstep[i];
          s_atmin = block < 0;
          if(block >= 0)
          {
            x[block] = side > 0 ? lim(block) : -lim(block);
            state[block] = lim(block) == 0.0 ? 2 : side;
          }
        }
        s_iter++;
        if(s_iter >= max_iter && !flag) flag = 2;
        s_flag = flag;
      }
      __syncthreads();
      if(s_flag == 1) break;
      if(s_flag == 2)
      {
        status = 3;
        break;
      }
    }
    __syncthreads();
  }
  if(bad) status = 2;
  if(status == 0 && too_few) status = 1;
  // ---- outputs + update (node.cpp:946-968) ----
  if(p.delta_out)
  {
    double * dout = p.delta_out + static_cast<size_t>(f) * p.dim_ref;
    for(int i = tid; i < p.dim_ref; i += THREADS) dout[i] = 0.0;
    __syncthreads();
    for(int i = tid; i < D; i += THREADS)
    {
      int c = i < p.theta_dim + p.phi_cols ? i : p.theta_dim + 2 * p.n + (i - p.theta_dim - p.phi_cols);
      dout[c] = status == 2 ? 0.0 : x[i];
    }
  }
  if(p.update_state && status == 0)
  {
    for(int i = tid; i < p.theta_dim; i += THREADS)
      p.theta_state[static_cast<size_t>(f) * p.theta_dim + i] += static_cast<float>(x[i]);
    if(p.beta_cols && p.beta)
      for(int i = tid; i < p.beta_cols; i += THREADS)
        p.beta[static_cast<size_t>(f) * p.beta_stride + i] += static_cast<float>(x[p.theta_dim + p.phi_cols + i]);
  }
  if(tid == 0) p.status[f] = status;
}

// ------------------------------------------------------------------------------------------------------------
// compact -> reference-layout Jacobian (the "Jacobian getter" path; HBM-bound)
// ------------------------------------------------------------------------------------------------------------
__global__ void expand_jacobian_kernel(long long total, int rows, int dim_ref, int theta_dim, int phi_cols, int two_n,
                                       int ld, const float * __restrict__ J, float * __restrict__ out)
{
  long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if(i >= total) return;
  const int c = static_cast<int>(i % dim_ref);
  const long long fr = i / dim_ref; // frame * rows + row
  int src = -1;
  if(c < theta_dim)
    src = c;
  else if(c < theta_dim + two_n)
    src = phi_cols ? c : -1;
  else
    src = theta_dim + phi_cols + (c - theta_dim - two_n);
  out[i] = src >= 0 ? J[fr * ld + src] : 0.f;
}

// ------------------------------------------------------------------------------------------------------------
// shared-beta stage: deterministic reduction of the per-frame Schur blocks and the apply step
// ------------------------------------------------------------------------------------------------------------
__global__ void schur_reduce_kernel(int B, const double * __restrict__ per_frame, double * __restrict__ reduced)
{
  // one block per scalar (111); fixed-order tree => bitwise reproducible sums
  __shared__ double s[256];
  const int k = blockIdx.x, tid = threadIdx.x;
  double acc = 0.0;
  for(int f = tid; f < B; f += 256) acc += per_frame[static_cast<size_t>(f) * 111 + k];
  s[tid] = acc;
  __syncthreads();
  for(int o = 128; o > 0; o >>= 1)
  {
    if(tid < o) s[tid] += s[tid + o];
    __syncthreads();
  }
  if(tid == 0) reduced[k] = s[0];
}

// single block: 10-dim box QP  min 1/2 x'(S + (reg + E2) I)x + r'x, |x| <= limit  (fp64 active set, thread 0)
__global__ void shared_beta_qp_kernel(const double * __restrict__ reduced, double reg, double limit, int enable_qp,
                                      double * __restrict__ dbeta, int * __restrict__ qp_status)
{
  if(threadIdx.x != 0) return;
  const int N = 10;
  double A[N][N], b[N], x[N], g[N], d[N], Lm[N][N];
  int st[N];
  const double e2 = reduced[110];
  for(int i = 0; i < N; i++)
  {
    for(int j = 0; j < N; j++) A[i][j] = reduced[i * 10 + j];
    A[i][i] += reg + e2;
    b[i] = reduced[100 + i];
    x[i] = 0.0;
    st[i] = 0;
  }
  int status = 3;
  bool atmin = false; // see ik_solve_kernel
  for(int iter = 0; iter < 20 * N + 50; iter++)
  {
    for(int i = 0; i < N; i++)
    {
      double acc = b[i];
      for(int k = 0; k < N; k++) acc += A[i][k] * x[k];
      g[i] = acc;
    }
    for(int i = 0; i < N; i++)
      for(int j = 0; j < N; j++) Lm[i][j] = (st[i] || st[j]) ? (i == j ? 1.0 : 0.0) : A[i][j];
    bool ok = true;
    for(int j = 0; j < N && ok; j++)
    {
      double dj = Lm[j][j];
      for(int k = 0; k < j; k++) dj -= Lm[j][k] * Lm[j][k];
      if(!(dj > 0.0))
      {
        ok = false;
        break;
      }
      dj = sqrt(dj);
      Lm[j][j] = dj;
      for(int i = j + 1; i < N; i++)
      {
        double s = Lm[i][j];
        for(int k = 0; k < j; k++) s -= Lm[i][k] * Lm[j][k];
        Lm[i][j] = s / dj;
      }
    }
    if(!ok)
    {
      status = 2;
      break;
    }
    for(int i = 0; i < N; i++) d[i] = st[i] ? 0.0 : -g[i];
    for(int i = 0; i < N; i++)
    {
      double s = d[i];
      for(int k = 0; k < i; k++) s -= Lm[i][k] * d[k];
      d[i] = s / Lm[i][i];
    }
    for(int i = N - 1; i >= 0; i--)
    {
      double s = d[i];
      for(int k = i + 1; k < N; k++) s -= Lm[k][i] * d[k];
      d[i] = s / Lm[i][i];
    }
    double dmax = 0.0, xmax = 1.0;
    for(int i = 0; i < N; i++) dmax = fmax(dmax, fabs(d[i])), xmax = fmax(xmax, fabs(x[i]));
    if(atmin || dmax <= 1e-14 * xmax)
    {
      atmin = false;
      int worst = -1;
      double wv = 1e-12;
      for(int i = 0; i < N; i++)
      {
        double viol = st[i] == -1 ? -g[i] : (st[i] == 1 ? g[i] : 0.0);
        if(viol > wv) wv = viol, worst = i;
      }
      if(worst < 0)
      {
        status = 0;
        break;
      }
      st[worst] = 0;
      continue;
    }
    double alpha = 1.0;
    int block = -1, side = 0;
    if(enable_qp)
      for(int i = 0; i < N; i++)
      {
        if(st[i]) continue;
        if(d[i] > 0.0)
        {
          double a = (limit - x[i]) / d[i];
          if(a < alpha) alpha = a, block = i, side = 1;
        }
        else if(d[i] < 0.0)
        {
          double a = (-limit - x[i]) / d[i];
          if(a < alpha) alpha = a, block = i, side = -1;
        }
      }
    for(int i = 0; i < N; i++)
      if(!st[i]) x[i] += alpha * d[i];
    atmin = block < 0;
    if(block >= 0) x[block] = side * limit, st[block] = side;
  }
  for(int i = 0; i < N; i++) dbeta[i] = status == 0 ? x[i] : 0.0;
  *qp_status = status;
}

// per frame (one warp): x_f = -L_ff^-T (y0 + Y dbeta); theta += x_f.  Frame 0's warp also updates the shared beta.
__global__ void shared_beta_apply_kernel(int B, int npiv, int nbeta, const double * __restrict__ factor_ws,
                                         const double * __restrict__ dbeta, const int * __restrict__ qp_status,
                                         const int * __restrict__ status, float * __restrict__ theta_state,
                                         float * __restrict__ shared_beta, int update_state)
{
  extern __shared__ double sx[]; // (warps, npiv)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int f = blockIdx.x * (blockDim.x >> 5) + warp;
  if(f >= B) return;
  if(*qp_status != 0) return;
  if(f == 0 && lane < nbeta && update_state) shared_beta[lane] += static_cast<float>(dbeta[lane]);
  if(status[f] != 0) return;
  const int P = npiv * (npiv + 1) / 2 + (nbeta + 1) * npiv;
  const double * fw = factor_ws + static_cast<size_t>(f) * P;
  const double * L = fw;
  const double * Y = fw + npiv * (npiv + 1) / 2; // rows 0..nbeta-1 = Y' (beta x npiv), row nbeta = y0'
  double * x = sx + warp * npiv;
  for(int i = lane; i < npiv; i += 32)
  {
    double acc = Y[nbeta * npiv + i];
    for(int k = 0; k < nbeta; k++) acc += Y[k * npiv + i] * dbeta[k];
    x[i] = -acc;
  }
  __syncwarp();
  for(int k = npiv - 1; k >= 0; k--)
  {
    double xk = x[k] / L[tri_idx(k, k)];
    __syncwarp();
    if(lane == 0) x[k] = xk;
    for(int i = lane; i < k; i += 32) x[i] -= L[tri_idx(k, i)] * xk;
    __syncwarp();
  }
  if(update_state)
    for(int i = lane; i < npiv; i += 32) theta_state[static_cast<size_t>(f) * npiv + i] += static_cast<float>(x[i]);
}

// ------------------------------------------------------------------------------------------------------------
// host: task set
// ------------------------------------------------------------------------------------------------------------
template<typename T>
static int upload_vec(smplpp_tasks * t, const T ** dst, const std::vector<T> & src)
{
  void * ptr = nullptr;
  SB_CUDA(cudaMalloc(&ptr, std::max<size_t>(src.size(), 1) * sizeof(T)));
  t->allocations.push_back(ptr);
  if(!src.empty()) SB_CUDA(cudaMemcpy(ptr, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice));
  *dst = static_cast<const T *>(ptr);
  return SMPLPP_OK;
}

extern "C" int smplpp_tasks_create(const smplpp_model_t * model, int32_t n, const int64_t * face_idx, smplpp_tasks_t ** out)
{
  if(!model || n < 1 || !face_idx || !out) return fail(SMPLPP_ERR_INVALID, "IkTask", "invalid task list!");
  const ModelDev & md = model->d;
  for(int m = 0; m < n; m++)
    if(face_idx[m] < 0 || face_idx[m] >= md.F) return fail(SMPLPP_ERR_INVALID, "IkTask", "face index out of range!");
  auto t = new smplpp_tasks();
  t->h_face_idx.assign(face_idx, face_idx + n);
  const auto & faces = model->h_faces;
  const auto & aoff = model->h_adj_offset;
  const auto & afaces = model->h_adj_faces;

  // local vertex numbering: distinct corners first, then ring-only vertices
  std::map<int32_t, int32_t> local;
  std::vector<int32_t> sub_vert;
  auto get_local = [&](int32_t v) {
    auto it = local.find(v);
    if(it != local.end()) return it->second;
    int32_t id = static_cast<int32_t>(sub_vert.size());
    local[v] = id;
    sub_vert.push_back(v);
    return id;
  };
  std::vector<int32_t> corner(3 * n);
  for(int m = 0; m < n; m++)
    for(int c = 0; c < 3; c++) corner[3 * m + c] = get_local(faces[3 * face_idx[m] + c]);
  const int nCorner = static_cast<int>(sub_vert.size());
  std::vector<int32_t> item_off(3 * n + 1, 0), item_verts;
  for(int m = 0; m < n; m++)
    for(int c = 0; c < 3; c++)
    {
      int32_t v = faces[3 * face_idx[m] + c];
      for(int k = aoff[v]; k < aoff[v + 1]; k++)
      {
        int g = afaces[k];
        for(int s = 0; s < 3; s++) item_verts.push_back(get_local(faces[3 * g + s]));
      }
      item_off[3 * m + c + 1] = static_cast<int32_t>(item_verts.size() / 3);
    }
  const int nU = static_cast<int>(sub_vert.size());
  const int nUpad = (nU + 63) / 64 * 64;
  const int nItems = static_cast<int>(item_verts.size() / 3);
  // pairs: corners 0,1,2 first, then the other ring vertices in order of first appearance
  std::vector<int32_t> pair_off(n + 1, 0), pair_vert, pair_task, pair_ref_off(1, 0), pair_refs;
  int maxPairs = 0;
  for(int m = 0; m < n; m++)
  {
    std::vector<int32_t> verts_m = {corner[3 * m], corner[3 * m + 1], corner[3 * m + 2]};
    for(int it = item_off[3 * m]; it < item_off[3 * m + 3]; it++)
      for(int s = 0; s < 3; s++)
      {
        int32_t u = item_verts[3 * it + s];
        if(std::find(verts_m.begin(), verts_m.end(), u) == verts_m.end()) verts_m.push_back(u);
      }
    for(int32_t u : verts_m)
    {
      pair_vert.push_back(u);
      pair_task.push_back(m);
      for(int it = item_off[3 * m]; it < item_off[3 * m + 3]; it++)
        for(int s = 0; s < 3; s++)
          if(item_verts[3 * it + s] == u) pair_refs.push_back(it * 4 + s);
      pair_ref_off.push_back(static_cast<int32_t>(pair_refs.size()));
    }
    pair_off[m + 1] = static_cast<int32_t>(pair_vert.size());
    maxPairs = std::max<int>(maxPairs, static_cast<int>(verts_m.size()));
  }
  const int nPairs = static_cast<int>(pair_vert.size());

  // compact model rows
  const int kmax = md.kmax;
  std::vector<float> basis(static_cast<size_t>(3) * nUpad * kBlendK, 0.f), lw(static_cast<size_t>(kmax) * nUpad, 0.f),
      ws(nUpad, 1.f);
  std::vector<uint8_t> lj(static_cast<size_t>(kmax) * nUpad, 0);
  std::vector<uint32_t> anc(kJoints, 0);
  for(int j = 0; j < kJoints; j++)
    for(int k = j; k >= 0; k = md.parent[k]) anc[j] |= 1u << k;
  std::vector<uint32_t> vert_mask(nU, 0);
  for(int u = 0; u < nU; u++)
  {
    int32_t v = sub_vert[u];
    std::copy(model->h_basis.begin() + static_cast<size_t>(3) * v * kBlendK,
              model->h_basis.begin() + static_cast<size_t>(3) * (v + 1) * kBlendK,
              basis.begin() + static_cast<size_t>(3) * u * kBlendK);
    int k = 0;
    float sum = 0.f;
    for(int j = 0; j < kJoints; j++)
    {
      float w = model->h_weights[static_cast<size_t>(v) * kJoints + j];
      sum += w;
      if(w != 0.f)
      {
        lj[static_cast<size_t>(k) * nUpad + u] = static_cast<uint8_t>(j);
        lw[static_cast<size_t>(k) * nUpad + u] = w;
        vert_mask[u] |= anc[j];
        k++;
      }
    }
    ws[u] = sum;
  }
  std::vector<uint32_t> mask_all(n, 0), mask_corner(n, 0);
  for(int m = 0; m < n; m++)
  {
    for(int q = pair_off[m]; q < pair_off[m + 1]; q++) mask_all[m] |= vert_mask[pair_vert[q]];
    for(int c = 0; c < 3; c++) mask_corner[m] |= vert_mask[corner[3 * m + c]];
  }

  TasksDev & d = t->d;
  d.n = n, d.nU = nU, d.nCorner = nCorner, d.nUpad = nUpad, d.nItems = nItems, d.nPairs = nPairs;
  d.maxPairs = maxPairs, d.kmax = kmax;
  int rc = upload_vec(t, &d.corner, corner);
  if(rc == SMPLPP_OK) rc = upload_vec(t, &d.item_off, item_off);
  if(rc == SMPLPP_OK) rc = upload_vec(t, &d.item_verts, item_verts);
  if(rc == SMPLPP_OK) rc = upload_vec(t, &d.pair_off, pair_off);
  if(rc == SMPLPP_OK) rc = upload_vec(t, &d.pair_vert, pair_vert);
  if(rc == SMPLPP_OK) rc = upload_vec(t, &d.pair_task, pair_task);
  if(rc == SMPLPP_OK) rc = upload_vec(t, &d.pair_ref_off, pair_ref_off);
  if(rc == SMPLPP_OK) rc = upload_vec(t, &d.pair_refs, pair_refs);
  if(rc == SMPLPP_OK)
  {
    std::vector<int32_t> order(nPairs);
    for(int i = 0; i < nPairs; i++) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) {
      return pair_ref_off[a + 1] - pair_ref_off[a] > pair_ref_off[b + 1] - pair_ref_off[b];
    });
    rc = upload_vec(t, &d.pair_order, order);
  }
  if(rc == SMPLPP_OK) rc = upload_vec(t, &d.task_joint_mask, mask_all);
  if(rc == SMPLPP_OK) rc = upload_vec(t, &d.task_joint_mask_corner, mask_corner);
  if(rc == SMPLPP_OK) rc = upload_vec(t, &d.basis, basis);
  if(rc == SMPLPP_OK)
  {
    std::vector<float4> basis4(static_cast<size_t>(nUpad) * kBlendK);
    for(int u = 0; u < nUpad; u++)
      for(int k = 0; k < kBlendK; k++)
        basis4[static_cast<size_t>(u) * kBlendK + k] =
            make_float4(basis[(static_cast<size_t>(3) * u) * kBlendK + k], basis[(static_cast<size_t>(3) * u + 1) * kBlendK + k],
                        basis[(static_cast<size_t>(3) * u + 2) * kBlendK + k], 0.f);
    rc = upload_vec(t, &d.basis4, basis4);
  }
  if(rc == SMPLPP_OK) rc = upload_vec(t, &d.lbs_joint, lj);
  if(rc == SMPLPP_OK) rc = upload_vec(t, &d.lbs_weight, lw);
  if(rc == SMPLPP_OK) rc = upload_vec(t, &d.lbs_wsum, ws);
  if(rc == SMPLPP_OK)
  {
    std::vector<float> swn(static_cast<size_t>(nU) * kmax);
    std::vector<uint8_t> sjf(static_cast<size_t>(nU) * kmax);
    for(int u = 0; u < nU; u++)
      for(int sl = 0; sl < kmax; sl++)
      {
        swn[static_cast<size_t>(u) * kmax + sl] = lw[static_cast<size_t>(sl) * nUpad + u] / ws[u];
        sjf[static_cast<size_t>(u) * kmax + sl] = lj[static_cast<size_t>(sl) * nUpad + u];
      }
    rc = upload_vec(t, &d.sw_norm, swn);
    if(rc == SMPLPP_OK) rc = upload_vec(t, &d.sj_flat, sjf);
  }
  if(rc != SMPLPP_OK)
  {
    smplpp_tasks_destroy(t);
    return rc;
  }
  // sparse-forward views
  t->sub = md;
  t->sub.V = nU, t->sub.Vpad = nUpad, t->sub.F = 0;
  t->sub.basis = const_cast<float *>(d.basis);
  t->sub.lbs_joint = const_cast<uint8_t *>(d.lbs_joint);
  t->sub.lbs_weight = const_cast<float *>(d.lbs_weight);
  t->sub.lbs_wsum = const_cast<float *>(d.lbs_wsum);
  t->sub.group_nj = nullptr, t->sub.group_joint = nullptr, t->sub.group_w = nullptr; // per-vertex slot path
  // the tensor-core operands and the dense (V,24) weight table of the full model are indexed by FULL-model vertex ids:
  // none of them may be reachable through the compact view (lbs_tc_usable() would otherwise accept an even nU >= 128
  // and skin sub-vertex u with the weights of model vertex u)
  t->sub.weights_dense = nullptr;
  t->sub.basis_split[0] = t->sub.basis_split[1] = nullptr;
  t->sub.basis_f16 = nullptr, t->sub.basis_img16 = nullptr;
  t->sub.tc_ready = t->sub.tc2_ready = t->sub.tc3_ready = false;
  t->sub.tc_tiles = t->sub.tc2_tiles = 0;
  t->sub.faces = nullptr, t->sub.adj_offset = nullptr, t->sub.adj_faces = nullptr;
  t->sub_corner = t->sub;
  t->sub_corner.V = nCorner;
  t->h_sub_vert = sub_vert;
  t->h_corner = corner;
  rc = poseblend_tc_prepare(basis, pair_off, pair_vert, t->pb, t->allocations);
  if(rc != SMPLPP_OK)
  {
    smplpp_tasks_destroy(t);
    return rc;
  }
  // self-contained per-task records of the fused step (ik2.cu)
  {
    std::vector<TaskRec> recs(n);
    int mp = 3, mi = 0, ml = 1;
    for(int m = 0; m < n; m++)
    {
      if(build_task_rec_host(model, face_idx[m], recs[m]) != 0)
      {
        smplpp_tasks_destroy(t);
        return fail(SMPLPP_ERR_INVALID, "IkTask", "the 1-ring of an attachment face exceeds the record limits (48 vertices / 48 faces)");
      }
      mp = std::max<int>(mp, recs[m].np), mi = std::max<int>(mi, recs[m].ni);
      ml = std::max<int>(ml, __builtin_popcount(recs[m].jmask));
    }
    rc = upload_vec(t, &t->recs, recs);
    if(rc == SMPLPP_OK && md.kmax <= 4)
    {
      std::vector<TaskSkin> skins(n);
      for(int m = 0; m < n; m++) build_task_skin_host(model, recs[m], skins[m]);
      rc = upload_vec(t, &t->skins, skins);
    }
    if(rc != SMPLPP_OK)
    {
      smplpp_tasks_destroy(t);
      return rc;
    }
    t->maxPairs = mp, t->maxItems = mi, t->maxLive = ml;
  }
  *out = t;
  return SMPLPP_OK;
}

extern "C" void smplpp_tasks_destroy(smplpp_tasks_t * t)
{
  if(!t) return;
  sb_release_host_solve(t);
  sb_release_marker_pipe(t);
  for(void * ptr : t->allocations) cudaFree(ptr);
  delete t;
}

extern "C" int32_t smplpp_tasks_count(const smplpp_tasks_t * t)
{
  return t ? t->d.n : 0;
}

// Rest shape T + S beta + P c of the task vertices only (SMPL::getRestShape restricted to the rows the IK step reads; the
// product the step runs on tcgen05).  vertex_ids (host, nullable): model vertex of every row.  variant 0: tensor cores where
// the task set has the operand images, 1: the FFMA kernel.
extern "C" int smplpp_tasks_rest_shape(const smplpp_model_t * model, const smplpp_tasks_t * tasks, void * stream, int64_t batch,
                                       const float * beta, int64_t beta_stride, const float * theta, float * rest_out,
                                       int32_t * vertex_ids, int32_t variant)
{
  if(!model || !tasks || batch < 1 || !beta || !theta || !rest_out) return fail(SMPLPP_ERR_INVALID, "IkTask", "invalid arguments!");
  cudaStream_t st = as_stream(stream);
  const int B = static_cast<int>(batch);
  const size_t cpad = align_up(static_cast<size_t>(B), 128);
  float * coef = nullptr;
  float * xf = nullptr;
  SB_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&coef), cpad * kBlendK * sizeof(float), st));
  SB_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&xf), cpad * kJoints * 12 * sizeof(float), st));
  int rc = launch_pose_chain(model->d, st, B, beta, beta_stride, theta, coef, xf, nullptr, nullptr);
  if(rc == SMPLPP_OK)
  {
    if(variant == 0 && tasks->pb.ready && tasks->pb.rest_ready)
      rc = launch_restshape_tc(tasks->pb, st, B, tasks->d.nU, coef, rest_out);
    else
      rc = launch_blend_skin_ffma(tasks->sub, st, B, coef, xf, theta, rest_out, false);
  }
  cudaFreeAsync(coef, st);
  cudaFreeAsync(xf, st);
  if(rc == SMPLPP_OK && vertex_ids)
    for(int u = 0; u < tasks->d.nU; u++) vertex_ids[u] = tasks->h_sub_vert[u];
  return rc;
}

extern "C" int32_t smplpp_tasks_vertex_count(const smplpp_tasks_t * t)
{
  return t ? t->d.nU : 0;
}

extern "C" int smplpp_triangle_vertex_weights(void * stream, int64_t n, const float * pos, const float * tri, float * w)
{
  if(n < 1 || !pos || !tri || !w) return fail(SMPLPP_ERR_INVALID, "GeometryUtils", "invalid triangle tensors!");
  triangle_weights_kernel<<<static_cast<unsigned>((n + 127) / 128), 128, 0, as_stream(stream)>>>(n, pos, tri, w);
  SB_LAUNCHED();
  return SMPLPP_OK;
}

extern "C" void smplpp_ik_options_default(smplpp_ik_options * o)
{
  if(!o) return;
  *o = smplpp_ik_options{};
  o->enable_vposer = 0;
  o->optimize_beta = 0;
  o->enable_qp = 1;
  o->enable_phi = 0;
  o->skip_if_too_few = 1;
  o->update_state = 1;
  o->normal_offset = 0.015f;     // node.cpp:560
  o->normal_task_weight = 0.f;   // node.cpp:558
  o->phi_limit = 0.f;            // node.cpp:699
  o->delta_theta_reg = 1e-3f;    // node.cpp:887
  o->delta_phi_reg = 1e-1f;      // node.cpp:888
  o->delta_beta_reg = 1e-3f;     // node.cpp:889
  o->delta_beta_limit = 0.5f;    // node.cpp:925
  o->vposer_latent_reg = 1e-5f;  // node.cpp:897
  o->vposer_hand_reg = 1e3f;     // node.cpp:900
}

extern "C" int32_t smplpp_ik_theta_dim(const smplpp_ik_options * o)
{
  return (o && o->enable_vposer) ? SMPLPP_LATENT_DIM + 12 : 3 * (kJoints + 1);
}

extern "C" int32_t smplpp_ik_dim(const smplpp_ik_options * o, int32_t n)
{
  return smplpp_ik_theta_dim(o) + 2 * n + ((o && o->optimize_beta) ? kShapeDim : 0);
}

extern "C" int smplpp_task_positions(const smplpp_model_t * model, const smplpp_tasks_t * tasks, void * stream, int64_t batch,
                                     const float * vertices, const float * vertex_weights, float normal_offset,
                                     float * positions, float * normals)
{
  if(!model || !tasks || batch < 1 || !vertices || !vertex_weights || !positions)
    return fail(SMPLPP_ERR_INVALID, "IkTask", "invalid task tensors!");
  // face indices on the device: reuse a small upload per call site is avoided by caching in the handle
  smplpp_tasks * t = const_cast<smplpp_tasks *>(tasks);
  if(!t->face_idx_dev)
  {
    std::vector<long long> tmp(t->h_face_idx.begin(), t->h_face_idx.end());
    if(upload_vec(t, &t->face_idx_dev, tmp) != SMPLPP_OK) return SMPLPP_ERR_CUDA;
  }
  const long long * cached = t->face_idx_dev;
  const ModelDev & d = model->d;
  long long total = batch * tasks->d.n;
  task_positions_kernel<<<static_cast<unsigned>((total + 63) / 64), 64, 0, as_stream(stream)>>>(
      d.faces, d.adj_offset, d.adj_faces, d.V, static_cast<int>(batch), tasks->d.n, cached, nullptr, vertices, vertex_weights,
      normal_offset, nullptr, positions, normals);
  SB_LAUNCHED();
  return SMPLPP_OK;
}

extern "C" int smplpp_task_tangents(const smplpp_model_t * model, const smplpp_tasks_t * tasks, void * stream, int64_t batch,
                                    const float * vertices, const int32_t * face_idx, float * tangents)
{
  if(!model || !tasks || batch < 1 || !vertices || !tangents) return fail(SMPLPP_ERR_INVALID, "IkTask", "invalid task tensors!");
  smplpp_tasks * t = const_cast<smplpp_tasks *>(tasks);
  const long long * shared = nullptr;
  if(!face_idx)
  {
    if(!t->face_idx_dev)
    {
      std::vector<long long> tmp(t->h_face_idx.begin(), t->h_face_idx.end());
      if(upload_vec(t, &t->face_idx_dev, tmp) != SMPLPP_OK) return SMPLPP_ERR_CUDA;
    }
    shared = t->face_idx_dev;
  }
  const ModelDev & d = model->d;
  const long long total = batch * tasks->d.n;
  task_tangents_kernel<<<static_cast<unsigned>((total + 63) / 64), 64, 0, as_stream(stream)>>>(
      d.faces, d.V, static_cast<int>(batch), tasks->d.n, shared, face_idx, vertices, tangents);
  SB_LAUNCHED();
  return SMPLPP_OK;
}

// ------------------------------------------------------------------------------------------------------------
// host: IK step orchestration
// ------------------------------------------------------------------------------------------------------------
namespace
{
struct IkLayout
{
  int n, theta_dim, phi_cols, beta_cols, D, ld, ldfull, dim_ref, rows_per_task, use_ring, nUse;
  bool vposer, qp_ws;
  size_t off_theta, off_coef, off_xf, off_verts, off_rest, off_e, off_j, off_jfull, off_vaa, off_vjac, off_vaux, off_info,
      off_aws, off_schur, off_factor, off_misc, off_ca, off_dr, total;
  bool pb_tc; // pose-blend columns by ik_poseblend_tc_kernel
  int chunk;
};

IkLayout make_layout(const smplpp_tasks_t * tasks, const smplpp_ik_options * o, int64_t batch, bool schur)
{
  IkLayout L{};
  L.n = tasks->d.n;
  L.vposer = o->enable_vposer != 0;
  L.theta_dim = L.vposer ? 44 : 75;
  L.phi_cols = (!schur && o->enable_phi && o->phi_limit > 0.f) ? 2 * L.n : 0;
  L.beta_cols = (schur || o->optimize_beta) ? kShapeDim : 0;
  L.D = L.theta_dim + L.phi_cols + L.beta_cols;
  L.ld = (L.D + 3) / 4 * 4;
  L.ldfull = (75 + L.phi_cols + L.beta_cols + 3) / 4 * 4;
  L.dim_ref = L.theta_dim + 2 * L.n + (o->optimize_beta ? kShapeDim : 0);
  L.rows_per_task = o->normal_task_weight > 0.f ? 4 : 3;
  L.use_ring = (o->normal_offset > 0.f || o->normal_task_weight > 0.f) ? 1 : 0;
  L.nUse = L.use_ring ? tasks->d.nU : tasks->d.nCorner;
  L.qp_ws = !schur && o->enable_qp && (L.phi_cols > 0 || L.beta_cols > 0);
  L.chunk = static_cast<int>(std::min<int64_t>(batch, 16384));
  const size_t C = static_cast<size_t>(L.chunk);
  const size_t cpad = align_up(C, 128);
  size_t off = 256;
  auto take = [&](size_t bytes) {
    size_t o2 = off;
    off += align_up(bytes);
    return o2;
  };
  L.off_theta = take(C * 75 * sizeof(float));
  L.off_coef = take(cpad * kBlendK * sizeof(float));
  L.off_xf = take(cpad * kJoints * 12 * sizeof(float));
  L.off_verts = take(C * L.nUse * 3 * sizeof(float));
  L.off_rest = take(C * L.nUse * 3 * sizeof(float));
  L.off_e = take(C * 4 * L.n * sizeof(float));
  L.off_j = take(C * 4 * L.n * L.ld * sizeof(float));
  L.off_jfull = L.vposer ? take(C * 4 * L.n * L.ldfull * sizeof(float)) : L.off_j;
  L.off_vjac = L.vposer ? take(C * 63 * 32 * sizeof(float)) : 0;
  L.off_vaux = L.vposer ? take(C * vposer_tc_aux_floats() * sizeof(float)) : 0; // d1 | d2 | daa of the tensor-core Jacobian
  L.off_info = take(C * 2 * sizeof(int));
  {
    const Ik2Dims dm = ik2_dims(L.n, L.vposer, L.phi_cols > 0, L.beta_cols > 0);
    const size_t per_frame = std::max<size_t>(static_cast<size_t>(L.D) * (L.D + 1) / 2, ik2_qp_ws_doubles(dm));
    L.off_aws = L.qp_ws ? take(C * per_frame * sizeof(double)) : 0;
  }
  L.off_schur = schur ? take(static_cast<size_t>(batch) * 111 * sizeof(double)) : 0;
  if(schur)
  {
    const int npiv = L.D - L.beta_cols;
    const size_t P = static_cast<size_t>(npiv) * (npiv + 1) / 2 + static_cast<size_t>(L.beta_cols + 1) * npiv;
    L.off_factor = take(static_cast<size_t>(batch) * P * sizeof(double));
  }
  L.off_misc = take(64 * sizeof(double));
  L.pb_tc = tasks->pb.ready && g_poseblend_variant != 1 && L.phi_cols == 0;
  L.off_ca = tasks->pb.ready ? take(C * tasks->pb.slots * 128 * sizeof(float)) : 0;
  L.off_dr = tasks->pb.ready ? take(C * 644 * sizeof(float)) : 0;
  L.total = off;
  return L;
}

size_t jac_smem_bytes(const TasksDev & t, const IkLayout & L)
{
  size_t fl = 76 + 12 + 216 + 648 + 72 + 288 + 72 + 648;
  if(L.beta_cols) fl += 3 * 720;
  fl += 2 * 3 * static_cast<size_t>(L.nUse);
  if(L.use_ring) fl += 4 * static_cast<size_t>(t.nItems) + 12 * static_cast<size_t>(t.n);
  fl += c1::TS * static_cast<size_t>(t.n);
  fl += 12 * static_cast<size_t>(t.nPairs);
  fl += 4 * static_cast<size_t>(L.nUse) * t.kmax; // normalised weights + wn * x
  return fl * sizeof(float) + static_cast<size_t>(L.nUse) * t.kmax + 2 + static_cast<size_t>(t.n) * kJoints * sizeof(uint16_t)
         + 64;
}

// one thread per 4x4 tile of the lower triangle of A, rounded up to whole warps: 192 for D = 75 (190 tiles)
int solve_block_threads(int D)
{
  const int nb = (D + 3) / 4;
  const int tiles = nb * (nb + 1) / 2;
  const int th = (tiles + 31) / 32 * 32;
  return (th < 160 || th > c2::THREADS) ? c2::THREADS : th; // small problems keep 8 warps for the Cholesky / QP phases
}

// byte offset of the J row staging area of ik_solve_kernel (16-byte aligned, behind everything else)
size_t solve_rows_off(const IkLayout & L, bool schur)
{
  const size_t D = L.D;
  size_t dbl = D * (D + 1) / 2 + 5 * D + 4 + (schur ? D + 2 : 0);
  return (dbl * sizeof(double) + D * sizeof(int) + 64 + 15) / 16 * 16;
}

size_t solve_smem_bytes(const IkLayout & L, bool schur)
{
  const size_t D = L.D;
  return solve_rows_off(L, schur) + 2 * 4 * static_cast<size_t>(L.ld) * sizeof(float) + 16;
}

// shared front end of smplpp_ik_step and smplpp_ik_shared_beta_reduce for one chunk of frames
int run_chunk(const smplpp_model_t * model, const smplpp_vposer_t * vposer, const smplpp_tasks_t * tasks,
              const smplpp_ik_options * o, const IkLayout & L, cudaStream_t st, int B, float * theta_state,
              const float * beta, long long beta_stride, float * vertex_weights, const float * target_pos,
              const float * target_normal, const float * pos_task_weight, char * ws)
{
  const ModelDev & md = model->d;
  float * theta = reinterpret_cast<float *>(ws + L.off_theta);
  float * coef = reinterpret_cast<float *>(ws + L.off_coef);
  float * xf = reinterpret_cast<float *>(ws + L.off_xf);
  float * verts = reinterpret_cast<float *>(ws + L.off_verts);
  float * rest = reinterpret_cast<float *>(ws + L.off_rest);
  float * vjac = L.vposer ? reinterpret_cast<float *>(ws + L.off_vjac) : nullptr;
  const float * theta_in = theta_state;
  if(L.vposer)
  {
    theta_assemble_kernel<<<(B * 12 + 127) / 128, 128, 0, st>>>(B, theta_state, theta);
    SB_LAUNCHED();
    int rc = launch_vposer_decode(vposer, st, B, theta_state + 6, 44, theta + 6, 75, vjac,
                                  reinterpret_cast<float *>(ws + L.off_vaux));
    if(rc != SMPLPP_OK) return rc;
    theta_in = theta;
  }
  int rc = launch_pose_chain(md, st, B, beta, beta_stride, theta_in, coef, xf, nullptr, nullptr);
  if(rc != SMPLPP_OK) return rc;
  const ModelDev & sub = L.use_ring ? tasks->sub : tasks->sub_corner;
  // rest shape of the task vertices: tcgen05 (blocked frame layout) where the task set has the operand images
  const bool rest_tc = L.pb_tc && tasks->pb.rest_ready && g_poseblend_variant == 0;
  if(rest_tc)
    rc = launch_restshape_tc(tasks->pb, st, B, L.nUse, coef, rest);
  else
    rc = launch_blend_skin_ffma(sub, st, B, coef, xf, theta_in, rest, false);
  if(rc != SMPLPP_OK) return rc;
  // skinning WITHOUT the root translation is what the chain derivatives need (x_uj), the translation is added
  // back analytically: vertices = skinned + trans.  launch_lbs with root = theta row 0.
  (void)verts; // the task vertices are skinned inside ik_jacobian_kernel

  IkJacParams jp{};
  jp.topo = make_topo(md);
  for(int j = 0; j < kJoints; j++)
  {
    uint32_t m = 0;
    for(int k = j; k >= 0; k = md.parent[k]) m |= 1u << k;
    jp.anc_mask[j] = m;
  }
  jp.t = tasks->d;
  jp.joint_template = md.joint_template;
  jp.joint_shape = md.joint_shape;
  jp.B = B;
  jp.use_ring = L.use_ring;
  jp.beta_cols = L.beta_cols;
  jp.phi_cols = L.phi_cols;
  jp.vposer = L.vposer ? 1 : 0;
  jp.update_weights = 1;
  jp.normal_offset = o->normal_offset;
  jp.normal_task_weight = o->normal_task_weight;
  jp.theta = theta_in;
  jp.beta = beta;
  jp.beta_stride = beta_stride;
  jp.verts = verts;
  jp.rest = rest;
  jp.nUse = L.nUse;
  jp.vertex_weights = vertex_weights;
  jp.target_pos = target_pos;
  jp.target_normal = target_normal;
  jp.pos_task_weight = pos_task_weight;
  jp.vposer_jac = vjac;
  jp.e_out = reinterpret_cast<float *>(ws + L.off_e);
  jp.jfull = reinterpret_cast<float *>(ws + L.off_jfull);
  jp.ldfull = L.vposer ? L.ldfull : L.ld;
  jp.jout = reinterpret_cast<float *>(ws + L.off_j);
  jp.ld = L.ld;
  jp.frame_info = reinterpret_cast<int *>(ws + L.off_info);
  if(L.pb_tc)
  {
    jp.ca_out = reinterpret_cast<float *>(ws + L.off_ca);
    jp.ca_slot_off = tasks->pb.slot_off;
    jp.ca_stride = tasks->pb.slots * 128;
    jp.dr_out = reinterpret_cast<float *>(ws + L.off_dr);
  }
  const size_t smem = jac_smem_bytes(tasks->d, L);
  if(smem > 227 * 1024) return fail(SMPLPP_ERR_INVALID, "IkTask", "task set too large for one CTA per frame");
  auto launch = [&](auto kernel) -> int {
    SB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    kernel<<<B, L.pb_tc ? c1::THREADS_TC : c1::THREADS, smem, st>>>(jp);
    return SMPLPP_OK;
  };
  if(L.rows_per_task == 4)
    rc = L.pb_tc ? launch(ik_jacobian_kernel<4, true>) : launch(ik_jacobian_kernel<4, false>);
  else
    rc = L.pb_tc ? launch(ik_jacobian_kernel<3, true>) : launch(ik_jacobian_kernel<3, false>);
  if(rc != SMPLPP_OK) return rc;
  SB_LAUNCHED();
  if(L.pb_tc)
  {
    rc = launch_poseblend_tc(tasks->pb, tasks->d, st, B, L.rows_per_task, L.use_ring, L.beta_cols ? 75 + L.phi_cols : -1,
                             jp.ca_out, jp.dr_out, jp.jfull, jp.ldfull);
    if(rc != SMPLPP_OK) return rc;
    if(L.vposer)
    {
      const int extra = L.phi_cols + L.beta_cols;
      if(L.rows_per_task == 4)
        ik_vposer_contract_kernel<4><<<B, 256, (64 * 32 + 128 * 64) * sizeof(float), st>>>(L.n, extra, jp.jfull, jp.ldfull, vjac, jp.jout, jp.ld);
      else
        ik_vposer_contract_kernel<3><<<B, 256, (64 * 32 + 128 * 64) * sizeof(float), st>>>(L.n, extra, jp.jfull, jp.ldfull, vjac, jp.jout, jp.ld);
      SB_LAUNCHED();
    }
  }
  return SMPLPP_OK;
}

IkSolveParams make_solve_params(const smplpp_ik_options * o, const IkLayout & L, int B, char * ws, bool schur)
{
  IkSolveParams sp{};
  sp.B = B, sp.n = L.n, sp.rows_per_task = L.rows_per_task;
  sp.theta_dim = L.theta_dim, sp.phi_cols = L.phi_cols, sp.beta_cols = L.beta_cols, sp.D = L.D, sp.ld = L.ld;
  sp.vposer = L.vposer ? 1 : 0;
  sp.enable_qp = o->enable_qp;
  sp.skip_if_too_few = o->skip_if_too_few;
  sp.update_state = o->update_state;
  sp.schur = schur ? 1 : 0;
  sp.reg_theta = o->delta_theta_reg, sp.reg_phi = o->delta_phi_reg, sp.reg_beta = o->delta_beta_reg;
  sp.phi_limit = o->phi_limit, sp.beta_limit = o->delta_beta_limit;
  sp.latent_reg = o->vposer_latent_reg, sp.hand_reg = o->vposer_hand_reg;
  sp.J = reinterpret_cast<const float *>(ws + L.off_j);
  sp.e = reinterpret_cast<const float *>(ws + L.off_e);
  sp.frame_info = reinterpret_cast<const int *>(ws + L.off_info);
  sp.dim_ref = L.dim_ref;
  sp.a_ws = L.qp_ws ? reinterpret_cast<double *>(ws + L.off_aws) : nullptr;
  return sp;
}
} // namespace

extern "C" size_t smplpp_ik_workspace_bytes(const smplpp_tasks_t * tasks, const smplpp_ik_options * opt, int64_t batch)
{
  if(!tasks || !opt || batch < 1) return 0;
  return make_layout(tasks, opt, batch, false).total;
}

namespace
{
// theta (B, 75) fed to the forward pass: the state itself, or [trans | root | decoder(latent) | hands] with the decoder
// Jacobian on the side (node.cpp:761-772)
int assemble_theta(const smplpp_vposer_t * vposer, const IkLayout & L, cudaStream_t st, int B, float * theta_state, char * ws,
                   const float ** theta75, const float ** vjac)
{
  *theta75 = theta_state;
  *vjac = nullptr;
  if(!L.vposer) return SMPLPP_OK;
  float * theta = reinterpret_cast<float *>(ws + L.off_theta);
  float * jac = reinterpret_cast<float *>(ws + L.off_vjac);
  theta_assemble_kernel<<<(B * 12 + 127) / 128, 128, 0, st>>>(B, theta_state, theta);
  SB_LAUNCHED();
  int rc = launch_vposer_decode(vposer, st, B, theta_state + 6, 44, theta + 6, 75, jac, reinterpret_cast<float *>(ws + L.off_vaux));
  if(rc != SMPLPP_OK) return rc;
  *theta75 = theta;
  *vjac = jac;
  return SMPLPP_OK;
}
} // namespace

// face_idx (B, n) int32, nullable: per-frame IkTask::faceIdx_ (re-seated by smplpp_ik_reproject); records_ws: B * n records
static int ik_step_impl(const smplpp_model_t * model, const smplpp_vposer_t * vposer, const smplpp_tasks_t * tasks,
                        const smplpp_ik_options * opt, void * stream, int64_t batch, float * theta_state, float * beta,
                        int64_t beta_stride, float * vertex_weights, const int32_t * face_idx, const float * target_pos,
                        const float * target_normal, const float * pos_task_weight, int32_t * status, float * e_out,
                        float * jac_out, double * a_out, double * b_out, double * delta_out, float * dphi_out,
                        void * workspace, size_t workspace_bytes, bool jacobian_only = false)
{
  if(!model || !tasks || !opt || batch < 1 || !theta_state || !beta || !vertex_weights || !target_pos || (!status && !jacobian_only))
    return fail(SMPLPP_ERR_INVALID, "IkTask", "invalid IK step arguments!");
  if(opt->enable_vposer && !vposer) return fail(SMPLPP_ERR_INVALID, "VPoser", "VPoser decoder is required!");
  if(opt->optimize_beta && beta_stride == 0 && batch > 1)
    return fail(SMPLPP_ERR_INVALID, "IkTask", "per-frame beta optimisation needs per-frame beta (use the shared-beta stage)");
  const IkLayout L = make_layout(tasks, opt, batch, false);
  const size_t rec_chunk = 4096; // frames per launch when every frame carries its own attachment records
  const size_t rec_only = face_idx ? align_up(ik2_rec_bytes(std::min<int64_t>(batch, rec_chunk), L.n)) : 0;
  const size_t rec_bytes = face_idx ? rec_only + align_up(ik2_skin_bytes(std::min<int64_t>(batch, rec_chunk), L.n)) : 0;
  if(!workspace || workspace_bytes < L.total + rec_bytes) return fail(SMPLPP_ERR_INVALID, "IkTask", "IK workspace too small!");
  cudaStream_t st = as_stream(stream);
  char * ws = align_up_ptr<char>(workspace);
  const int n = L.n;
  if((g_ik_variant == 2 && !jacobian_only) || face_idx) // fused kernel: per-frame attachments always, shared ones when selected
  {
    TaskRec * recs = face_idx ? reinterpret_cast<TaskRec *>(ws + L.total) : nullptr;
    TaskSkin * skins = face_idx ? reinterpret_cast<TaskSkin *>(ws + L.total + rec_only) : nullptr;
    const int64_t chunk = face_idx ? static_cast<int64_t>(rec_chunk) : L.chunk;
    for(int64_t s = 0; s < batch; s += chunk)
    {
      const int B = static_cast<int>(std::min<int64_t>(chunk, batch - s));
      Ik2Call c;
      c.model = model, c.vposer = vposer, c.tasks = tasks, c.opt = opt, c.st = st, c.B = B, c.schur = false;
      c.theta_state = theta_state + s * L.theta_dim;
      int rc = assemble_theta(vposer, L, st, B, c.theta_state, ws, &c.theta75, &c.vjac);
      if(rc != SMPLPP_OK) return rc;
      c.beta = beta + s * beta_stride, c.beta_stride = beta_stride;
      c.vertex_weights = vertex_weights + s * n * 3;
      c.target_pos = target_pos + s * n * 3;
      c.target_normal = target_normal ? target_normal + s * n * 3 : nullptr;
      c.pos_task_weight = pos_task_weight ? pos_task_weight + s * n : nullptr;
      if(face_idx)
      {
        rc = launch_task_topo(model->d, st, static_cast<long long>(B) * n, face_idx + s * n, recs, skins);
        if(rc != SMPLPP_OK) return rc;
        c.frame_recs = recs;
        c.frame_skins = skins;
      }
      c.status = status + s;
      c.e_out = e_out ? e_out + s * 4 * n : nullptr;
      c.j_out = jac_out ? jac_out + s * 4 * n * L.dim_ref : nullptr;
      c.a_out = a_out ? a_out + s * L.dim_ref * L.dim_ref : nullptr;
      c.b_out = b_out ? b_out + s * L.dim_ref : nullptr;
      c.delta_out = delta_out ? delta_out + s * L.dim_ref : nullptr;
      c.dphi_out = dphi_out ? dphi_out + s * 2 * n : nullptr;
      c.a_ws = L.qp_ws ? reinterpret_cast<double *>(ws + L.off_aws) : nullptr;
      rc = launch_ik_fused(c);
      if(rc != SMPLPP_OK) return rc;
    }
    return SMPLPP_OK;
  }
  for(int64_t s = 0; s < batch; s += L.chunk)
  {
    const int B = static_cast<int>(std::min<int64_t>(L.chunk, batch - s));
    float * th = theta_state + s * L.theta_dim;
    float * be = beta + s * beta_stride;
    float * vw = vertex_weights + s * n * 3;
    int rc = run_chunk(model, vposer, tasks, opt, L, st, B, th, be, beta_stride, vw, target_pos + s * n * 3,
                       target_normal ? target_normal + s * n * 3 : nullptr,
                       pos_task_weight ? pos_task_weight + s * n : nullptr, ws);
    if(rc != SMPLPP_OK) return rc;
    if(e_out)
      SB_CUDA(cudaMemcpyAsync(e_out + s * 4 * n, ws + L.off_e, static_cast<size_t>(B) * 4 * n * sizeof(float),
                              cudaMemcpyDeviceToDevice, st));
    if(jac_out)
    {
      long long total = static_cast<long long>(B) * 4 * n * L.dim_ref;
      expand_jacobian_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, st>>>(
          total, 4 * n, L.dim_ref, L.theta_dim, L.phi_cols, 2 * n, L.ld, reinterpret_cast<const float *>(ws + L.off_j),
          jac_out + s * 4 * n * L.dim_ref);
      SB_LAUNCHED();
    }
    if(jacobian_only) continue; // smplpp_ik_jacobian: the linearisation alone
    IkSolveParams sp = make_solve_params(opt, L, B, ws, false);
    sp.theta_state = th;
    sp.beta = be;
    sp.beta_stride = beta_stride;
    sp.status = status + s;
    sp.a_out = a_out ? a_out + s * L.dim_ref * L.dim_ref : nullptr;
    sp.b_out = b_out ? b_out + s * L.dim_ref : nullptr;
    sp.delta_out = delta_out ? delta_out + s * L.dim_ref : nullptr;
    const size_t smem = solve_smem_bytes(L, false);
    sp.rows_off = static_cast<int>(solve_rows_off(L, false));
    bool handled = false;
    rc = launch_ik_solve_mma(sp, st, &handled); // J'J on the fp64 tensor cores where the problem shape allows
    if(rc != SMPLPP_OK) return rc;
    if(handled) continue;
    if(smem > 227 * 1024) return fail(SMPLPP_ERR_INVALID, "IkTask", "IK problem too large for one CTA per frame");
    SB_CUDA(cudaFuncSetAttribute(ik_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    ik_solve_kernel<<<B, solve_block_threads(L.D), smem, st>>>(sp);
    SB_LAUNCHED();
  }
  return SMPLPP_OK;
}

extern "C" int smplpp_ik_step(const smplpp_model_t * model, const smplpp_vposer_t * vposer, const smplpp_tasks_t * tasks,
                              const smplpp_ik_options * opt, void * stream, int64_t batch, float * theta_state,
                              float * beta, int64_t beta_stride, float * vertex_weights, const float * target_pos,
                              const float * target_normal, const float * pos_task_weight, int32_t * status,
                              float * e_out, float * jac_out, double * a_out, double * b_out, double * delta_out,
                              void * workspace, size_t workspace_bytes)
{
  return ik_step_impl(model, vposer, tasks, opt, stream, batch, theta_state, beta, beta_stride, vertex_weights, nullptr,
                      target_pos, target_normal, pos_task_weight, status, e_out, jac_out, a_out, b_out, delta_out, nullptr,
                      workspace, workspace_bytes);
}

extern "C" int smplpp_ik_jacobian(const smplpp_model_t * model, const smplpp_vposer_t * vposer, const smplpp_tasks_t * tasks,
                                  const smplpp_ik_options * opt, void * stream, int64_t batch, const float * theta_state,
                                  const float * beta, int64_t beta_stride, float * vertex_weights, const float * target_pos,
                                  const float * target_normal, const float * pos_task_weight, float * e_out, float * jac_out,
                                  void * workspace, size_t workspace_bytes)
{
  if(!e_out && !jac_out) return fail(SMPLPP_ERR_INVALID, "IkTask", "invalid IK Jacobian arguments!");
  // the state is only read on this path (no solve, no update)
  return ik_step_impl(model, vposer, tasks, opt, stream, batch, const_cast<float *>(theta_state), const_cast<float *>(beta),
                      beta_stride, vertex_weights, nullptr, target_pos, target_normal, pos_task_weight, nullptr, e_out, jac_out,
                      nullptr, nullptr, nullptr, nullptr, workspace, workspace_bytes, true);
}

extern "C" size_t smplpp_ik_faces_workspace_bytes(const smplpp_tasks_t * tasks, const smplpp_ik_options * opt, int64_t batch)
{
  if(!tasks || !opt || batch < 1) return 0;
  return make_layout(tasks, opt, batch, false).total + align_up(ik2_rec_bytes(std::min<int64_t>(batch, 4096), tasks->d.n))
         + align_up(ik2_skin_bytes(std::min<int64_t>(batch, 4096), tasks->d.n)) + 256;
}

extern "C" int smplpp_ik_step_faces(const smplpp_model_t * model, const smplpp_vposer_t * vposer, const smplpp_tasks_t * tasks,
                                    const smplpp_ik_options * opt, void * stream, int64_t batch, float * theta_state,
                                    float * beta, int64_t beta_stride, float * vertex_weights, const int32_t * face_idx,
                                    const float * target_pos, const float * target_normal, const float * pos_task_weight,
                                    int32_t * status, float * e_out, float * jac_out, double * a_out, double * b_out,
                                    double * delta_out, float * dphi_out, void * workspace, size_t workspace_bytes)
{
  if(!face_idx) return fail(SMPLPP_ERR_INVALID, "IkTask", "invalid IK step arguments! (face indices)");
  return ik_step_impl(model, vposer, tasks, opt, stream, batch, theta_state, beta, beta_stride, vertex_weights, face_idx,
                      target_pos, target_normal, pos_task_weight, status, e_out, jac_out, a_out, b_out, delta_out, dphi_out,
                      workspace, workspace_bytes);
}

// ------------------------------------------------------------------------------------------------------------
// the tail of the reference's iteration (node.cpp:949-1001), batched: p = calcActualPos() + tangents * dphi on the mesh
// of the given (PRE-update) state -> closest face and point of that mesh -> faceIdx_ and vertexWeights_ re-seated
// ------------------------------------------------------------------------------------------------------------
namespace
{
struct ReprojLayout
{
  int64_t chunk;
  size_t off_theta, off_vaa, off_verts, off_points, off_fwd, total, fwd_bytes;
};
ReprojLayout reproj_layout(const smplpp_model_t * model, const smplpp_tasks_t * tasks, int64_t batch)
{
  ReprojLayout R{};
  R.chunk = std::min<int64_t>(batch, 2048);
  size_t off = 256;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off += align_up(bytes);
    return o;
  };
  const size_t C = static_cast<size_t>(R.chunk);
  R.off_theta = take(C * 75 * sizeof(float));
  R.off_vaa = take(C * vposer_tc_aux_floats() * sizeof(float));
  R.off_verts = take(C * model->d.V * 3 * sizeof(float));
  R.off_points = take(C * tasks->d.n * 3 * sizeof(float));
  R.fwd_bytes = smplpp_forward_workspace_bytes(model, R.chunk);
  R.off_fwd = take(R.fwd_bytes);
  R.total = off;
  return R;
}
} // namespace

extern "C" size_t smplpp_ik_reproject_workspace_bytes(const smplpp_model_t * model, const smplpp_tasks_t * tasks, int64_t batch)
{
  if(!model || !tasks || batch < 1) return 0;
  return reproj_layout(model, tasks, batch).total + 256;
}

extern "C" int smplpp_ik_reproject(const smplpp_model_t * model, const smplpp_vposer_t * vposer, const smplpp_tasks_t * tasks,
                                   const smplpp_ik_options * opt, void * stream, int64_t batch, const float * theta_state,
                                   const float * beta, int64_t beta_stride, float * vertex_weights, int32_t * face_idx,
                                   const float * dphi, float * sq_dist, void * workspace, size_t workspace_bytes)
{
  if(!model || !tasks || !opt || batch < 1 || !theta_state || !beta || !vertex_weights || !face_idx)
    return fail(SMPLPP_ERR_INVALID, "IkTask", "Failed to project points onto the mesh!");
  if(opt->enable_vposer && !vposer) return fail(SMPLPP_ERR_INVALID, "VPoser", "VPoser decoder is required!");
  const ReprojLayout R = reproj_layout(model, tasks, batch);
  if(!workspace || workspace_bytes < R.total) return fail(SMPLPP_ERR_INVALID, "IkTask", "IK workspace too small!");
  cudaStream_t st = as_stream(stream);
  char * ws = align_up_ptr<char>(workspace);
  const ModelDev & d = model->d;
  const int n = tasks->d.n;
  const int theta_dim = opt->enable_vposer ? 44 : 75;
  float * theta = reinterpret_cast<float *>(ws + R.off_theta);
  float * verts = reinterpret_cast<float *>(ws + R.off_verts);
  float * points = reinterpret_cast<float *>(ws + R.off_points);
  for(int64_t s = 0; s < batch; s += R.chunk)
  {
    const int B = static_cast<int>(std::min<int64_t>(R.chunk, batch - s));
    const float * th = theta_state + s * theta_dim;
    const float * theta75 = th;
    if(opt->enable_vposer)
    {
      theta_assemble_kernel<<<(B * 12 + 127) / 128, 128, 0, st>>>(B, th, theta);
      SB_LAUNCHED();
      int rc = launch_vposer_decode(vposer, st, B, th + 6, 44, theta + 6, 75, nullptr, reinterpret_cast<float *>(ws + R.off_vaa));
      if(rc != SMPLPP_OK) return rc;
      theta75 = theta;
    }
    int rc = smplpp_forward(model, st, B, beta + s * beta_stride, beta_stride, theta75, verts, nullptr, nullptr, nullptr,
                            ws + R.off_fwd, R.fwd_bytes);
    if(rc != SMPLPP_OK) return rc;
    const long long total = static_cast<long long>(B) * n;
    task_positions_kernel<<<static_cast<unsigned>((total + 63) / 64), 64, 0, st>>>(
        d.faces, d.adj_offset, d.adj_faces, d.V, B, n, nullptr, face_idx + s * n, verts, vertex_weights + s * n * 3,
        opt->normal_offset, dphi ? dphi + s * n * 2 : nullptr, points, nullptr);
    SB_LAUNCHED();
    rc = smplpp_closest_points(model, st, B, n, verts, points, face_idx + s * n, nullptr, sq_dist ? sq_dist + s * n : nullptr,
                               vertex_weights + s * n * 3);
    if(rc != SMPLPP_OK) return rc;
  }
  return SMPLPP_OK;
}

extern "C" size_t smplpp_ik_shared_beta_workspace_bytes(const smplpp_tasks_t * tasks, const smplpp_ik_options * opt,
                                                        int64_t batch)
{
  if(!tasks || !opt || batch < 1) return 0;
  return make_layout(tasks, opt, batch, true).total;
}

extern "C" int smplpp_ik_shared_beta_reduce(const smplpp_model_t * model, const smplpp_vposer_t * vposer,
                                            const smplpp_tasks_t * tasks, const smplpp_ik_options * opt, void * stream,
                                            int64_t batch, const float * theta_state, const float * shared_beta,
                                            float * vertex_weights, const float * target_pos,
                                            const float * pos_task_weight, int32_t * status, double * reduced,
                                            void * workspace, size_t workspace_bytes)
{
  if(!model || !tasks || !opt || batch < 1 || !theta_state || !shared_beta || !vertex_weights || !target_pos || !status
     || !reduced)
    return fail(SMPLPP_ERR_INVALID, "IkTask", "invalid shared-beta arguments!");
  if(opt->enable_vposer && !vposer) return fail(SMPLPP_ERR_INVALID, "VPoser", "VPoser decoder is required!");
  const IkLayout L = make_layout(tasks, opt, batch, true);
  if(!workspace || workspace_bytes < L.total) return fail(SMPLPP_ERR_INVALID, "IkTask", "IK workspace too small!");
  cudaStream_t st = as_stream(stream);
  char * ws = align_up_ptr<char>(workspace);
  const int n = L.n;
  const int npiv = L.D - L.beta_cols;
  const size_t P = static_cast<size_t>(npiv) * (npiv + 1) / 2 + static_cast<size_t>(L.beta_cols + 1) * npiv;
  for(int64_t s = 0; s < batch && g_ik_variant == 2; s += L.chunk)
  {
    const int B = static_cast<int>(std::min<int64_t>(L.chunk, batch - s));
    Ik2Call c;
    c.model = model, c.vposer = vposer, c.tasks = tasks, c.opt = opt, c.st = st, c.B = B, c.schur = true;
    c.theta_state = const_cast<float *>(theta_state) + s * L.theta_dim;
    int rc = assemble_theta(vposer, L, st, B, c.theta_state, ws, &c.theta75, &c.vjac);
    if(rc != SMPLPP_OK) return rc;
    c.beta = const_cast<float *>(shared_beta), c.beta_stride = 0;
    c.vertex_weights = vertex_weights + s * n * 3;
    c.target_pos = target_pos + s * n * 3;
    c.pos_task_weight = pos_task_weight ? pos_task_weight + s * n : nullptr;
    c.status = status + s;
    c.schur_out = reinterpret_cast<double *>(ws + L.off_schur) + s * 111;
    c.factor_ws = reinterpret_cast<double *>(ws + L.off_factor) + s * P;
    rc = launch_ik_fused(c);
    if(rc != SMPLPP_OK) return rc;
  }
  for(int64_t s = 0; s < batch && g_ik_variant != 2; s += L.chunk)
  {
    const int B = static_cast<int>(std::min<int64_t>(L.chunk, batch - s));
    int rc = run_chunk(model, vposer, tasks, opt, L, st, B, const_cast<float *>(theta_state) + s * L.theta_dim,
                       shared_beta, 0, vertex_weights + s * n * 3, target_pos + s * n * 3, nullptr,
                       pos_task_weight ? pos_task_weight + s * n : nullptr, ws);
    if(rc != SMPLPP_OK) return rc;
    IkSolveParams sp = make_solve_params(opt, L, B, ws, true);
    sp.theta_state = const_cast<float *>(theta_state) + s * L.theta_dim;
    sp.beta = nullptr;
    sp.status = status + s;
    sp.schur_out = reinterpret_cast<double *>(ws + L.off_schur) + s * 111;
    sp.factor_ws = reinterpret_cast<double *>(ws + L.off_factor) + s * P;
    const size_t smem = solve_smem_bytes(L, true);
    sp.rows_off = static_cast<int>(solve_rows_off(L, true));
    bool handled = false;
    rc = launch_ik_solve_mma(sp, st, &handled);
    if(rc != SMPLPP_OK) return rc;
    if(handled) continue;
    SB_CUDA(cudaFuncSetAttribute(ik_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    ik_solve_kernel<<<B, solve_block_threads(L.D), smem, st>>>(sp);
    SB_LAUNCHED();
  }
  schur_reduce_kernel<<<111, 256, 0, st>>>(static_cast<int>(batch), reinterpret_cast<const double *>(ws + L.off_schur), reduced);
  SB_LAUNCHED();
  return SMPLPP_OK;
}

extern "C" int smplpp_ik_shared_beta_apply(const smplpp_tasks_t * tasks, const smplpp_ik_options * opt, void * stream,
                                           int64_t batch, float * theta_state, float * shared_beta, const int32_t * status,
                                           const double * reduced, void * workspace, size_t workspace_bytes)
{
  if(!tasks || !opt || batch < 1 || !theta_state || !shared_beta || !status || !reduced)
    return fail(SMPLPP_ERR_INVALID, "IkTask", "invalid shared-beta arguments!");
  const IkLayout L = make_layout(tasks, opt, batch, true);
  if(!workspace || workspace_bytes < L.total) return fail(SMPLPP_ERR_INVALID, "IkTask", "IK workspace too small!");
  cudaStream_t st = as_stream(stream);
  char * ws = align_up_ptr<char>(workspace);
  double * misc = reinterpret_cast<double *>(ws + L.off_misc);
  double * dbeta = misc;
  int * qp_status = reinterpret_cast<int *>(misc + 16);
  shared_beta_qp_kernel<<<1, 32, 0, st>>>(reduced, static_cast<double>(opt->delta_beta_reg),
                                         static_cast<double>(opt->delta_beta_limit), opt->enable_qp, dbeta, qp_status);
  SB_LAUNCHED();
  const int npiv = L.D - L.beta_cols;
  const int warps = 4;
  const int grid = static_cast<int>((batch + warps - 1) / warps);
  shared_beta_apply_kernel<<<grid, warps * 32, warps * npiv * sizeof(double), st>>>(
      static_cast<int>(batch), npiv, L.beta_cols, reinterpret_cast<const double *>(ws + L.off_factor), dbeta, qp_status,
      status, theta_state, shared_beta, opt->update_state);
  SB_LAUNCHED();
  return SMPLPP_OK;
}
