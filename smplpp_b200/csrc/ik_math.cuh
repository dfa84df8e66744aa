// Device arithmetic of the IK step and of the task positions, shared by the two-kernel path (ik_jacobian_kernel, ik.cu),
// the fused kernel (ik_fused_kernel, ik2.cu), task_tangents_kernel (ik.cu) and the markers-only forward pass
// (task_points_kernel, task_forward.cu): 3-vectors, the normalisation of
// torch::nn::functional::normalize and its derivative, calcTriangleVertexWeights, BlendShape::rodrigues with its derivative,
// the chain prologue, skinning, face and corner normals, tangents and the per-task residual and Jacobian terms.
// Each helper does one thread's work item; loops, thread mappings, barriers and where results are stored stay with the
// kernels.  The reference quirks are reproduced on purpose (DESIGN §5): rodrigues of |theta + 1e-8|, re-weighting from the
// off-plane point, normalize clamped at 1e-12, uniform 1 / deg corner normals.
#pragma once
#include "common.cuh"
#include "forward.cuh"

struct f3
{
  float x, y, z;
};
__device__ __forceinline__ f3 mk3(float x, float y, float z)
{
  f3 r;
  r.x = x, r.y = y, r.z = z;
  return r;
}
__device__ __forceinline__ f3 ld3(const float * p)
{
  return mk3(p[0], p[1], p[2]);
}
__device__ __forceinline__ f3 operator+(f3 a, f3 b)
{
  return mk3(a.x + b.x, a.y + b.y, a.z + b.z);
}
__device__ __forceinline__ f3 operator-(f3 a, f3 b)
{
  return mk3(a.x - b.x, a.y - b.y, a.z - b.z);
}
__device__ __forceinline__ f3 operator*(float s, f3 a)
{
  return mk3(s * a.x, s * a.y, s * a.z);
}
__device__ __forceinline__ float dot3(f3 a, f3 b)
{
  return a.x * b.x + a.y * b.y + a.z * b.z;
}
__device__ __forceinline__ f3 cross3(f3 a, f3 b)
{
  return mk3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__device__ __forceinline__ float norm3(f3 a)
{
  return sqrtf(dot3(a, a));
}
// torch::nn::functional::normalize: v / max(||v||, 1e-12); returns 1 / max(||v||, eps), negative when clamped
__device__ __forceinline__ f3 normalize_inv(f3 a, float & inv)
{
  float n = norm3(a);
  bool clamped = !(n > 1e-12f);
  float i = 1.f / fmaxf(n, 1e-12f);
  inv = clamped ? -i : i;
  return i * a;
}
// derivative of normalize at output direction n (unit) applied to x: (x - n (n.x)) / |v|   (or x / eps when clamped)
__device__ __forceinline__ f3 proj_apply(f3 n, float inv, f3 x)
{
  if(inv < 0.f) return (-inv) * x;
  return inv * (x - dot3(n, x) * n);
}
// calcTriangleVertexWeights (include/smplpp/toolbox/GeometryUtils.h:42-52)
__device__ __forceinline__ void triangle_weights(f3 pos, f3 v0, f3 v1, f3 v2, float * w)
{
  float a0 = norm3(cross3(v1 - pos, v2 - pos));
  float a1 = norm3(cross3(v2 - pos, v0 - pos));
  float a2 = norm3(cross3(v0 - pos, v1 - pos));
  float s = a0 + a1 + a2;
  w[0] = a0 / s, w[1] = a1 / s, w[2] = a2 / s;
}

// BlendShape::rodrigues (src/BlendShape.cpp:803-844) with the derivative of THAT formula (da/dtheta uses theta+eps)
__device__ inline void rodrigues_grad(float x, float y, float z, float * R, float * dR /* [3][9] */)
{
  const float eps = 1e-8f;
  float th[3] = {x, y, z};
  float ax = x + eps, ay = y + eps, az = z + eps;
  float a = sqrtf(ax * ax + ay * ay + az * az);
  float inv_a = 1.f / a;
  float u[3] = {x / a, y / a, z / a};
  float s, c;
  sincosf(a, &s, &c);
  float oc = 1.f - c;
  float uu = u[0] * u[0] + u[1] * u[1] + u[2] * u[2];
  R[0] = 1.f + oc * (-(u[2] * u[2]) - u[1] * u[1]);
  R[1] = s * (-u[2]) + oc * (u[1] * u[0]);
  R[2] = s * u[1] + oc * (u[2] * u[0]);
  R[3] = s * u[2] + oc * (u[0] * u[1]);
  R[4] = 1.f + oc * (-(u[2] * u[2]) - u[0] * u[0]);
  R[5] = s * (-u[0]) + oc * (u[2] * u[1]);
  R[6] = s * (-u[1]) + oc * (u[0] * u[2]);
  R[7] = s * u[0] + oc * (u[1] * u[2]);
  R[8] = 1.f + oc * (-(u[1] * u[1]) - u[0] * u[0]);
  const float K[9] = {0.f, -u[2], u[1], u[2], 0.f, -u[0], -u[1], u[0], 0.f};
  float da[3] = {ax * inv_a, ay * inv_a, az * inv_a};
#pragma unroll
  for(int q = 0; q < 3; q++)
  {
    float du[3];
#pragma unroll
    for(int i = 0; i < 3; i++) du[i] = ((i == q) ? inv_a : 0.f) - u[i] * da[q] * inv_a;
    (void)th;
    const float dK[9] = {0.f, -du[2], du[1], du[2], 0.f, -du[0], -du[1], du[0], 0.f};
    float udu = u[0] * du[0] + u[1] * du[1] + u[2] * du[2];
#pragma unroll
    for(int i = 0; i < 3; i++)
#pragma unroll
      for(int k = 0; k < 3; k++)
      {
        float K2 = u[i] * u[k] - ((i == k) ? uu : 0.f);
        float dK2 = du[i] * u[k] + u[i] * du[k] - ((i == k) ? 2.f * udu : 0.f);
        dR[q * 9 + i * 3 + k] = c * da[q] * K[i * 3 + k] + s * dK[i * 3 + k] + s * da[q] * K2 + oc * dK2;
      }
  }
}

// ------------------------------------------------------------------------------------------------------------
// chain prologue of a frame (shared arrays: R 9 / joint, dR 27, Jt 3, G 12 = [Rg | tg] rows, t' 3, M 9 per (joint, axis),
// JS, dTg, dTp (3 j + r) * 10 + beta index)
// ------------------------------------------------------------------------------------------------------------
// joint j: its rotation and derivative, and the rest joint J_j = joint_template_j + joint_shape_j beta; keep_js also keeps
// the joint-shape rows for the beta columns
__device__ __forceinline__ void chain_joint(int j, const float * s_theta, const float * s_beta, const float * joint_template,
                                            const float * joint_shape, bool keep_js, float * s_R, float * s_dR, float * s_Jt,
                                            float * s_JS)
{
  rodrigues_grad(s_theta[3 + 3 * j], s_theta[4 + 3 * j], s_theta[5 + 3 * j], s_R + 9 * j, s_dR + 27 * j);
#pragma unroll
  for(int k = 0; k < 3; k++)
  {
    float acc = joint_template[3 * j + k];
#pragma unroll
    for(int i = 0; i < sb::kShapeDim; i++)
    {
      const float js = joint_shape[(3 * j + k) * sb::kShapeDim + i];
      acc = fmaf(js, s_beta[i], acc);
      if(keep_js) s_JS[(3 * j + k) * sb::kShapeDim + i] = js;
    }
    s_Jt[3 * j + k] = acc;
  }
}

// global transforms level by level, then t'_j = tg_j - Rg_j J_j.  Called by all 32 lanes of one warp, lane = joint: the
// levels are ordered by __syncwarp
__device__ __forceinline__ void chain_globals_warp(int j, const sb::ChainTopo & topo, const float * s_R, const float * s_Jt,
                                                   float * s_G, float * s_tp)
{
  const int parent = j < sb::kJoints ? topo.parent[j] : -1;
  const int depth = j < sb::kJoints ? topo.depth[j] : -1;
  for(int d = 0; d <= topo.max_depth; d++)
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
        const float tl[3] = {s_Jt[3 * j] - s_Jt[3 * parent], s_Jt[3 * j + 1] - s_Jt[3 * parent + 1],
                             s_Jt[3 * j + 2] - s_Jt[3 * parent + 2]};
        for(int r = 0; r < 3; r++)
        {
          const float p0 = P[4 * r], p1 = P[4 * r + 1], p2 = P[4 * r + 2], p3 = P[4 * r + 3];
          for(int c = 0; c < 3; c++) G[4 * r + c] = p0 * R[c] + p1 * R[3 + c] + p2 * R[6 + c];
          G[4 * r + 3] = p0 * tl[0] + p1 * tl[1] + p2 * tl[2] + p3;
        }
      }
    }
    __syncwarp();
  }
  if(j < sb::kJoints)
  {
    const float * G = s_G + 12 * j;
    for(int r = 0; r < 3; r++)
      s_tp[3 * j + r] = G[4 * r + 3] - (G[4 * r] * s_Jt[3 * j] + G[4 * r + 1] * s_Jt[3 * j + 1] + G[4 * r + 2] * s_Jt[3 * j + 2]);
  }
}

// M_kc = Rg_parent(k) dR_kc Rg_k^T  (d x_j / d theta_kc = M_kc (x_j - tg_k)) for kc = 3 k + c
__device__ __forceinline__ void chain_dM(int kc, const sb::ChainTopo & topo, const float * s_dR, const float * s_G, float * s_M)
{
  const int k = kc / 3;
  const float * A = s_dR + 9 * kc;
  const float * Rk = s_G + 12 * k;
  const int parent = topo.parent[k];
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
      s_M[9 * kc + 3 * a + b] = T[3 * a] * Rk[4 * b] + T[3 * a + 1] * Rk[4 * b + 1] + T[3 * a + 2] * Rk[4 * b + 2];
}

// d tg_j / d beta_i (3 rows): the parent's column plus Rg_parent d(J_j - J_parent) / d beta_i; the parent's level first
__device__ __forceinline__ void chain_dtg_dbeta(int j, int i, int parent, const float * s_G, const float * s_JS, float * s_dTg)
{
  if(parent < 0)
  {
    for(int r = 0; r < 3; r++) s_dTg[(3 * j + r) * sb::kShapeDim + i] = s_JS[(3 * j + r) * sb::kShapeDim + i];
  }
  else
  {
    const float * P = s_G + 12 * parent;
    float dl[3];
    for(int r = 0; r < 3; r++) dl[r] = s_JS[(3 * j + r) * sb::kShapeDim + i] - s_JS[(3 * parent + r) * sb::kShapeDim + i];
    for(int r = 0; r < 3; r++)
      s_dTg[(3 * j + r) * sb::kShapeDim + i] =
          s_dTg[(3 * parent + r) * sb::kShapeDim + i] + P[4 * r] * dl[0] + P[4 * r + 1] * dl[1] + P[4 * r + 2] * dl[2];
  }
}

// d t'_j / d beta_i = d tg_j / d beta_i - Rg_j d J_j / d beta_i (3 rows)
__device__ __forceinline__ void chain_dtp_dbeta(int j, int i, const float * s_G, const float * s_JS, const float * s_dTg,
                                                float * s_dTp)
{
  const float * G = s_G + 12 * j;
  const float js[3] = {s_JS[(3 * j) * sb::kShapeDim + i], s_JS[(3 * j + 1) * sb::kShapeDim + i], s_JS[(3 * j + 2) * sb::kShapeDim + i]};
  for(int r = 0; r < 3; r++)
    s_dTp[(3 * j + r) * sb::kShapeDim + i] =
        s_dTg[(3 * j + r) * sb::kShapeDim + i] - (G[4 * r] * js[0] + G[4 * r + 1] * js[1] + G[4 * r + 2] * js[2]);
}

// one bone's skinning term w_j (Rg_j r + t'_j) with the normalised weight w_j = W[u, j] / sum W (LinearBlendSkinning.cpp:
// 445-553); G: the bone's 3 x 4 rows [Rg_j | .], t'_j at tp[0], tp[tp_stride], tp[2 tp_stride].  The posed vertex is the
// root translation plus the sum of these.
__device__ __forceinline__ f3 skin_term(const float * G, const float * tp, int tp_stride, f3 ru, float wj)
{
  return mk3(wj * (G[0] * ru.x + G[1] * ru.y + G[2] * ru.z + tp[0]),
             wj * (G[4] * ru.x + G[5] * ru.y + G[6] * ru.z + tp[tp_stride]),
             wj * (G[8] * ru.x + G[9] * ru.y + G[10] * ru.z + tp[2 * tp_stride]));
}

// ------------------------------------------------------------------------------------------------------------
// task geometry
// ------------------------------------------------------------------------------------------------------------
// SMPL::calcNormal of one face: normalize((b - a) x (c - a)); inv as in normalize_inv
__device__ __forceinline__ f3 face_normal(f3 a, f3 b, f3 c, float & inv)
{
  return normalize_inv(cross3(b - a, c - a), inv);
}

// SMPL::calcVertexNormal (src/SMPL.cpp:527-535) of one corner: the uniform 1 / deg mean of the normals item_normal(k) of its
// ring faces k in [s0, s1), normalised
template<class ItemNormal>
__device__ __forceinline__ f3 corner_normal(int s0, int s1, ItemNormal item_normal, float & inv)
{
  const float wg = 1.f / static_cast<float>(s1 - s0);
  f3 q = mk3(0.f, 0.f, 0.f);
  for(int k = s0; k < s1; k++) q = q + wg * item_normal(k);
  return normalize_inv(q, inv);
}

// IkTask::calcTangents (src/IkTask.cpp:33-47): t[0] = normalize(v1 - v0), t[1] = normalize(((v1 - v0) x (v2 - v0)) x (v1 - v0))
__device__ __forceinline__ void tangent_frame(f3 v0, f3 v1, f3 v2, f3 * t)
{
  const f3 t1 = v1 - v0;
  const f3 t2 = cross3(cross3(t1, v2 - v0), t1);
  float inv;
  t[0] = normalize_inv(t1, inv), t[1] = normalize_inv(t2, inv);
}

// The per-task helpers below (reweight_task, task_residual, phi_frame / phi_column, store_task_scratch) serve
// ik_jacobian_kernel only.  ik_fused_kernel writes the same arithmetic inline (through them it spills more), so a change
// here has to be made there too.
//
// one task of the IK step, first half: the actual position at the attachment weights w (+ normal offset), which it returns
// (the point that phi moves), the new weights wn from that off-plane point (node.cpp:803-804) and the normal nh at them
// (0 without rings; inv_s as in normalize_inv).  v, nc: corner vertices and corner normals (nc is read only with rings)
__device__ __forceinline__ f3 reweight_task(const f3 * v, const f3 * nc, const float * w, bool ring, float offset, float * wn,
                                            f3 & nh, float & inv_s)
{
  // written out, not accumulated from zero as in task_positions_kernel: the two forms contract to different FMAs
  f3 pos = w[0] * v[0] + w[1] * v[1] + w[2] * v[2];
  inv_s = 0.f;
  if(ring && offset > 0.f) pos = pos + offset * normalize_inv(w[0] * nc[0] + w[1] * nc[1] + w[2] * nc[2], inv_s);
  triangle_weights(pos, v[0], v[1], v[2], wn);
  nh = mk3(0.f, 0.f, 0.f);
  if(ring) nh = normalize_inv(wn[0] * nc[0] + wn[1] * nc[1] + wn[2] * nc[2], inv_s);
  return pos;
}

// second half: the point at the new weights and the residual rows e (node.cpp:807-820); nt = (0, 0, 1) without target normals
__device__ __forceinline__ void task_residual(const f3 * v, const float * wn, f3 nh, float offset, float posw, f3 tgt, f3 nt,
                                              float normal_task_weight, float * e)
{
  f3 pn = wn[0] * v[0] + wn[1] * v[1] + wn[2] * v[2];
  if(offset > 0.f) pn = pn + offset * nh;
  e[0] = posw * (pn.x - tgt.x), e[1] = posw * (pn.y - tgt.y), e[2] = posw * (pn.z - tgt.z);
  e[3] = normal_task_weight > 0.f ? normal_task_weight * (dot3(nh, nt) + 1.f) : 0.f;
}

// phi columns of a task: d w' / d pos (pos = detached actual position + tangents phi, IkTask.cpp:49-57) and the tangents
// (:33-47), shared by the two columns
__device__ __forceinline__ void phi_frame(f3 pos, const float * wn, const f3 * v, f3 * dw, f3 * tang)
{
  const f3 r0 = cross3(v[1] - pos, v[2] - pos), r1 = cross3(v[2] - pos, v[0] - pos), r2 = cross3(v[0] - pos, v[1] - pos);
  const float a0 = norm3(r0), a1 = norm3(r1), a2 = norm3(r2), S = a0 + a1 + a2;
  const f3 g0 = cross3((1.f / a0) * r0, v[2] - v[1]), g1 = cross3((1.f / a1) * r1, v[0] - v[2]),
           g2 = cross3((1.f / a2) * r2, v[1] - v[0]);
  const f3 gs = g0 + g1 + g2;
  dw[0] = (1.f / S) * (g0 - wn[0] * gs), dw[1] = (1.f / S) * (g1 - wn[1] * gs), dw[2] = (1.f / S) * (g2 - wn[2] * gs);
  tangent_frame(v[0], v[1], v[2], tang);
}
// column k: d(residual row r) / d phi_k in col[r], row 3 is the normal-task row
__device__ __forceinline__ void phi_column(const f3 * dw, const f3 * tang, int k, const f3 * v, const f3 * nc, f3 nh, float inv_s,
                                           bool ring, float offset, float posw, f3 nt, float normal_task_weight, float * col)
{
  const float dwk[3] = {dot3(dw[0], tang[k]), dot3(dw[1], tang[k]), dot3(dw[2], tang[k])};
  f3 dp = dwk[0] * v[0] + dwk[1] * v[1] + dwk[2] * v[2];
  f3 dn = mk3(0.f, 0.f, 0.f);
  if(ring) dn = proj_apply(nh, inv_s, dwk[0] * nc[0] + dwk[1] * nc[1] + dwk[2] * nc[2]);
  if(offset > 0.f) dp = dp + offset * dn;
  col[0] = posw * dp.x, col[1] = posw * dp.y, col[2] = posw * dp.z;
  col[3] = normal_task_weight > 0.f ? normal_task_weight * dot3(nt, dn) : 0.f;
}

// per-task scratch read by the dN/dv and C4 phases: [0..2] new weights, [3..5] nh, [6] inv_s, [7] posw, [8..10] target normal
__device__ __forceinline__ void store_task_scratch(float * ts, const float * wn, f3 nh, float inv_s, float posw, f3 nt)
{
  ts[0] = wn[0], ts[1] = wn[1], ts[2] = wn[2];
  ts[3] = nh.x, ts[4] = nh.y, ts[5] = nh.z, ts[6] = inv_s, ts[7] = posw;
  ts[8] = nt.x, ts[9] = nt.y, ts[10] = nt.z;
}

// one reference of d(normal) / d(vertex): the vertex in slot `slot` of ring face v0 v1 v2 moves the face normal by
// P(n_g) [a]x, a = the edge opposite the slot; ax[c] = a x e_c
__device__ __forceinline__ void ref_edge_cross(f3 v0, f3 v1, f3 v2, int slot, f3 * ax)
{
  const f3 e1 = v1 - v0, e2 = v2 - v0;
  const f3 a = slot == 0 ? (e2 - e1) : (slot == 1 ? mk3(-e2.x, -e2.y, -e2.z) : e1);
  ax[0] = mk3(0.f, a.z, -a.y), ax[1] = mk3(-a.z, 0.f, a.x), ax[2] = mk3(a.y, -a.x, 0.f);
}

// C4 = d(residual rows) / d(vertex) (ROWS x 3, padded to 4 x 3) of pair q of the task with scratch ts, from D = d nh / d v
template<int ROWS>
__device__ __forceinline__ void c4_block(const float * ts, int q, const float * D, float offset, float normal_task_weight, float * C)
{
  const float posw = ts[7];
  const float wc = q < 3 ? ts[q] : 0.f; // pairs 0..2 of a task are its corners 0..2
#pragma unroll
  for(int r = 0; r < 3; r++)
#pragma unroll
    for(int c = 0; c < 3; c++) C[3 * r + c] = posw * (((r == c) ? wc : 0.f) + offset * D[3 * r + c]);
  if(ROWS == 4)
  {
#pragma unroll
    for(int c = 0; c < 3; c++) C[9 + c] = normal_task_weight * (ts[8] * D[c] + ts[9] * D[3 + c] + ts[10] * D[6 + c]);
  }
  else
    C[9] = C[10] = C[11] = 0.f;
}
