// Model handle: packs the tensors of SMPL::init (reference src/SMPL.cpp:560-643) into the device layouts
// used by the kernels.  All precomputation happens once here, on the host, in double precision.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <memory>

#include "forward.cuh"

namespace sb
{
thread_local std::string g_last_error;
std::atomic<uint64_t> g_launch_count{0};

int fail(int code, const char * module, const std::string & msg)
{
  // reference message convention: "<module> Error: <text>" (src/toolbox/Exception.cpp:77-91)
  g_last_error = std::string(module) + " Error: " + msg;
  return code;
}
} // namespace sb

using namespace sb;

extern "C" const char * smplpp_last_error(void)
{
  return g_last_error.c_str();
}

extern "C" uint64_t smplpp_launch_count(void)
{
  return g_launch_count.load();
}

extern "C" int smplpp_device_count(void)
{
  int n = 0;
  if(cudaGetDeviceCount(&n) != cudaSuccess)
  {
    cudaGetLastError();
    return 0;
  }
  return n;
}

template<typename T>
static int upload(T ** dst, const std::vector<T> & src)
{
  SB_CUDA(cudaMalloc(reinterpret_cast<void **>(dst), std::max<size_t>(src.size(), 1) * sizeof(T)));
  if(!src.empty()) SB_CUDA(cudaMemcpy(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice));
  return SMPLPP_OK;
}

extern "C" int smplpp_model_create(const smplpp_model_desc * desc, smplpp_model_t ** out)
{
  if(!desc || !out) return fail(SMPLPP_ERR_INVALID, "SMPL", "Cannot initialize a SMPL model!");
  if(desc->vertex_num < 1 || !desc->shape_blend_shapes || !desc->pose_blend_shapes || !desc->vertices_template
     || !desc->joint_regressor || !desc->kinematic_tree || !desc->weights)
    return fail(SMPLPP_ERR_INVALID, "SMPL", "Cannot initialize a SMPL model!");
  if(desc->face_num > 0 && !desc->face_indices) return fail(SMPLPP_ERR_INVALID, "SMPL", "Failed to get face indices!");
  if(smplpp_device_count() < 1) return fail(SMPLPP_ERR_CUDA, "CUDA", "no CUDA device (there is no CPU fallback)");

  const int V = static_cast<int>(desc->vertex_num);
  const int F = static_cast<int>(desc->face_num);
  const int Vpad = (V + 63) / 64 * 64;
  // owned by a guard until the very end: every early return below releases the device buffers allocated so far
  // (smplpp_model_destroy is nullptr-safe member by member)
  std::unique_ptr<smplpp_model, void (*)(smplpp_model *)> guard(new smplpp_model(), smplpp_model_destroy);
  smplpp_model * m = guard.get();
  ModelDev & d = m->d;
  d.V = V;
  d.Vpad = Vpad;
  d.F = F;

  // kinematic tree (WorldTransformation.cpp:508-536 reads row 0 as parents; root stored as 4294967295)
  for(int j = 0; j < kJoints; j++)
  {
    int64_t p = desc->kinematic_tree[j];
    d.parent[j] = (j > 0 && p >= 0 && p < kJoints) ? static_cast<int>(p) : -1;
    if(j > 0 && (d.parent[j] < 0 || d.parent[j] >= j))
      return fail(SMPLPP_ERR_INVALID, "WorldTransformation", "Cannot transform bones locally!"); // the guard frees m
  }
  d.max_depth = 0;
  for(int j = 0; j < kJoints; j++)
  {
    d.depth[j] = j == 0 ? 0 : d.depth[d.parent[j]] + 1;
    d.max_depth = std::max(d.max_depth, d.depth[j]);
  }

  // fused blend basis, K-major
  m->h_basis.assign(static_cast<size_t>(3) * V * kBlendK, 0.f);
  for(int v = 0; v < V; v++)
    for(int k = 0; k < 3; k++)
    {
      float * row = &m->h_basis[(static_cast<size_t>(3) * v + k) * kBlendK];
      std::memcpy(row, desc->pose_blend_shapes + (static_cast<size_t>(3) * v + k) * kPoseDim, sizeof(float) * kPoseDim);
      std::memcpy(row + kPoseDim, desc->shape_blend_shapes + (static_cast<size_t>(3) * v + k) * kShapeDim,
                  sizeof(float) * kShapeDim);
      row[kPoseDim + kShapeDim] = desc->vertices_template[3 * v + k];
    }
  {
    std::vector<float> padded(static_cast<size_t>(3) * Vpad * kBlendK, 0.f);
    std::memcpy(padded.data(), m->h_basis.data(), m->h_basis.size() * sizeof(float));
    if(upload(&d.basis, padded) != SMPLPP_OK) return SMPLPP_ERR_CUDA;
  }

  // joints: Jreg (T + S beta) = J_T + J_S beta   (JointRegression.cpp:588-590), accumulated in double
  m->h_joint_template.assign(kJoints * 3, 0.f);
  m->h_joint_shape.assign(kJoints * 3 * kShapeDim, 0.f);
  for(int j = 0; j < kJoints; j++)
  {
    double jt[3] = {0, 0, 0};
    double js[3][kShapeDim] = {};
    const float * reg = desc->joint_regressor + static_cast<size_t>(j) * V;
    for(int v = 0; v < V; v++)
    {
      double w = reg[v];
      if(w == 0.0) continue;
      for(int k = 0; k < 3; k++)
      {
        jt[k] += w * desc->vertices_template[3 * v + k];
        const float * s = desc->shape_blend_shapes + (static_cast<size_t>(3) * v + k) * kShapeDim;
        for(int i = 0; i < kShapeDim; i++) js[k][i] += w * s[i];
      }
    }
    for(int k = 0; k < 3; k++)
    {
      m->h_joint_template[3 * j + k] = static_cast<float>(jt[k]);
      for(int i = 0; i < kShapeDim; i++) m->h_joint_shape[(3 * j + k) * kShapeDim + i] = static_cast<float>(js[k][i]);
    }
  }
  if(upload(&d.joint_template, m->h_joint_template) != SMPLPP_OK) return SMPLPP_ERR_CUDA;
  if(upload(&d.joint_shape, m->h_joint_shape) != SMPLPP_OK) return SMPLPP_ERR_CUDA;

  // skinning weights -> ELL (dense (V,24) input stays legal: kmax grows up to 24)
  m->h_weights.assign(desc->weights, desc->weights + static_cast<size_t>(V) * kJoints);
  int kmax = 1;
  for(int v = 0; v < V; v++)
  {
    int nnz = 0;
    for(int j = 0; j < kJoints; j++) nnz += desc->weights[static_cast<size_t>(v) * kJoints + j] != 0.f;
    kmax = std::max(kmax, nnz);
  }
  d.kmax = kmax;
  {
    std::vector<uint8_t> lj(static_cast<size_t>(kmax) * Vpad, 0);
    std::vector<float> lw(static_cast<size_t>(kmax) * Vpad, 0.f), ws(Vpad, 1.f);
    for(int v = 0; v < V; v++)
    {
      int k = 0;
      float sum = 0.f;
      for(int j = 0; j < kJoints; j++)
      {
        float w = desc->weights[static_cast<size_t>(v) * kJoints + j];
        sum += w; // float accumulation in joint order, like the reference's tensordot over 24 terms
        if(w != 0.f)
        {
          lj[static_cast<size_t>(k) * Vpad + v] = static_cast<uint8_t>(j);
          lw[static_cast<size_t>(k) * Vpad + v] = w;
          k++;
        }
      }
      ws[v] = sum;
    }
    if(upload(&d.lbs_joint, lj) != SMPLPP_OK) return SMPLPP_ERR_CUDA;
    if(upload(&d.lbs_weight, lw) != SMPLPP_OK) return SMPLPP_ERR_CUDA;
    if(upload(&d.lbs_wsum, ws) != SMPLPP_OK) return SMPLPP_ERR_CUDA;
  }
  {
    const int groups = Vpad / kGroupVerts;
    std::vector<int8_t> nj(groups, 0);
    std::vector<uint8_t> gj(static_cast<size_t>(groups) * kGroupJoints, 0);
    std::vector<float> gw(static_cast<size_t>(groups) * kGroupJoints * kGroupVerts, 0.f);
    for(int g = 0; g < groups; g++)
    {
      std::vector<int> list;
      for(int v = g * kGroupVerts; v < std::min(V, (g + 1) * kGroupVerts); v++)
        for(int j = 0; j < kJoints; j++)
          if(desc->weights[static_cast<size_t>(v) * kJoints + j] != 0.f && std::find(list.begin(), list.end(), j) == list.end())
            list.push_back(j);
      std::sort(list.begin(), list.end());
      if(static_cast<int>(list.size()) > kGroupJoints)
      {
        nj[g] = -1;
        continue;
      }
      nj[g] = static_cast<int8_t>(list.size());
      for(size_t k = 0; k < list.size(); k++)
      {
        gj[static_cast<size_t>(g) * kGroupJoints + k] = static_cast<uint8_t>(list[k]);
        for(int u = 0; u < kGroupVerts; u++)
        {
          const int v = g * kGroupVerts + u;
          if(v < V)
            gw[(static_cast<size_t>(g) * kGroupJoints + k) * kGroupVerts + u] =
                desc->weights[static_cast<size_t>(v) * kJoints + list[k]];
        }
      }
    }
    if(upload(&d.group_nj, nj) != SMPLPP_OK) return SMPLPP_ERR_CUDA;
    if(upload(&d.group_joint, gj) != SMPLPP_OK) return SMPLPP_ERR_CUDA;
    if(upload(&d.group_w, gw) != SMPLPP_OK) return SMPLPP_ERR_CUDA;
  }
  if(upload(&d.weights_dense, m->h_weights) != SMPLPP_OK) return SMPLPP_ERR_CUDA;
  {
    // per vertex: the joints whose rotation moves it = ancestor closure of its influencing joints (IK Jacobian sparsity)
    uint32_t anc[kJoints];
    for(int j = 0; j < kJoints; j++)
    {
      anc[j] = 0;
      for(int k = j; k >= 0; k = d.parent[k]) anc[j] |= 1u << k;
    }
    m->h_vert_jmask.assign(V, 0u);
    for(int v = 0; v < V; v++)
      for(int j = 0; j < kJoints; j++)
        if(m->h_weights[static_cast<size_t>(v) * kJoints + j] != 0.f) m->h_vert_jmask[v] |= anc[j];
    if(upload(&d.vert_jmask, m->h_vert_jmask) != SMPLPP_OK) return SMPLPP_ERR_CUDA;
  }

  // topology: 0-based faces + vertex -> adjacent faces (SMPL.cpp:619-640; uniform weights 1/deg)
  m->h_faces.resize(static_cast<size_t>(F) * 3);
  for(size_t i = 0; i < m->h_faces.size(); i++)
  {
    int32_t id = desc->face_indices[i] - 1;
    if(id < 0 || id >= V) return fail(SMPLPP_ERR_INVALID, "SMPL", "Failed to get face indices!"); // the guard frees m
    m->h_faces[i] = id;
  }
  m->h_adj_offset.assign(V + 1, 0);
  {
    std::vector<std::vector<int32_t>> adj(V);
    for(int f = 0; f < F; f++)
      for(int i = 0; i < 3; i++)
      {
        auto & lst = adj[m->h_faces[3 * f + i]];
        if(std::find(lst.begin(), lst.end(), f) == lst.end()) lst.push_back(f);
      }
    for(int v = 0; v < V; v++) m->h_adj_offset[v + 1] = m->h_adj_offset[v] + static_cast<int32_t>(adj[v].size());
    m->h_adj_faces.reserve(m->h_adj_offset[V]);
    for(int v = 0; v < V; v++) m->h_adj_faces.insert(m->h_adj_faces.end(), adj[v].begin(), adj[v].end());
  }
  if(upload(&d.faces, m->h_faces) != SMPLPP_OK) return SMPLPP_ERR_CUDA;
  if(upload(&d.adj_offset, m->h_adj_offset) != SMPLPP_OK) return SMPLPP_ERR_CUDA;
  if(upload(&d.adj_faces, m->h_adj_faces) != SMPLPP_OK) return SMPLPP_ERR_CUDA;

  {
    float mx = 0.f; // largest pose / shape basis entry (the template column stays out of the tensor-core product)
    for(size_t r = 0; r < static_cast<size_t>(3) * V; r++)
      for(int k = 0; k < kPoseDim + kShapeDim; k++) mx = std::max(mx, std::fabs(m->h_basis[r * kBlendK + k]));
    if(tc3_prepare_model(d, mx, m->h_weights.data()) != SMPLPP_OK) return SMPLPP_ERR_CUDA;
  }
  *out = guard.release();
  return SMPLPP_OK;
}

extern "C" void smplpp_model_destroy(smplpp_model_t * m)
{
  if(!m) return;
  ModelDev & d = m->d;
  cudaFree(d.basis);
  cudaFree(d.lbs_joint);
  cudaFree(d.lbs_weight);
  cudaFree(d.lbs_wsum);
  cudaFree(d.group_nj);
  cudaFree(d.group_joint);
  cudaFree(d.group_w);
  cudaFree(d.joint_template);
  cudaFree(d.joint_shape);
  cudaFree(d.faces);
  cudaFree(d.adj_offset);
  cudaFree(d.adj_faces);
  cudaFree(d.weights_dense);
  cudaFree(d.vert_jmask);
  tc3_release_model(d);
  release_host_pipe(m);
  delete m;
}

extern "C" int64_t smplpp_model_vertex_num(const smplpp_model_t * m)
{
  return m ? m->d.V : 0;
}

extern "C" int smplpp_model_max_influences(const smplpp_model_t * m)
{
  return m ? m->d.kmax : 0;
}
