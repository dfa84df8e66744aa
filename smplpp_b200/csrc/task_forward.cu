// Markers-only forward pass: IkTask::calcActualPos / calcActualNormal (src/IkTask.cpp:59-86) of every task for a batch of
// poses, without the 6890-vertex mesh that SMPL::launch (src/SMPL.cpp:671-737) builds first.
//
//   K1  pose_chain_kernel        coefficients + (B, 24, 3x4) relative transforms            (forward.cu)
//   K2  ik_restshape_tc_kernel   rest shape T + S beta + P c of the task vertices only       (ik_poseblend_tc.cu, tcgen05)
//       or blend_skin_ffma_kernel on the compact rows of the task set                       (forward.cu, FFMA)
//   K3  task_points_kernel       skinning of those rows, 1-ring face normals, corner normals, the interpolated task
//                                point (+ normal offset) and normal                          (this file)
//
// Without the normal offset and without normals only the face corners are needed (nCorner rows, corners come first in
// the task set's layout).  smplpp_task_forward_host runs the same three kernels on chunks of host frames with the
// uploads, the compute and the downloads of consecutive chunks overlapped on three streams.
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "forward.cuh"
#include "host_copy.cuh"
#include "ik_math.cuh"
#include "tasks.cuh"

using namespace sb;

namespace
{
constexpr int kPointsThreads = 128;
// frames per chunk of smplpp_task_forward_host (SMPLPP_TASK_CHUNK overrides): a frame moves ~0.8-1.3 KB over the link,
// so a chunk of this size is ~13-21 MB of copies against ~10 us of per-chunk overhead
constexpr int kDefaultChunk = 16384;
} // namespace

namespace sb
{
struct TaskPointsParams
{
  TasksDev t;
  int nUse;             // rows of `rest`: nU when normals are needed, else nCorner
  int use_ring;         // normals needed (normal_offset > 0 or normals requested)
  const float * rest;   // (B, nUse, 3)
  const float * xf;     // (B, 24, 12) relative transforms [Rg | tg - Rg J]
  const float * theta;  // (B, 25, 3): row 0 = root translation
  const float * vw;     // (n, 3) or (B, n, 3)
  long long vw_stride;  // 0 or 3n
  float offset;
  float * pos;          // (B, n, 3)
  float * nrm;          // (B, n, 3) or null
};
} // namespace sb

namespace
{
size_t points_smem_bytes(const TasksDev & t, int nUse, bool use_ring)
{
  size_t fl = kJoints * kXformFloats + 3 * static_cast<size_t>(nUse);
  if(use_ring) fl += 3 * static_cast<size_t>(t.nItems) + 9 * static_cast<size_t>(t.n);
  return fl * sizeof(float);
}
} // namespace

// One CTA per frame.  Skinning, face and corner normals are skin_term, face_normal and corner_normal of ik_math.cuh
// (homogeneous weights W / sum W, any number of influences).  calcActualPos stays written out here and in
// task_positions_kernel: through one shared helper that takes the corners by callable, the normals of this kernel came
// out different in the last bits.
__global__ void __launch_bounds__(kPointsThreads) task_points_kernel(const TaskPointsParams p)
{
  extern __shared__ __align__(16) float sm[];
  const TasksDev & t = p.t;
  const int tid = threadIdx.x;
  const int f = blockIdx.x;
  float * s_xf = sm;                                            // 24 x 12
  float * s_verts = s_xf + kJoints * kXformFloats;              // nUse x 3 posed rows
  float * s_itemN = s_verts + 3 * p.nUse;                       // nItems x 3 unit normals of the ring faces
  float * s_cornN = s_itemN + (p.use_ring ? 3 * t.nItems : 0);  // 3n x 3 unit corner normals
  __shared__ float s_trans[3];

  const float4 * gx = reinterpret_cast<const float4 *>(p.xf + static_cast<size_t>(f) * kJoints * kXformFloats);
  for(int i = tid; i < kJoints * kXformFloats / 4; i += kPointsThreads) reinterpret_cast<float4 *>(s_xf)[i] = __ldg(gx + i);
  if(tid < 3) s_trans[tid] = p.theta[static_cast<size_t>(f) * (kJoints + 1) * 3 + tid];
  __syncthreads();

  // ---- skinning of the rows (LinearBlendSkinning.cpp:445-553 on the task vertices) ----
  const float * rest = p.rest + static_cast<size_t>(f) * p.nUse * 3;
  for(int u = tid; u < p.nUse; u += kPointsThreads)
  {
    const f3 ru = ld3(rest + 3 * u);
    f3 v = mk3(s_trans[0], s_trans[1], s_trans[2]);
    f3 acc = mk3(0.f, 0.f, 0.f);
    for(int sl = 0; sl < t.kmax; sl++)
    {
      const int i = u * t.kmax + sl;
      const int j = __ldg(t.sj_flat + i);
      const float wj = __ldg(t.sw_norm + i);
      const float * G = s_xf + kXformFloats * j;
      acc = acc + skin_term(G, G + 3, 4, ru, wj);
    }
    v = v + acc;
    s_verts[3 * u] = v.x, s_verts[3 * u + 1] = v.y, s_verts[3 * u + 2] = v.z;
  }
  __syncthreads();
  if(p.use_ring)
  {
    // ---- face normals of the 1-ring items (SMPL::calcNormal) ----
    for(int it = tid; it < t.nItems; it += kPointsThreads)
    {
      float inv;
      const f3 nn = face_normal(ld3(s_verts + 3 * __ldg(t.item_verts + 3 * it)), ld3(s_verts + 3 * __ldg(t.item_verts + 3 * it + 1)),
                                ld3(s_verts + 3 * __ldg(t.item_verts + 3 * it + 2)), inv);
      s_itemN[3 * it] = nn.x, s_itemN[3 * it + 1] = nn.y, s_itemN[3 * it + 2] = nn.z;
    }
    __syncthreads();
    // ---- vertex normals of the corners (SMPL::calcVertexNormal) ----
    for(int ci = tid; ci < 3 * t.n; ci += kPointsThreads)
    {
      float inv;
      const f3 nn = corner_normal(__ldg(t.item_off + ci), __ldg(t.item_off + ci + 1), [&](int it) { return ld3(s_itemN + 3 * it); },
                                  inv);
      s_cornN[3 * ci] = nn.x, s_cornN[3 * ci + 1] = nn.y, s_cornN[3 * ci + 2] = nn.z;
    }
    __syncthreads();
  }
  // ---- calcActualPos / calcActualNormal (IkTask.cpp:59-86) ----
  for(int m = tid; m < t.n; m += kPointsThreads)
  {
    const float * w = p.vw + static_cast<size_t>(f) * p.vw_stride + 3 * m;
    const size_t o = (static_cast<size_t>(f) * t.n + m) * 3;
    f3 pos = mk3(0.f, 0.f, 0.f), s = mk3(0.f, 0.f, 0.f);
    for(int c = 0; c < 3; c++)
    {
      const float wc = __ldg(w + c);
      pos = pos + wc * ld3(s_verts + 3 * __ldg(t.corner + 3 * m + c));
      if(p.use_ring) s = s + wc * ld3(s_cornN + 3 * (3 * m + c));
    }
    if(p.use_ring)
    {
      float inv;
      const f3 nh = normalize_inv(s, inv);
      if(p.offset > 0.f) pos = pos + p.offset * nh;
      if(p.nrm) p.nrm[o] = nh.x, p.nrm[o + 1] = nh.y, p.nrm[o + 2] = nh.z;
    }
    p.pos[o] = pos.x, p.pos[o + 1] = pos.y, p.pos[o + 2] = pos.z;
  }
}

namespace
{
struct TfLayout
{
  size_t off_coef, off_xf, off_rest, total;
};

// workspace: coefficients and transforms of the 128-frame padded batch (the tcgen05 rest-shape kernel reads whole
// 128-frame tiles), rest rows of every frame; 256 bytes of slack for the alignment of the caller's pointer
TfLayout tf_layout(const smplpp_tasks_t * t, int64_t batch)
{
  TfLayout L{};
  const size_t cpad = align_up(static_cast<size_t>(batch), 128);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += align_up(bytes);
    return o;
  };
  L.off_coef = take(cpad * kBlendK * sizeof(float));
  L.off_xf = take(cpad * kJoints * kXformFloats * sizeof(float));
  L.off_rest = take(static_cast<size_t>(batch) * t->d.nU * 3 * sizeof(float));
  L.total = off + 256;
  return L;
}

int task_chunk_frames()
{
  const char * e = getenv("SMPLPP_TASK_CHUNK");
  const int n = e ? atoi(e) : kDefaultChunk;
  return std::max(1, std::min(n, 1 << 20));
}

int check_task_forward_args(const smplpp_model_t * model, const smplpp_tasks_t * tasks, int64_t batch, const float * beta,
                            int64_t beta_stride, const float * theta, const float * vertex_weights,
                            int64_t vertex_weights_stride, const float * positions)
{
  if(!model || !tasks || batch < 1 || !beta || !theta || !vertex_weights || !positions)
    return fail(SMPLPP_ERR_INVALID, "IkTask", "invalid task tensors!");
  if(batch > (1ll << 24)) return fail(SMPLPP_ERR_INVALID, "IkTask", "invalid task tensors! (batch too large)");
  if(beta_stride != 0 && beta_stride < kShapeDim) return fail(SMPLPP_ERR_INVALID, "BlendShape", "Failed to set beta!");
  if(vertex_weights_stride != 0 && vertex_weights_stride != 3ll * tasks->d.n)
    return fail(SMPLPP_ERR_INVALID, "IkTask", "invalid task tensors! (vertex weights stride must be 0 or 3n)");
  return SMPLPP_OK;
}
} // namespace

void sb_release_marker_pipe(smplpp_tasks * t)
{
  smplpp_tasks::MarkerPipe & mp = t->marker;
  for(int i = 0; i < 2; i++)
  {
    if(mp.uploaded[i]) cudaEventDestroy(mp.uploaded[i]);
    if(mp.computed[i]) cudaEventDestroy(mp.computed[i]);
    if(mp.drained[i]) cudaEventDestroy(mp.drained[i]);
    if(mp.dev_in[i]) cudaFree(mp.dev_in[i]);
    if(mp.dev_out[i]) cudaFree(mp.dev_out[i]);
    if(mp.pin_in[i]) cudaFreeHost(mp.pin_in[i]);
    if(mp.pin_out[i]) cudaFreeHost(mp.pin_out[i]);
  }
  if(mp.dev_shared) cudaFree(mp.dev_shared);
  if(mp.ws) cudaFree(mp.ws);
  if(mp.h2d) cudaStreamDestroy(mp.h2d);
  if(mp.compute) cudaStreamDestroy(mp.compute);
  if(mp.d2h) cudaStreamDestroy(mp.d2h);
  mp = smplpp_tasks::MarkerPipe();
}

extern "C" size_t smplpp_task_forward_workspace_bytes(const smplpp_tasks_t * tasks, int64_t batch)
{
  if(!tasks || batch < 1) return 0;
  return tf_layout(tasks, batch).total;
}

extern "C" int smplpp_task_forward(const smplpp_model_t * model, const smplpp_tasks_t * tasks, void * stream, int64_t batch,
                                   const float * beta, int64_t beta_stride, const float * theta, const float * vertex_weights,
                                   int64_t vertex_weights_stride, float normal_offset, float * positions, float * normals,
                                   void * workspace, size_t workspace_bytes)
{
  int rc = check_task_forward_args(model, tasks, batch, beta, beta_stride, theta, vertex_weights, vertex_weights_stride,
                                   positions);
  if(rc != SMPLPP_OK) return rc;
  const TfLayout L = tf_layout(tasks, batch);
  if(!workspace || workspace_bytes < L.total)
    return fail(SMPLPP_ERR_INVALID, "IkTask", "invalid task tensors! (workspace too small)");
  const int B = static_cast<int>(batch);
  cudaStream_t st = as_stream(stream);
  char * ws = align_up_ptr<char>(workspace);
  float * coef = reinterpret_cast<float *>(ws + L.off_coef);
  float * xf = reinterpret_cast<float *>(ws + L.off_xf);
  float * rest = reinterpret_cast<float *>(ws + L.off_rest);
  const bool use_ring = normal_offset > 0.f || normals != nullptr;
  const int nUse = use_ring ? tasks->d.nU : tasks->d.nCorner;

  rc = launch_pose_chain(model->d, st, B, beta, beta_stride, theta, coef, xf, nullptr, nullptr);
  if(rc != SMPLPP_OK) return rc;
  // rest rows: tcgen05 where the task set has the operand images (the rule of the IK step), else the FFMA kernel
  if(tasks->pb.rest_ready && g_poseblend_variant == 0)
    rc = launch_restshape_tc(tasks->pb, st, B, nUse, coef, rest);
  else
    rc = launch_blend_skin_ffma(use_ring ? tasks->sub : tasks->sub_corner, st, B, coef, xf, theta, rest, false);
  if(rc != SMPLPP_OK) return rc;

  // 17 KB for the 41-marker set; larger task sets opt in to more (the call fails if one frame does not fit an SM)
  const size_t smem = points_smem_bytes(tasks->d, nUse, use_ring);
  if(smem > 48 * 1024)
    SB_CUDA(cudaFuncSetAttribute(task_points_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  TaskPointsParams p{};
  p.t = tasks->d;
  p.nUse = nUse;
  p.use_ring = use_ring ? 1 : 0;
  p.rest = rest, p.xf = xf, p.theta = theta;
  p.vw = vertex_weights, p.vw_stride = vertex_weights_stride;
  p.offset = normal_offset;
  p.pos = positions, p.nrm = normals;
  task_points_kernel<<<static_cast<unsigned>(B), kPointsThreads, smem, st>>>(p);
  SB_LAUNCHED();
  return SMPLPP_OK;
}

extern "C" int smplpp_task_forward_host(const smplpp_model_t * model, smplpp_tasks_t * tasks, int64_t batch,
                                        const float * beta_host, int64_t beta_stride, const float * theta_host,
                                        const float * vertex_weights_host, int64_t vertex_weights_stride, float normal_offset,
                                        float * positions_host, float * normals_host)
{
  int rc = check_task_forward_args(model, tasks, batch, beta_host, beta_stride, theta_host, vertex_weights_host,
                                   vertex_weights_stride, positions_host);
  if(rc != SMPLPP_OK) return rc;
  smplpp_tasks::MarkerPipe & mp = tasks->marker;
  const size_t n = tasks->d.n;
  const size_t theta_row = (kJoints + 1) * 3;
  const int64_t chunk = std::min<int64_t>(batch, task_chunk_frames());
  const size_t C = static_cast<size_t>(chunk);
  const bool beta_pf = beta_stride != 0, vw_pf = vertex_weights_stride != 0;

  if(!mp.compute)
  {
    SB_CUDA(cudaStreamCreateWithFlags(&mp.h2d, cudaStreamNonBlocking));
    SB_CUDA(cudaStreamCreateWithFlags(&mp.compute, cudaStreamNonBlocking));
    SB_CUDA(cudaStreamCreateWithFlags(&mp.d2h, cudaStreamNonBlocking));
    for(int i = 0; i < 2; i++)
    {
      SB_CUDA(cudaEventCreateWithFlags(&mp.uploaded[i], cudaEventDisableTiming));
      SB_CUDA(cudaEventCreateWithFlags(&mp.computed[i], cudaEventDisableTiming));
      SB_CUDA(cudaEventCreateWithFlags(&mp.drained[i], cudaEventDisableTiming));
    }
  }
  // per-chunk layouts: inputs theta | beta (per frame) | weights (per frame), outputs positions | normals
  const size_t o_beta = align_up(C * theta_row * sizeof(float));
  const size_t o_vw = o_beta + (beta_pf ? align_up(C * beta_stride * sizeof(float)) : 0);
  const size_t in_bytes = o_vw + (vw_pf ? align_up(C * 3 * n * sizeof(float)) : 0);
  const size_t o_nrm = align_up(C * n * 3 * sizeof(float));
  const size_t out_bytes = o_nrm + (normals_host ? align_up(C * n * 3 * sizeof(float)) : 0);
  const size_t o_shared_vw = align_up(kShapeDim * sizeof(float));
  const size_t shared_bytes = o_shared_vw + align_up(3 * n * sizeof(float));
  for(int i = 0; i < 2; i++)
  {
    size_t hi = mp.dev_in_bytes, ho = mp.dev_out_bytes;
    if((rc = grow_dev(&mp.dev_in[i], &hi, in_bytes)) != SMPLPP_OK) return rc;
    if((rc = grow_dev(&mp.dev_out[i], &ho, out_bytes)) != SMPLPP_OK) return rc;
    if(i == 1) mp.dev_in_bytes = hi, mp.dev_out_bytes = ho;
  }
  if((rc = grow_dev(&mp.dev_shared, &mp.dev_shared_bytes, shared_bytes)) != SMPLPP_OK) return rc;
  if((rc = grow_dev(&mp.ws, &mp.ws_bytes, smplpp_task_forward_workspace_bytes(tasks, chunk))) != SMPLPP_OK) return rc;

  const bool in_locked = is_page_locked(theta_host) && (!beta_pf || is_page_locked(beta_host))
                         && (!vw_pf || is_page_locked(vertex_weights_host));
  const bool out_locked = is_page_locked(positions_host) && (!normals_host || is_page_locked(normals_host));
  for(int i = 0; i < 2; i++)
  {
    size_t hi = mp.pin_in_bytes, ho = mp.pin_out_bytes;
    if(!in_locked && (rc = grow_pinned(&mp.pin_in[i], &hi, in_bytes)) != SMPLPP_OK) return rc;
    if(!out_locked && (rc = grow_pinned(&mp.pin_out[i], &ho, out_bytes)) != SMPLPP_OK) return rc;
    if(i == 1) mp.pin_in_bytes = hi, mp.pin_out_bytes = ho;
  }
  // shared beta / weights: uploaded once, ahead of every chunk on the upload stream
  char * shared = static_cast<char *>(mp.dev_shared);
  if(!beta_pf) SB_CUDA(cudaMemcpyAsync(shared, beta_host, kShapeDim * sizeof(float), cudaMemcpyHostToDevice, mp.h2d));
  if(!vw_pf)
    SB_CUDA(cudaMemcpyAsync(shared + o_shared_vw, vertex_weights_host, 3 * n * sizeof(float), cudaMemcpyHostToDevice, mp.h2d));

  const int64_t nchunks = (batch + chunk - 1) / chunk;
  const int threads = host_threads();
  const size_t out_floats = n * 3;
  auto drain_to_pageable = [&](int64_t c) -> int {
    const int buf = static_cast<int>(c & 1);
    SB_CUDA(cudaEventSynchronize(mp.drained[buf]));
    const int64_t f0 = c * chunk, nb = std::min(chunk, batch - f0);
    const size_t bytes = static_cast<size_t>(nb) * out_floats * sizeof(float);
    const char * pin = static_cast<const char *>(mp.pin_out[buf]);
    parallel_memcpy(positions_host + static_cast<size_t>(f0) * out_floats, pin, bytes, threads);
    if(normals_host) parallel_memcpy(normals_host + static_cast<size_t>(f0) * out_floats, pin + o_nrm, bytes, threads);
    return SMPLPP_OK;
  };
  auto abort_all = [&](int code) {
    cudaStreamSynchronize(mp.h2d);
    cudaStreamSynchronize(mp.compute);
    cudaStreamSynchronize(mp.d2h);
    return code;
  };
  for(int64_t c = 0; c < nchunks; c++)
  {
    const int buf = static_cast<int>(c & 1);
    const int64_t f0 = c * chunk, nb = std::min(chunk, batch - f0);
    // ---- inputs of chunk c ----
    struct Piece
    {
      const void * src;
      size_t off, bytes;
    } pieces[3];
    int np = 0;
    pieces[np++] = {theta_host + static_cast<size_t>(f0) * theta_row, 0, static_cast<size_t>(nb) * theta_row * sizeof(float)};
    if(beta_pf)
      pieces[np++] = {beta_host + static_cast<size_t>(f0) * beta_stride, o_beta,
                      (static_cast<size_t>(nb - 1) * beta_stride + kShapeDim) * sizeof(float)};
    if(vw_pf)
      pieces[np++] = {vertex_weights_host + static_cast<size_t>(f0) * 3 * n, o_vw, static_cast<size_t>(nb) * 3 * n * sizeof(float)};
    if(!in_locked)
    {
      // pin_in[buf] is free once the upload of chunk c-2 has left it
      if(c >= 2) SB_CUDA(cudaEventSynchronize(mp.uploaded[buf]));
      for(int i = 0; i < np; i++)
        parallel_memcpy(static_cast<char *>(mp.pin_in[buf]) + pieces[i].off, pieces[i].src, pieces[i].bytes, threads);
    }
    // dev_in[buf] is free once the compute of chunk c-2 has read it
    if(c >= 2) SB_CUDA(cudaStreamWaitEvent(mp.h2d, mp.computed[buf], 0));
    char * din = static_cast<char *>(mp.dev_in[buf]);
    for(int i = 0; i < np; i++)
    {
      const void * src = in_locked ? pieces[i].src : static_cast<const void *>(static_cast<char *>(mp.pin_in[buf]) + pieces[i].off);
      SB_CUDA(cudaMemcpyAsync(din + pieces[i].off, src, pieces[i].bytes, cudaMemcpyHostToDevice, mp.h2d));
    }
    SB_CUDA(cudaEventRecord(mp.uploaded[buf], mp.h2d));
    // ---- compute of chunk c: after its upload, into dev_out[buf] once the download of chunk c-2 has left it ----
    SB_CUDA(cudaStreamWaitEvent(mp.compute, mp.uploaded[buf], 0));
    if(c >= 2) SB_CUDA(cudaStreamWaitEvent(mp.compute, mp.drained[buf], 0));
    char * dout = static_cast<char *>(mp.dev_out[buf]);
    rc = smplpp_task_forward(model, tasks, mp.compute, nb, beta_pf ? reinterpret_cast<float *>(din + o_beta) : reinterpret_cast<float *>(shared),
                             beta_stride, reinterpret_cast<float *>(din),
                             vw_pf ? reinterpret_cast<float *>(din + o_vw) : reinterpret_cast<float *>(shared + o_shared_vw),
                             vertex_weights_stride, normal_offset, reinterpret_cast<float *>(dout),
                             normals_host ? reinterpret_cast<float *>(dout + o_nrm) : nullptr, mp.ws, mp.ws_bytes);
    if(rc != SMPLPP_OK) return abort_all(rc);
    SB_CUDA(cudaEventRecord(mp.computed[buf], mp.compute));
    // ---- download of chunk c ----
    SB_CUDA(cudaStreamWaitEvent(mp.d2h, mp.computed[buf], 0));
    const size_t bytes = static_cast<size_t>(nb) * out_floats * sizeof(float);
    char * pin = static_cast<char *>(mp.pin_out[buf]); // emptied by the host when chunk c-1 was issued (drain of c-2)
    SB_CUDA(cudaMemcpyAsync(out_locked ? static_cast<void *>(positions_host + static_cast<size_t>(f0) * out_floats) : pin, dout,
                            bytes, cudaMemcpyDeviceToHost, mp.d2h));
    if(normals_host)
      SB_CUDA(cudaMemcpyAsync(out_locked ? static_cast<void *>(normals_host + static_cast<size_t>(f0) * out_floats) : pin + o_nrm,
                              dout + o_nrm, bytes, cudaMemcpyDeviceToHost, mp.d2h));
    SB_CUDA(cudaEventRecord(mp.drained[buf], mp.d2h));
    if(!out_locked && c >= 1)
    {
      rc = drain_to_pageable(c - 1);
      if(rc != SMPLPP_OK) return abort_all(rc);
    }
  }
  if(!out_locked)
  {
    rc = drain_to_pageable(nchunks - 1);
    if(rc != SMPLPP_OK) return abort_all(rc);
  }
  SB_CUDA(cudaStreamSynchronize(mp.d2h));
  SB_CUDA(cudaStreamSynchronize(mp.compute));
  SB_CUDA(cudaStreamSynchronize(mp.h2d));
  return SMPLPP_OK;
}
