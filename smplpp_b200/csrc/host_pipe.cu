// smplpp_forward_host: the forward pass with HOST buffers (the call a user of smplpp::SMPL::launch + getVertex +
// getRestJoint makes, src/SMPL.cpp:671-737, 386-516), as a chunked, double-buffered pipeline:
//
//   compute stream :  H2D(beta, theta) | fwd(chunk 0) | fwd(chunk 1) | fwd(chunk 2) ...
//   copy stream    :                                 D2H(chunk 0)  | D2H(chunk 1) ...
//   host threads   :                                                memcpy(chunk 0) ...   (pageable destinations only)
//
// A mesh is 82 680 B of output against 340 B of input, so the call is bound by the device->host link; the pipeline
// keeps that link busy from the first chunk on.  Page-locked caller buffers (smplpp_host_alloc, smplpp_host_register
// or any cudaHostAlloc/cudaHostRegister memory) are the DMA source/target themselves; pageable buffers are staged
// through two pinned chunk buffers and copied out by a few host threads while the next chunk is in flight.
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "forward.cuh"
#include "host_copy.cuh"

using namespace sb;

namespace
{
int chunk_frames()
{
  static int n = 0;
  if(n == 0)
  {
    const char * e = getenv("SMPLPP_HOST_CHUNK");
    n = e ? atoi(e) : 256;
    n = std::max(1, std::min(n, 1 << 16));
  }
  return n;
}
} // namespace

namespace sb
{
void release_host_pipe(smplpp_model * m)
{
  smplpp_model::HostPipe & hp = m->pipe;
  for(int i = 0; i < 2; i++)
  {
    if(hp.done[i]) cudaEventDestroy(hp.done[i]);
    if(hp.drained[i]) cudaEventDestroy(hp.drained[i]);
    if(hp.dev_out[i]) cudaFree(hp.dev_out[i]);
    if(hp.pin_out[i]) cudaFreeHost(hp.pin_out[i]);
  }
  if(hp.dev_in) cudaFree(hp.dev_in);
  if(hp.dev_joints) cudaFree(hp.dev_joints);
  if(hp.ws) cudaFree(hp.ws);
  if(hp.pin_in) cudaFreeHost(hp.pin_in);
  if(hp.compute) cudaStreamDestroy(hp.compute);
  if(hp.copy) cudaStreamDestroy(hp.copy);
  hp = smplpp_model::HostPipe();
}
} // namespace sb

extern "C" int smplpp_host_alloc(void ** out, size_t bytes)
{
  if(!out || bytes == 0) return fail(SMPLPP_ERR_INVALID, "SMPL", "smplpp_host_alloc: bad arguments");
  *out = nullptr;
  SB_CUDA(cudaHostAlloc(out, bytes, cudaHostAllocPortable));
  return SMPLPP_OK;
}

extern "C" void smplpp_host_free(void * p)
{
  if(p) cudaFreeHost(p);
}

extern "C" int smplpp_host_register(void * p, size_t bytes)
{
  if(!p || bytes == 0) return fail(SMPLPP_ERR_INVALID, "SMPL", "smplpp_host_register: bad arguments");
  SB_CUDA(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
  return SMPLPP_OK;
}

extern "C" int smplpp_host_unregister(void * p)
{
  if(!p) return SMPLPP_OK;
  SB_CUDA(cudaHostUnregister(p));
  return SMPLPP_OK;
}

extern "C" int smplpp_forward_host(const smplpp_model_t * model_c, int64_t batch, const float * beta_host,
                                   int64_t beta_stride, const float * theta_host, float * vertices_host,
                                   float * joints_host)
{
  smplpp_model_t * model = const_cast<smplpp_model_t *>(model_c);
  if(!model || batch < 1 || !beta_host || !theta_host)
    return fail(SMPLPP_ERR_INVALID, "SMPL", "Cannot launch a SMPL model!");
  if(beta_stride != 0 && beta_stride < kShapeDim) return fail(SMPLPP_ERR_INVALID, "BlendShape", "Failed to set beta!");
  smplpp_model::HostPipe & hp = model->pipe;
  const size_t V = model->d.V;
  const size_t theta_row = (kJoints + 1) * 3;
  const size_t n_beta = beta_stride == 0 ? kShapeDim : static_cast<size_t>(batch - 1) * beta_stride + kShapeDim;
  const size_t n_theta = static_cast<size_t>(batch) * theta_row;
  const int64_t chunk = std::min<int64_t>(batch, chunk_frames());
  const size_t chunk_vert_bytes = align_up(static_cast<size_t>(chunk) * V * 3 * sizeof(float));

  if(!hp.compute)
  {
    SB_CUDA(cudaStreamCreateWithFlags(&hp.compute, cudaStreamNonBlocking));
    SB_CUDA(cudaStreamCreateWithFlags(&hp.copy, cudaStreamNonBlocking));
    for(int i = 0; i < 2; i++)
    {
      SB_CUDA(cudaEventCreateWithFlags(&hp.done[i], cudaEventDisableTiming));
      SB_CUDA(cudaEventCreateWithFlags(&hp.drained[i], cudaEventDisableTiming));
    }
  }
  const size_t beta_bytes = align_up(n_beta * sizeof(float));
  const size_t in_bytes = beta_bytes + align_up(n_theta * sizeof(float));
  int rc = grow_dev(&hp.dev_in, &hp.dev_in_bytes, in_bytes);
  if(rc != SMPLPP_OK) return rc;
  if(vertices_host)
  {
    size_t have = hp.dev_out_bytes;
    for(int i = 0; i < 2; i++)
    {
      size_t h = have;
      rc = grow_dev(&hp.dev_out[i], &h, chunk_vert_bytes);
      if(rc != SMPLPP_OK) return rc;
      if(i == 1) hp.dev_out_bytes = h;
    }
  }
  if(joints_host)
  {
    rc = grow_dev(&hp.dev_joints, &hp.dev_joints_bytes, static_cast<size_t>(batch) * kJoints * 3 * sizeof(float));
    if(rc != SMPLPP_OK) return rc;
  }
  const size_t ws_need = smplpp_forward_workspace_bytes(model, chunk);
  rc = grow_dev(&hp.ws, &hp.ws_bytes, ws_need);
  if(rc != SMPLPP_OK) return rc;

  // ---- inputs ----
  float * d_beta = static_cast<float *>(hp.dev_in);
  float * d_theta = reinterpret_cast<float *>(static_cast<char *>(hp.dev_in) + beta_bytes);
  const bool in_locked = is_page_locked(beta_host) && is_page_locked(theta_host);
  if(in_locked)
  {
    SB_CUDA(cudaMemcpyAsync(d_beta, beta_host, n_beta * sizeof(float), cudaMemcpyHostToDevice, hp.compute));
    SB_CUDA(cudaMemcpyAsync(d_theta, theta_host, n_theta * sizeof(float), cudaMemcpyHostToDevice, hp.compute));
  }
  else
  {
    rc = grow_pinned(&hp.pin_in, &hp.pin_in_bytes, in_bytes);
    if(rc != SMPLPP_OK) return rc;
    char * pin = static_cast<char *>(hp.pin_in);
    memcpy(pin, beta_host, n_beta * sizeof(float));
    memcpy(pin + beta_bytes, theta_host, n_theta * sizeof(float));
    SB_CUDA(cudaMemcpyAsync(hp.dev_in, pin, in_bytes, cudaMemcpyHostToDevice, hp.compute));
  }

  // ---- chunks ----
  const bool out_locked = vertices_host && is_page_locked(vertices_host);
  const bool staged = vertices_host && !out_locked;
  if(staged)
  {
    size_t have = hp.pin_out_bytes;
    for(int i = 0; i < 2; i++)
    {
      size_t h = have;
      rc = grow_pinned(&hp.pin_out[i], &h, chunk_vert_bytes);
      if(rc != SMPLPP_OK) return rc;
      if(i == 1) hp.pin_out_bytes = h;
    }
  }
  const int64_t nchunks = (batch + chunk - 1) / chunk;
  const int threads = host_threads();
  auto drain_to_pageable = [&](int64_t c) -> int {
    const int buf = static_cast<int>(c & 1);
    SB_CUDA(cudaEventSynchronize(hp.drained[buf]));
    const int64_t f0 = c * chunk, nb = std::min(chunk, batch - f0);
    parallel_memcpy(vertices_host + static_cast<size_t>(f0) * V * 3, hp.pin_out[buf],
                    static_cast<size_t>(nb) * V * 3 * sizeof(float), threads);
    return SMPLPP_OK;
  };
  for(int64_t c = 0; c < nchunks; c++)
  {
    const int buf = static_cast<int>(c & 1);
    const int64_t f0 = c * chunk, nb = std::min(chunk, batch - f0);
    // dev_out[buf] is free again once chunk c-2 left the device
    if(c >= 2 && vertices_host) SB_CUDA(cudaStreamWaitEvent(hp.compute, hp.drained[buf], 0));
    float * d_vert = vertices_host ? static_cast<float *>(hp.dev_out[buf]) : nullptr;
    float * d_joint = joints_host ? static_cast<float *>(hp.dev_joints) + static_cast<size_t>(f0) * kJoints * 3 : nullptr;
    rc = smplpp_forward(model, hp.compute, nb, d_beta + static_cast<size_t>(f0) * beta_stride, beta_stride,
                        d_theta + static_cast<size_t>(f0) * theta_row, d_vert, d_joint, nullptr, nullptr, hp.ws, hp.ws_bytes);
    if(rc != SMPLPP_OK)
    {
      cudaStreamSynchronize(hp.compute);
      cudaStreamSynchronize(hp.copy);
      return rc;
    }
    if(vertices_host)
    {
      SB_CUDA(cudaEventRecord(hp.done[buf], hp.compute));
      SB_CUDA(cudaStreamWaitEvent(hp.copy, hp.done[buf], 0));
      // pin_out[buf] was emptied by the host when chunk c-1 was issued (drain of chunk c-2 below)
      void * dst = staged ? hp.pin_out[buf] : static_cast<void *>(vertices_host + static_cast<size_t>(f0) * V * 3);
      SB_CUDA(cudaMemcpyAsync(dst, d_vert, static_cast<size_t>(nb) * V * 3 * sizeof(float), cudaMemcpyDeviceToHost, hp.copy));
      SB_CUDA(cudaEventRecord(hp.drained[buf], hp.copy));
      if(staged && c >= 1)
      {
        rc = drain_to_pageable(c - 1);
        if(rc != SMPLPP_OK) return rc;
      }
    }
  }
  if(joints_host)
  {
    const size_t jb = static_cast<size_t>(batch) * kJoints * 3 * sizeof(float);
    SB_CUDA(cudaMemcpyAsync(joints_host, hp.dev_joints, jb, cudaMemcpyDeviceToHost, hp.compute));
  }
  if(staged)
  {
    rc = drain_to_pageable(nchunks - 1);
    if(rc != SMPLPP_OK) return rc;
  }
  SB_CUDA(cudaStreamSynchronize(hp.copy));
  SB_CUDA(cudaStreamSynchronize(hp.compute));
  return SMPLPP_OK;
}
