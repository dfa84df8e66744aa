// Internal launch helpers shared by forward.cu, skin_tc3.cu, lbs_tc.cu and ik.cu.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace sb
{
struct ChainTopo
{
  int parent[kJoints];
  int depth[kJoints];
  int max_depth;
};

ChainTopo make_topo(const ModelDev & d);

// K1: rodrigues + pose features + joints + kinematic chain (one warp per frame)
// tc3_scratch (nullable, tc3_frame_operand_bytes(B) bytes): also write the stage images of K2'''
int launch_pose_chain(const ModelDev & d, cudaStream_t st, int B, const float * beta, long long beta_stride,
                      const float * theta, float * coef, float * xforms, float * joints, float * xforms44,
                      void * tc3_scratch = nullptr);
// K2 (FFMA): fused blend contraction (+ skinning when skin == true, else writes the rest shape)
int launch_blend_skin_ffma(const ModelDev & d, cudaStream_t st, int B, const float * coef, const float * xforms,
                           const float * theta, float * out, bool skin);
// K2''' (skin_tc3.cu): fp16 split-precision blend AND skinning matrices on tcgen05 in a persistent CTA per SM; GEMM 1 of
// item i+1 runs under GEMM 2 + epilogue of item i.  tc3_prepare_model sets d.tc3_ready when the device and the model can
// run it; basis_max_abs is the largest pose / shape basis entry
int tc3_prepare_model(ModelDev & d, float basis_max_abs, const float * weights);
void tc3_release_model(ModelDev & d);
size_t tc3_frame_operand_bytes(int64_t batch);
// images_ready: the scratch area already holds the stage images (written by K1); else they are built from coef / xforms
int launch_blend_skin_tc3(const ModelDev & d, cudaStream_t st, int B, const float * coef, const float * xforms, void * scratch,
                          const float * theta, float * out, bool images_ready = false);
// K3: standalone skinning; affine: xforms are (B,24,3,4) else (B,24,4,4)
int launch_lbs(const ModelDev & d, cudaStream_t st, int B, const float * rest, const float * xforms, bool affine,
               const float * root, int root_stride, float * out);

// K3' (lbs_tma.cu): per-warp TMA pipelines; needs even V, 16-byte aligned tensors, affine (3x4) transforms
bool lbs_tma_usable(const ModelDev & d, const float * rest, const float * out, const float * xforms);
int launch_lbs_tma(const ModelDev & d, cudaStream_t st, int B, const float * rest, const float * xforms, const float * root,
                   int root_stride, float * out);
// K3'' (lbs_tc.cu): skinning matrices on tcgen05; needs the tc3 model data, even V >= 128, 16-byte aligned tensors
bool lbs_tc_usable(const ModelDev & d, const float * rest, const float * out, const float * xforms);
int launch_lbs_tc(const ModelDev & d, cudaStream_t st, int B, const float * rest, const float * xforms, int xf_floats,
                  const float * root, int root_stride, float * out);
// cuTensorMapEncodeTiled of the driver (lbs_tc.cu), nullptr when the driver does not provide it
using EncodeTiledFn = CUresult (*)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                   const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn();
extern std::atomic<int> g_lbs_variant; // 0: FFMA TMA pipeline when usable, 1: FFMA register-pipelined kernel, 2: tcgen05 (default)
// frees the streams, events and buffers of smplpp_forward_host (host_pipe.cu)
void release_host_pipe(smplpp_model * m);

extern std::atomic<int> g_forward_variant;
} // namespace sb
