// Shared declarations of the smplpp_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/smplpp_b200.h"

namespace sb
{
constexpr int kJoints = SMPLPP_JOINT_NUM;
constexpr int kShapeDim = SMPLPP_SHAPE_DIM;
constexpr int kPoseDim = SMPLPP_POSE_DIM;
// K of the fused blend contraction: 207 pose features | 10 betas | 1 (template) | zero padding
constexpr int kBlendK = 224;
constexpr int kBlendKUsed = kPoseDim + kShapeDim + 1; // 218
constexpr int kXformFloats = 12;                      // 3x4 row-major [R | t] per joint
constexpr int kGroupVerts = 4;                        // consecutive vertices handled by one skinning lane
constexpr int kGroupJoints = 8;                       // max distinct joints of a group on the register-reuse path

extern thread_local std::string g_last_error;
extern std::atomic<uint64_t> g_launch_count;

int fail(int code, const char * module, const std::string & msg);

#define SB_CUDA(expr)                                                                                   \
  do                                                                                                    \
  {                                                                                                     \
    cudaError_t err__ = (expr);                                                                         \
    if(err__ != cudaSuccess)                                                                            \
      return ::sb::fail(SMPLPP_ERR_CUDA, "CUDA", std::string(#expr) + ": " + cudaGetErrorString(err__)); \
  } while(0)

#define SB_LAUNCHED()                                                              \
  do                                                                               \
  {                                                                                \
    ::sb::g_launch_count.fetch_add(1, std::memory_order_relaxed);                  \
    cudaError_t err__ = cudaPeekAtLastError();                                     \
    if(err__ != cudaSuccess)                                                       \
      return ::sb::fail(SMPLPP_ERR_CUDA, "CUDA", std::string("kernel launch: ") + cudaGetErrorString(err__)); \
  } while(0)

inline cudaStream_t as_stream(void * s)
{
  return static_cast<cudaStream_t>(s);
}

template<typename T>
inline T * align_up_ptr(void * p, size_t a = 256)
{
  return reinterpret_cast<T *>((reinterpret_cast<uintptr_t>(p) + a - 1) / a * a);
}

inline size_t align_up(size_t n, size_t a = 256)
{
  return (n + a - 1) / a * a;
}

// true the first time it is called on the current device with this flag array (function attributes and memory-pool
// settings are per device; one process may drive several devices)
inline bool first_call_on_device(bool (&done)[64])
{
  int dev = 0;
  if(cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
  if(done[dev]) return false;
  done[dev] = true;
  return true;
}

// Device-resident constants of one model.  Immutable after create => shareable across streams/threads.
struct ModelDev
{
  int V = 0;      // vertices
  int Vpad = 0;   // V rounded up to the blend tile (64 vertices)
  int F = 0;      // faces
  int kmax = 0;   // max skinning influences per vertex
  // fused blend basis, K-major: row (3 v + k) holds [pose basis 207 | shape basis 10 | template | 0 x 6]
  float * basis = nullptr; // (3 Vpad, 224)
  // skinning weights, ELL, structure-of-arrays over influences: [kmax][Vpad]
  uint8_t * lbs_joint = nullptr;
  float * lbs_weight = nullptr;
  float * lbs_wsum = nullptr; // (Vpad) sum_j W[v,j]  (homogeneous coordinate h[3])
  // per group of 4 consecutive vertices (one lane of the skinning kernel): the union of the joints influencing
  // the group (<= kGroupJoints, 0xFF padded; count = -1 marks an overflowing group) and dense weights over it.
  // A lane then fetches each transform ONCE for its 4 vertices: ~3.7 instead of 16 transform fetches per group.
  int8_t * group_nj = nullptr;      // (Vpad / 4)
  uint8_t * group_joint = nullptr;  // (Vpad / 4, kGroupJoints)
  float * group_w = nullptr;        // (Vpad / 4, kGroupJoints, 4)  [joint slot][vertex in group]
  // joints = J_T + J_S beta  (Jreg (T + S beta), JointRegression.cpp:588-590)
  float * joint_template = nullptr; // (24, 3)
  float * joint_shape = nullptr;    // (24, 3, 10)
  int parent[kJoints];              // -1 for the root
  int depth[kJoints];
  int max_depth = 0;
  // topology
  int32_t * faces = nullptr;     // (F, 3) 0-based
  int32_t * adj_offset = nullptr; // (V + 1) CSR: vertex -> adjacent faces
  int32_t * adj_faces = nullptr;
  // originals kept for the task builder and the generic module kernels
  float * weights_dense = nullptr; // (V, 24)
  uint32_t * vert_jmask = nullptr; // (V) joints whose rotation moves the vertex (ancestor closure of its influences)
  // tcgen05 blend + skinning (skin_tc3.cu): fp16 hi | lo split basis scaled by 2^tc3_basis_exp.  tc3_ready also
  // gates the tcgen05 standalone skinning kernel (lbs_tc.cu).
  void * basis_img16 = nullptr; // [tile][K-block][hi | lo][plane][128][32 fp16]: SWIZZLE_64B stage images
  // the two 16-slot joint windows of the skinning product (tc3_layout.cuh): slot s (window s / 16) holds joint
  // tc3_slot_joint[s] or -1; a joint in both windows has its primary slot (tc3_joint_slot) in window 0
  int8_t tc3_slot_joint[32] = {};
  int8_t tc3_joint_slot[kJoints] = {};
  uint8_t * tc3_tile_mode = nullptr; // (tc3_tiles) per 128-vertex tile: 0 / 1 = its joints fit window 0 / 1, 2 = both
  int tc3_basis_exp = 0;
  int tc3_tiles = 0;
  bool tc3_ready = false;
  int sm_count = 0;
};
} // namespace sb

struct smplpp_model
{
  sb::ModelDev d;
  // host copies used by smplpp_tasks_create
  std::vector<int32_t> h_faces;      // 0-based
  std::vector<int32_t> h_adj_offset; // CSR
  std::vector<int32_t> h_adj_faces;
  std::vector<float> h_basis;        // (3V, 224) same row layout as d.basis (unpadded V)
  std::vector<float> h_weights;      // (V, 24)
  std::vector<uint32_t> h_vert_jmask; // (V)
  std::vector<float> h_joint_template, h_joint_shape;
  // smplpp_forward_host: chunked, double-buffered pipeline (compute stream + copy stream)
  struct HostPipe
  {
    cudaStream_t compute = nullptr, copy = nullptr;
    cudaEvent_t done[2] = {nullptr, nullptr};    // chunk computed (compute stream)
    cudaEvent_t drained[2] = {nullptr, nullptr}; // chunk copied out (copy stream)
    void * dev_in = nullptr;                     // beta | theta of the whole batch
    size_t dev_in_bytes = 0;
    void * dev_out[2] = {nullptr, nullptr};      // vertices of one chunk
    size_t dev_out_bytes = 0;
    void * dev_joints = nullptr;                 // joints of the whole batch
    size_t dev_joints_bytes = 0;
    void * ws = nullptr;                         // forward workspace of one chunk
    size_t ws_bytes = 0;
    void * pin_in = nullptr;                     // staging for pageable inputs
    size_t pin_in_bytes = 0;
    void * pin_out[2] = {nullptr, nullptr};      // staging for pageable outputs (one chunk each)
    size_t pin_out_bytes = 0;
  } pipe;
};
