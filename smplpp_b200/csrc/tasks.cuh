// IK task set: attachment faces of n markers, the 1-ring topology needed by IkTask::calcActualNormal
// (reference src/IkTask.cpp:74-86 -> SMPL::calcVertexNormal src/SMPL.cpp:527-535) and a compact copy of the
// blend basis / skinning rows of the vertices the tasks depend on.
#pragma once
#include "common.cuh"
#include "ik_poseblend.cuh"

namespace sb
{
// Device-side view handed to kernels by value.
struct TasksDev
{
  int n = 0;        // tasks (markers)
  int nU = 0;       // distinct mesh vertices used: corners first (nCorner), then 1-ring-only vertices
  int nCorner = 0;  // distinct corner vertices
  int nUpad = 0;    // nU rounded up to 64 (tile of the sparse forward)
  int nItems = 0;   // (task, corner, adjacent face) triples
  int nPairs = 0;   // (task, vertex) pairs; per task: corners 0,1,2 first, then ring vertices
  int maxPairs = 0; // max pairs of one task
  int kmax = 0;     // skinning influences per vertex (as in the model)
  const int32_t * corner = nullptr;       // (n, 3)   local vertex id of the face corners
  const int32_t * item_off = nullptr;     // (3n + 1) CSR (task, corner) -> items
  const int32_t * item_verts = nullptr;   // (nItems, 3) local vertex ids of the adjacent face, in face order
  const int32_t * pair_off = nullptr;     // (n + 1)  CSR task -> pairs
  const int32_t * pair_vert = nullptr;    // (nPairs) local vertex id
  const int32_t * pair_task = nullptr;    // (nPairs) owning task
  const int32_t * pair_ref_off = nullptr; // (nPairs + 1) CSR pair -> references
  const int32_t * pair_refs = nullptr;    // item * 4 + slot (slot = position of the vertex in the item's face)
  const int32_t * pair_order = nullptr;   // (nPairs) pairs by decreasing reference count (balanced warps in ik_jacobian_kernel)
  const uint32_t * task_joint_mask = nullptr; // (n) joints that move any vertex of the task (corners only: bit 24+)
  const uint32_t * task_joint_mask_corner = nullptr; // (n) same, restricted to the three corners
  // compact model rows of the nU vertices (same layouts as ModelDev, V -> nU)
  const float * basis = nullptr;       // (3 nUpad, 224)
  const float4 * basis4 = nullptr;     // (nUpad, 224): (x, y, z, 0) of every basis column, one 16-byte load in the IK Jacobian
  const uint8_t * lbs_joint = nullptr; // [kmax][nUpad]
  const float * lbs_weight = nullptr;  // [kmax][nUpad]
  const float * lbs_wsum = nullptr;    // (nUpad)
  const float * sw_norm = nullptr;     // (nU, kmax) W[u, slot] / sum_j W[u, j]: the layout ik_jacobian_kernel keeps in shared memory
  const uint8_t * sj_flat = nullptr;   // (nU, kmax) joint of the slot
};
// ---- fused IK step (ik2.cu): one self-contained topology record per task -------------------------------------------
// Everything the step needs about ONE attachment face: its three corners, their 1-rings (SMPL::calcVertexNormal,
// src/SMPL.cpp:527-535) and the distinct vertices ("pairs") these touch, as GLOBAL vertex ids of the model.  A task set
// holds n of them (all frames share the topology); per-frame attachments (IkTask::faceIdx_ re-seated by the projection of
// node/node.cpp:993-1001) are (B, n) records built on the device by task_topo_kernel.
constexpr int kRecPairs = 48; // distinct vertices of a task: 3 corners + ring
constexpr int kRecItems = 48; // (corner, adjacent face) items of a task = sum of the three corner valences
struct alignas(16) TaskRec
{
  int32_t face;          // 0-based row of face_indices; < 0 marks a record that does not fit (valence too high)
  uint32_t jmask;        // joints that move any pair (ancestor closure of the influencing joints)
  uint32_t jmask_corner; // the same for the three corners only
  uint8_t np;            // pairs; pairs 0..2 are corners 0..2 of the face (in face order)
  uint8_t ni;            // items, ordered by corner
  uint8_t nic[3];        // items per corner
  uint8_t pad[3];
  int32_t gv[kRecPairs];            // global vertex id of every pair
  uint8_t item[kRecItems][4];       // pair-local ids of the adjacent face's vertices in face order; [3] = corner
  uint8_t ref_off[kRecPairs + 1];   // CSR pair -> references
  uint8_t refs[3 * kRecItems];      // item * 4 + slot (slot = position of the pair in the item's face)
  uint8_t pad2[3];
};
static_assert(sizeof(TaskRec) == 608, "TaskRec layout");
// skinning rows of the pairs of a record (models with at most 4 influences per vertex, i.e. SMPL): fetched with the
// record, so that the skinning phase of a task starts without a dependent chain of global loads
struct alignas(16) TaskSkin
{
  float w[kRecPairs][4];   // raw weights W[v, j] of the (up to) four influences
  float ws[kRecPairs];     // sum_j W[v, j] (the homogeneous coordinate)
  uint8_t j[kRecPairs][4]; // joints
};
static_assert(sizeof(TaskSkin) == 1152, "TaskSkin layout");
} // namespace sb

struct smplpp_tasks
{
  sb::TasksDev d;
  sb::ModelDev sub;      // sparse-forward view (basis/lbs arrays alias the TasksDev ones)
  sb::ModelDev sub_corner; // same arrays, V = nCorner (no normals needed)
  sb::PoseBlendTc pb;   // operand images of ik_poseblend_tc_kernel
  std::vector<void *> allocations;
  std::vector<int64_t> h_face_idx;
  std::vector<int32_t> h_sub_vert; // local -> global vertex id
  std::vector<int32_t> h_corner;
  // fused IK step (ik2.cu)
  const sb::TaskRec * recs = nullptr; // (n) device
  const sb::TaskSkin * skins = nullptr; // (n) device, null when the model has more than 4 influences per vertex
  const long long * face_idx_dev = nullptr; // (n) device copy of the attachment faces (smplpp_task_positions / _tangents)
  int maxPairs = 0, maxItems = 0, maxLive = 0, maxPairsCorner = 3;
  // smplpp_ik_solve_host (ik_host.cu): grow-only device buffers and the stream of the host-buffer call
  struct HostSolve
  {
    cudaStream_t stream = nullptr;
    void * buf = nullptr;
    size_t buf_bytes = 0;
    void * ws = nullptr;
    size_t ws_bytes = 0;
  } host;
  // smplpp_task_forward_host (task_forward.cu): chunked pipeline, H2D of chunk c+1 | compute of chunk c | D2H of chunk c-1
  struct MarkerPipe
  {
    cudaStream_t h2d = nullptr, compute = nullptr, d2h = nullptr;
    cudaEvent_t uploaded[2] = {nullptr, nullptr}; // inputs of the chunk on the device (h2d stream)
    cudaEvent_t computed[2] = {nullptr, nullptr}; // outputs of the chunk written, inputs consumed (compute stream)
    cudaEvent_t drained[2] = {nullptr, nullptr};  // outputs of the chunk copied out (d2h stream)
    void * dev_in[2] = {nullptr, nullptr};        // theta | beta (per frame) | vertex weights (per frame) of one chunk
    size_t dev_in_bytes = 0;
    void * dev_out[2] = {nullptr, nullptr};       // positions | normals of one chunk
    size_t dev_out_bytes = 0;
    void * dev_shared = nullptr;                  // shared beta | shared vertex weights
    size_t dev_shared_bytes = 0;
    void * ws = nullptr;                          // smplpp_task_forward workspace of one chunk
    size_t ws_bytes = 0;
    void * pin_in[2] = {nullptr, nullptr};        // staging of pageable inputs
    size_t pin_in_bytes = 0;
    void * pin_out[2] = {nullptr, nullptr};       // staging of pageable outputs
    size_t pin_out_bytes = 0;
  } marker;
};
void sb_release_host_solve(smplpp_tasks * t);
void sb_release_marker_pipe(smplpp_tasks * t);
