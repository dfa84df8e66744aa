/* smplpp_b200 — C ABI of the B200-native (sm_100a) SMPL forward + MoSh/MoSh++ IK hot path.
 *
 * This is the drop-in boundary for the data-parallel path of mmurooka/SMPLpp.  The reference exposes the
 * path as plain C++ classes in libsmplpp.so (no FFI, no plugin registry; SURVEY.md §8b); every entry point
 * below names the reference interface it replaces (file:line, relative to the reference tree).  Signatures
 * use only plain pointers, sizes and opaque handles: no libtorch / CUDA runtime types.
 *
 * Conventions
 *   - all arrays are dense, row-major, float32 unless stated; `_dev` pointers are device memory on the
 *     current CUDA device, `_host` pointers are host memory;
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); device entry points only enqueue
 *     work on it and never synchronise;
 *   - every function returns SMPLPP_OK (0) or a negative error code; smplpp_last_error() returns the
 *     reference-style message ("<module> Error: <text>", src/toolbox/Exception.cpp:77-91) of the last
 *     failure on the calling thread;
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     SMPLPP_ERR_CUDA.
 */
#ifndef SMPLPP_B200_H
#define SMPLPP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMPLPP_OK 0
#define SMPLPP_ERR_INVALID (-1) /* bad argument / shape (the reference throws smpl_error) */
#define SMPLPP_ERR_CUDA (-2)    /* CUDA runtime failure, or no device */
#define SMPLPP_ERR_ALLOC (-3)
#define SMPLPP_ERR_IO (-4)      /* missing / malformed parameter or mocap file */

/* shape constants of include/smplpp/definition/def.h:8-14 */
#define SMPLPP_VERTEX_NUM 6890
#define SMPLPP_FACE_NUM 13776
#define SMPLPP_JOINT_NUM 24
#define SMPLPP_SHAPE_DIM 10
#define SMPLPP_POSE_DIM 207
#define SMPLPP_LATENT_DIM 32
#define SMPLPP_VPOSER_HIDDEN 512
#define SMPLPP_VPOSER_JOINTS 21

typedef struct smplpp_model smplpp_model_t;
typedef struct smplpp_vposer smplpp_vposer_t;
typedef struct smplpp_tasks smplpp_tasks_t;
typedef struct smplpp_json smplpp_json_t;
typedef struct smplpp_c3d smplpp_c3d_t;
typedef struct smplpp_mocap_body smplpp_mocap_body_t;

const char * smplpp_last_error(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches evidence) */
uint64_t smplpp_launch_count(void);
int smplpp_device_count(void);

/* ---------------------------------------------------------------------------------------------------------
 * Model (replaces SMPL::init, src/SMPL.cpp:560-643: the tensors loaded from the model JSON)
 * ------------------------------------------------------------------------------------------------------- */
typedef struct smplpp_model_desc
{
  int64_t vertex_num;               /* 6890 for SMPL; any V >= 1 is accepted (Tester KATs use V = 1, 5) */
  int64_t face_num;                 /* 13776; may be 0 when no normals / IK tasks are needed */
  const int32_t * face_indices;     /* (face_num, 3), 1-BASED vertex ids as stored (SMPL.cpp:520) */
  const float * shape_blend_shapes; /* (V, 3, 10) */
  const float * pose_blend_shapes;  /* (V, 3, 207) */
  const float * vertices_template;  /* (V, 3) */
  const float * joint_regressor;    /* (24, V) */
  const int64_t * kinematic_tree;   /* (2, 24): row 0 parents (root: any value outside 0..23) */
  const float * weights;            /* (V, 24) dense; rows need not sum to 1 (homogeneous divide kept) */
} smplpp_model_desc;

int smplpp_model_create(const smplpp_model_desc * desc_host, smplpp_model_t ** out);
void smplpp_model_destroy(smplpp_model_t * model);
int64_t smplpp_model_vertex_num(const smplpp_model_t * model);
/* max non-zeros per row of `weights` found at create time (4 for SMPL) */
int smplpp_model_max_influences(const smplpp_model_t * model);

/* ---------------------------------------------------------------------------------------------------------
 * Forward pass (replaces SMPL::launch, src/SMPL.cpp:671-737 = BlendShape::blend + JointRegression::regress +
 * WorldTransformation::transform + LinearBlendSkinning::skinning, and the getters SMPL.cpp:386-516)
 *
 *   beta_dev   (B, 10) with row stride `beta_stride` floats; beta_stride == 0 shares one beta by all frames
 *   theta_dev  (B, 25, 3): row 0 = root translation, rows 1..24 = axis-angle (SMPL.cpp:685-686, 726-727)
 *   vertices   (B, V, 3)        SMPL::getVertex           (nullable)
 *   joints     (B, 24, 3)       SMPL::getRestJoint        (nullable)
 *   transforms (B, 24, 4, 4)    WorldTransformation::getTransformation (nullable)
 *   rest_shape (B, V, 3)        SMPL::getRestShape        (nullable; forces the unfused path for that output)
 *   workspace  smplpp_forward_workspace_bytes(B) bytes of device scratch owned by the caller
 * ------------------------------------------------------------------------------------------------------- */
size_t smplpp_forward_workspace_bytes(const smplpp_model_t * model, int64_t batch);

int smplpp_forward(const smplpp_model_t * model, void * stream, int64_t batch, const float * beta_dev,
                   int64_t beta_stride, const float * theta_dev, float * vertices_dev, float * joints_dev,
                   float * transforms_dev, float * rest_shape_dev, void * workspace_dev, size_t workspace_bytes);

/* Same call with HOST buffers: copies in, runs, copies out, synchronises.  This is the call a user of
 * smplpp::SMPL::launch + getVertex + getRestJoint makes (node/node.cpp:777, 1114-1117); bench.py's `e2e` times it.
 * The batch is processed in chunks on a compute stream while a copy stream drains the previous chunk, so the
 * device->host link (82 680 B per mesh) is the only thing the call waits for.  Page-locked buffers (from
 * smplpp_host_alloc / smplpp_host_register, or any cudaHostAlloc memory) are DMA targets themselves; pageable
 * buffers are staged through pinned chunk buffers and copied by host threads (SMPLPP_HOST_THREADS, default
 * cores/2) while the next chunk is in flight.  SMPLPP_HOST_CHUNK sets the frames per chunk (default 256).
 * Not re-entrant per model handle (the reference's SMPL object is not thread-safe either, SMPL.h:210-270). */
int smplpp_forward_host(const smplpp_model_t * model, int64_t batch, const float * beta_host, int64_t beta_stride,
                        const float * theta_host, float * vertices_host, float * joints_host);

/* Page-locked host memory for the host-buffer calls (the counterpart of torch's pinned tensors a libtorch caller
 * of the reference would use for `.to(device, non_blocking)` / `.cpu()`). */
int smplpp_host_alloc(void ** out, size_t bytes);
void smplpp_host_free(void * ptr);
int smplpp_host_register(void * ptr, size_t bytes);
int smplpp_host_unregister(void * ptr);

/* TEST / TUNING switch, process-wide (atomic; it affects the calls issued after it, on every handle): production code
 * never needs it - every default is "auto".  The parity tests use it to run one input through every implementation.
 *   0 1 3 6   smplpp_forward: 0 = auto, 1 = FFMA fused blend+skinning, 3 = unfused (blend GEMM -> rest shape ->
 *             standalone skinning), 6 = tcgen05 3xFP16 blend + skinning matrices on the tensor cores, persistent and
 *             pipelined (the default when available: a CC 10.x device and an even vertex count >= 128).
 *   200..202  standalone skinning: FFMA TMA pipeline / FFMA register kernel / tcgen05 (default)
 *   300 / 301 VPoser decoder Jacobian: tcgen05 (default) / FFMA
 *   400..402  IK step: auto (two kernels for shared attachments, fused kernel for per-frame ones) / two kernels / fused
 *   410 / 411 normal equations + solve of the two-kernel path: fp64 tensor cores (ik_solve_mma_kernel, default where the
 *             problem shape allows) / scalar ik_solve_kernel
 *   420..422  pose-blend columns of the IK Jacobian and rest shape of the task vertices: tcgen05 (ik_poseblend_tc_kernel,
 *             ik_restshape_tc_kernel; default) / FFMA phase of ik_jacobian_kernel + FFMA blend kernel / tcgen05 columns on
 *             the FFMA rest shape */
int smplpp_set_forward_variant(int variant);

/* ---------------------------------------------------------------------------------------------------------
 * The four pipeline modules on caller-supplied tensors (any V), mirroring the setter/compute/getter triples
 * of BlendShape.h:221-244, JointRegression.h:194-204, WorldTransformation.h:174-191,
 * LinearBlendSkinning.h:175-198.  All pointers are device pointers.
 * ------------------------------------------------------------------------------------------------------- */
/* BlendShape::blend (src/BlendShape.cpp:620-647): theta (B,24,3) axis-angle */
int smplpp_blend_shape(void * stream, int64_t batch, int64_t vertex_num, const float * beta, const float * theta,
                       const float * shape_basis, const float * pose_basis, float * shape_blend_shape,
                       float * pose_blend_shape, float * pose_rotation);
/* JointRegression::regress (src/JointRegression.cpp:507-598) */
int smplpp_joint_regression(void * stream, int64_t batch, int64_t vertex_num, const float * templ,
                            const float * joint_regressor, const float * shape_blend_shape,
                            const float * pose_blend_shape, float * rest_shape, float * joints);
/* WorldTransformation::transform (src/WorldTransformation.cpp:421-468); kinematic_tree (2,24) int64 on device */
int smplpp_world_transformation(void * stream, int64_t batch, const int64_t * kinematic_tree, const float * joints,
                                const float * pose_rotation, float * transforms);
/* LinearBlendSkinning::skinning (src/LinearBlendSkinning.cpp:445-483); root_pos (B,3) nullable.
 * weights (V,24) dense.  This is the standalone HBM-bound skinning kernel (roofline row of SURVEY §8d). */
int smplpp_linear_blend_skinning(void * stream, int64_t batch, int64_t vertex_num, const float * weights,
                                 const float * rest_shape, const float * transforms, const float * root_pos,
                                 float * vertices);
/* Same kernel driven from a model handle (pre-packed sparse weights): rest_shape (B,V,3), transforms (B,24,4,4) */
int smplpp_model_skinning(const smplpp_model_t * model, void * stream, int64_t batch, const float * rest_shape,
                          const float * transforms, const float * root_pos, float * vertices);
/* Same with affine 3x4 transforms [R | t] (B,24,3,4): the bottom row (0,0,0,1) of the reference's 4x4 is implied,
 * the homogeneous divide uses sum_j W[v,j].  This is the layout the fused pipeline keeps internally. */
int smplpp_model_skinning34(const smplpp_model_t * model, void * stream, int64_t batch, const float * rest_shape,
                            const float * transforms34, const float * root_pos, float * vertices);

/* ---------------------------------------------------------------------------------------------------------
 * Normals (replaces SMPL::calcNormal / calcVertexNormal, src/SMPL.cpp:518-535) — batched over frames.
 *   face_normals   (B, n_faces, 3)  for the listed 0-based face rows
 *   vertex_normals (B, n_verts, 3)  for the listed 0-based vertex ids
 * ------------------------------------------------------------------------------------------------------- */
int smplpp_normals(const smplpp_model_t * model, void * stream, int64_t batch, const float * vertices_dev,
                   int64_t n_faces, const int64_t * face_idx_dev, float * face_normals_dev, int64_t n_verts,
                   const int64_t * vert_idx_dev, float * vertex_normals_dev);

/* ---------------------------------------------------------------------------------------------------------
 * VPoser decoder (replaces VPoserDecoderImpl, src/VPoser.cpp:143-238)
 * ------------------------------------------------------------------------------------------------------- */
typedef struct smplpp_vposer_desc
{
  const float * w0; /* decoder_net.0.weight (512, 32)  */
  const float * b0; /* decoder_net.0.bias   (512)      */
  const float * w3; /* decoder_net.3.weight (512, 512) */
  const float * b3; /* decoder_net.3.bias   (512)      */
  const float * w5; /* decoder_net.5.weight (126, 512) */
  const float * b5; /* decoder_net.5.bias   (126)      */
} smplpp_vposer_desc;

int smplpp_vposer_create(const smplpp_vposer_desc * desc_host, smplpp_vposer_t ** out);
void smplpp_vposer_destroy(smplpp_vposer_t * vposer);
/* VPoserDecoderImpl::forward (VPoser.cpp:163-167): latent (B,32) -> axis_angle (B,21,3);
 * jacobian (B,63,32) = d axis_angle / d latent (nullable; what autograd yields in the reference). */
int smplpp_vposer_decode(const smplpp_vposer_t * vposer, void * stream, int64_t batch, const float * latent_dev,
                         float * axis_angle_dev, float * jacobian_dev);
/* convertRotMatToAxisAngle (VPoser.cpp:25-120): (n,3,3) -> (n,3) */
int smplpp_rotmat_to_axis_angle(void * stream, int64_t n, const float * rotmat_dev, float * axis_angle_dev);

/* ---------------------------------------------------------------------------------------------------------
 * IK tasks (replaces smplpp::IkTask, include/smplpp/IkTask.h:13-85, src/IkTask.cpp, and
 * calcTriangleVertexWeights, include/smplpp/toolbox/GeometryUtils.h:42-52)
 *
 * A task set fixes the attachment faces of n markers (IkTask::faceIdx_, 0-based rows of face_indices);
 * create() gathers the 1-ring topology needed by calcActualNormal and packs the blend-shape rows of those
 * vertices so that the IK kernels never touch the full 17 MB pose basis.
 * Per-frame task state lives in caller-owned device arrays (see smplpp_ik_step).
 * ------------------------------------------------------------------------------------------------------- */
int smplpp_tasks_create(const smplpp_model_t * model, int32_t n_tasks, const int64_t * face_idx_host,
                        smplpp_tasks_t ** out);
void smplpp_tasks_destroy(smplpp_tasks_t * tasks);
int32_t smplpp_tasks_count(const smplpp_tasks_t * tasks);
/* number of distinct mesh vertices the task set depends on (face corners + their 1-rings) */
int32_t smplpp_tasks_vertex_count(const smplpp_tasks_t * tasks);

/* SMPL::getRestShape (src/SMPL.cpp:446-461, JointRegression.cpp:557) restricted to the vertices the task set depends on:
 * rest_out (B, n_vertices, 3) device, vertex_ids (n_vertices) host (nullable): the model vertex of every row.  This is the
 * product the IK step runs per iteration; variant 0 = tcgen05 where available, 1 = FFMA kernel. */
int smplpp_tasks_rest_shape(const smplpp_model_t * model, const smplpp_tasks_t * tasks, void * stream, int64_t batch,
                            const float * beta_dev, int64_t beta_stride, const float * theta_dev, float * rest_out_dev,
                            int32_t * vertex_ids, int32_t variant);

/* calcTriangleVertexWeights on n (pos (n,3), triangle (n,3,3)) pairs -> weights (n,3) */
int smplpp_triangle_vertex_weights(void * stream, int64_t n, const float * pos_dev, const float * triangles_dev,
                                   float * weights_dev);

typedef struct smplpp_ik_options
{
  int32_t enable_vposer;   /* node.cpp:316-322: state = [trans 3 | root 3 | latent 32 | hands 6] (44) else 75 */
  int32_t optimize_beta;   /* node.cpp:652-656: per-frame beta columns (10) with |dbeta| <= delta_beta_limit */
  int32_t enable_qp;       /* node.cpp:907: box-QP (phi / beta bounds); 0 = plain LLT (node.cpp:933-938) */
  int32_t enable_phi;      /* 1: tasks with phi_limit > 0 get their 2 phi columns (node.cpp:716-733) */
  int32_t skip_if_too_few; /* node.cpp:785: skip frames with fewer than n/2 valid markers (motion mode) */
  int32_t update_state;    /* apply node.cpp:946-968 to theta / beta */
  float normal_offset;     /* IkTask::normalOffset_ (0.015 in mocap modes, node.cpp:560) */
  float normal_task_weight;/* IkTask::normalTaskWeight_ (0 in mocap modes, node.cpp:558) */
  float phi_limit;         /* IkTask::phiLimit_ (node.cpp:695-700) */
  float delta_theta_reg;   /* 1e-3 node.cpp:887 */
  float delta_phi_reg;     /* 1e-1 node.cpp:888 */
  float delta_beta_reg;    /* 1e-3 node.cpp:889 */
  float delta_beta_limit;  /* 0.5  node.cpp:925 */
  float vposer_latent_reg; /* 1e-5 node.cpp:897 */
  float vposer_hand_reg;   /* 1e3  node.cpp:900 */
  int32_t reserved[3];
} smplpp_ik_options;

void smplpp_ik_options_default(smplpp_ik_options * opt); /* the constants of node/node.cpp cited above */

/* state dimension helpers: theta_dim = 75 or 44; dim = theta_dim + 2 n (phi) + (optimize_beta ? 10 : 0) */
int32_t smplpp_ik_theta_dim(const smplpp_ik_options * opt);
int32_t smplpp_ik_dim(const smplpp_ik_options * opt, int32_t n_tasks);

/* IkTask::calcActualPos / calcActualNormal batched (src/IkTask.cpp:59-86) on an existing vertex buffer:
 *   vertices (B,V,3), vertex_weights (B,n,3) -> positions (B,n,3) [+ normal_offset * normal], normals (B,n,3) */
int smplpp_task_positions(const smplpp_model_t * model, const smplpp_tasks_t * tasks, void * stream, int64_t batch,
                          const float * vertices_dev, const float * vertex_weights_dev, float normal_offset,
                          float * positions_dev, float * normals_dev);

/* Markers-only forward pass: SMPL::launch followed by IkTask::calcActualPos / calcActualNormal of every task
 * (src/SMPL.cpp:671-737, src/IkTask.cpp:59-86) WITHOUT the full mesh.  Only the rest rows, posed rows and 1-ring normals
 * of the vertices the task set depends on are computed (the face corners alone when normal_offset <= 0 and normals are
 * not requested).
 *   beta            (B, 10) with beta_stride >= 10, or (10) shared with beta_stride = 0
 *   theta           (B, 25, 3): row 0 = root translation (as in smplpp_forward)
 *   vertex_weights  (n, 3) shared with vertex_weights_stride = 0 (the MocapBody.yaml case), or (B, n, 3) with stride 3n
 *   positions       (B, n, 3) out: calcActualPos (+ normal_offset * normal when normal_offset > 0)
 *   normals         (B, n, 3) out, nullable: calcActualNormal
 *   workspace       smplpp_task_forward_workspace_bytes(tasks, batch) bytes of device scratch */
size_t smplpp_task_forward_workspace_bytes(const smplpp_tasks_t * tasks, int64_t batch);
int smplpp_task_forward(const smplpp_model_t * model, const smplpp_tasks_t * tasks, void * stream, int64_t batch,
                        const float * beta_dev, int64_t beta_stride, const float * theta_dev,
                        const float * vertex_weights_dev, int64_t vertex_weights_stride, float normal_offset,
                        float * positions_dev, float * normals_dev, void * workspace_dev, size_t workspace_bytes);
/* The same with HOST arrays (pageable or page-locked), as a chunked pipeline: the upload of chunk c+1, the compute of
 * chunk c and the download of chunk c-1 overlap on three internal streams; synchronises before returning.
 * SMPLPP_TASK_CHUNK sets the frames per chunk (default 16384).  Not re-entrant per task-set handle. */
int smplpp_task_forward_host(const smplpp_model_t * model, smplpp_tasks_t * tasks, int64_t batch,
                             const float * beta_host, int64_t beta_stride, const float * theta_host,
                             const float * vertex_weights_host, int64_t vertex_weights_stride, float normal_offset,
                             float * positions_host, float * normals_host);

/* Projection of the task points onto the posed mesh and the re-seated attachment (replaces the
 * igl::point_mesh_squared_distance call and the faceIdx_ / calcVertexWeights update of node/node.cpp:970-1001):
 *   vertices        (B, V, 3)   posed mesh of every frame (smplpp_forward)
 *   points          (B, n, 3)   actualPos + tangents * phi of every task (node.cpp:957-959); n <= 512
 *   face_idx        (B, n)      out: closest face, 0-BASED like igl's closestFaceIndices (ties: lowest face index)
 *   closest         (B, n, 3)   out (optional): closest point on that face
 *   sq_dist         (B, n)      out (optional): squared distance
 *   vertex_weights  (B, n, 3)   out (optional): calcTriangleVertexWeights(closest, face) (GeometryUtils.h:42-52)
 * All pointers are device pointers. */
int smplpp_closest_points(const smplpp_model_t * model, void * stream, int64_t batch, int64_t n_points,
                          const float * vertices_dev, const float * points_dev, int32_t * face_idx_dev,
                          float * closest_dev, float * sq_dist_dev, float * vertex_weights_dev);

/* Sweep grid of ONE posed mesh (replaces node/node.cpp:1023-1073 and toolbox/GridUtils.hpp:28-63; igl::winding_number is
 * un-vendored: generalized winding number = sum of the signed solid angles of the faces / 4 pi):
 *   smplpp_sweep_grid_bounds   vertices (V, 3) device -> grid_idx_min[3] = getGridIdxFloor(min corner),
 *                              grid_num[3] = getGridIdxCeil(max corner) - grid_idx_min + 1   (host arrays; synchronises)
 *   smplpp_sweep_grid_winding  winding number (optional) and occupancy (optional, 1 where winding > 0.5, node.cpp:1056) of
 *                              the grid points 0.025 * (grid_idx_min + (ix, iy, iz)), ix outermost / iz innermost like the
 *                              reference's loop (node.cpp:1038-1048); both outputs hold grid_num[0]*[1]*[2] entries (device) */
int smplpp_sweep_grid_bounds(const smplpp_model_t * model, void * stream, const float * vertices_dev, int32_t * grid_idx_min,
                             int32_t * grid_num);
int smplpp_sweep_grid_winding(const smplpp_model_t * model, void * stream, const float * vertices_dev,
                              const int32_t * grid_idx_min, const int32_t * grid_num, float * winding_dev,
                              uint8_t * occupied_dev);

/* One IK iteration for B independent frames (replaces node/node.cpp:753-968 per frame):
 *   theta assembly (+VPoser) -> sparse forward on the task vertices -> tangents + re-weighting (:803-804) ->
 *   residual e (:807-820) -> analytic Jacobian J (what the one-hot backward rows of :823-873 yield) ->
 *   A = J'J + damping (+ prior), b = J'e in fp64 (:884-904) -> Cholesky / box-QP (:907-939) -> update (:946-968).
 *
 *   theta_state     (B, theta_dim)  in/out   g_theta
 *   beta            (B, 10) stride beta_stride (0 = shared, read-only unless optimize_beta)   g_beta
 *   vertex_weights  (B, n, 3)       in/out   IkTask::vertexWeights_
 *   target_pos      (B, n, 3)                IkTask::targetPos_
 *   target_normal   (B, n, 3)       nullable (default (0,0,1), IkTask.cpp:13-16)
 *   pos_task_weight (B, n)          nullable (default 1; 0 marks a missing marker, node.cpp:682-683)
 *   status          (B) int32       out: 0 ok, 1 skipped (too few markers), 2 numerical issue (LLT pivot <= 0
 *                                        or non-finite residual), 3 QP iteration cap
 *   e_out (B,4n) f32, jac_out (B,4n,dim) f32, a_out (B,dim,dim) f64, b_out (B,dim) f64, delta_out (B,dim) f64:
 *   optional materialised intermediates (the "Jacobian getter" path; nullable)
 *   workspace: smplpp_ik_workspace_bytes(...) bytes of device scratch
 */
size_t smplpp_ik_workspace_bytes(const smplpp_tasks_t * tasks, const smplpp_ik_options * opt, int64_t batch);

int smplpp_ik_step(const smplpp_model_t * model, const smplpp_vposer_t * vposer, const smplpp_tasks_t * tasks,
                   const smplpp_ik_options * opt, void * stream, int64_t batch, float * theta_state_dev,
                   float * beta_dev, int64_t beta_stride, float * vertex_weights_dev, const float * target_pos_dev,
                   const float * target_normal_dev, const float * pos_task_weight_dev, int32_t * status_dev,
                   float * e_out_dev, float * jac_out_dev, double * a_out_dev, double * b_out_dev,
                   double * delta_out_dev, void * workspace_dev, size_t workspace_bytes);

/* The linearisation of that step alone -- the "Jacobian getter" SURVEY 8(b) asks for, because the reference has none
 * (callers run Tensor::backward once per residual row and read .grad(), node/node.cpp:823-873): theta assembly (+VPoser),
 * sparse forward, tangents + re-weighting (vertex_weights is updated in place exactly as the step does, node.cpp:803-804),
 * residual and Jacobian.  theta_state / beta are read only; no normal equations, no solve, no update.
 *   e_out (B,4n) f32 and / or jac_out (B,4n,dim) f32 in the layout of smplpp_ik_step; workspace as for smplpp_ik_step. */
int smplpp_ik_jacobian(const smplpp_model_t * model, const smplpp_vposer_t * vposer, const smplpp_tasks_t * tasks,
                       const smplpp_ik_options * opt, void * stream, int64_t batch, const float * theta_state_dev,
                       const float * beta_dev, int64_t beta_stride, float * vertex_weights_dev, const float * target_pos_dev,
                       const float * target_normal_dev, const float * pos_task_weight_dev, float * e_out_dev,
                       float * jac_out_dev, void * workspace_dev, size_t workspace_bytes);

/* The same step with PER-FRAME attachments: face_idx_dev (B, n) int32 holds IkTask::faceIdx_ of every (frame, task) as
 * re-seated by the projection of node/node.cpp:993-1001 (smplpp_ik_reproject); the 1-ring topology of every attachment is
 * gathered on the device.  dphi_out_dev (B, n, 2), nullable: the phi part of the step (node.cpp:955-958), which
 * smplpp_ik_reproject consumes.  Workspace: smplpp_ik_faces_workspace_bytes. */
size_t smplpp_ik_faces_workspace_bytes(const smplpp_tasks_t * tasks, const smplpp_ik_options * opt, int64_t batch);
int smplpp_ik_step_faces(const smplpp_model_t * model, const smplpp_vposer_t * vposer, const smplpp_tasks_t * tasks,
                         const smplpp_ik_options * opt, void * stream, int64_t batch, float * theta_state_dev,
                         float * beta_dev, int64_t beta_stride, float * vertex_weights_dev, const int32_t * face_idx_dev,
                         const float * target_pos_dev, const float * target_normal_dev, const float * pos_task_weight_dev,
                         int32_t * status_dev, float * e_out_dev, float * jac_out_dev, double * a_out_dev,
                         double * b_out_dev, double * delta_out_dev, float * dphi_out_dev, void * workspace_dev,
                         size_t workspace_bytes);

/* The tail of the reference's iteration (node/node.cpp:949-1001) for B frames: on the mesh of the given state -- the node
 * uses the PRE-update theta / beta of the iteration, i.e. the state the step linearised at -- every task point
 * p = calcActualPos() + tangents * dphi (IkTask.cpp:33-47, 59-72) is projected onto the mesh
 * (igl::point_mesh_squared_distance there) and the attachment is re-seated in place:
 *   face_idx_dev       (B, n) int32  in: IkTask::faceIdx_ per frame  out: the closest face
 *   vertex_weights_dev (B, n, 3)     in: the weights the step left   out: calcTriangleVertexWeights(closest point, face)
 *   dphi_dev           (B, n, 2)     nullable: the phi part of the step (smplpp_ik_step_faces)
 *   sq_dist_dev        (B, n)        nullable out: squared distance of the point to the mesh */
size_t smplpp_ik_reproject_workspace_bytes(const smplpp_model_t * model, const smplpp_tasks_t * tasks, int64_t batch);
int smplpp_ik_reproject(const smplpp_model_t * model, const smplpp_vposer_t * vposer, const smplpp_tasks_t * tasks,
                        const smplpp_ik_options * opt, void * stream, int64_t batch, const float * theta_state_dev,
                        const float * beta_dev, int64_t beta_stride, float * vertex_weights_dev, int32_t * face_idx_dev,
                        const float * dphi_dev, float * sq_dist_dev, void * workspace_dev, size_t workspace_bytes);

/* `iterations` IK steps for B frames with HOST arrays (the mocap modes of node/node.cpp:645-1002 as one call: targets of
 * every frame in, theta / re-weighted attachments / status out).  Copies in, iterates smplpp_ik_step on an internal
 * stream, copies out, synchronises; bench.py's `ik.e2e` times this call.  Arrays as in smplpp_ik_step;
 * beta_host is written back only with optimize_beta; residual_host (B, nullable) receives the mean over the valid
 * markers of |e_m| at the last linearisation point (metres).  Not re-entrant per task-set handle. */
int smplpp_ik_solve_host(const smplpp_model_t * model, const smplpp_vposer_t * vposer, smplpp_tasks_t * tasks,
                         const smplpp_ik_options * opt, int64_t batch, int32_t iterations, float * theta_state_host,
                         float * beta_host, int64_t beta_stride, float * vertex_weights_host,
                         const float * target_pos_host, const float * pos_task_weight_host, int32_t * status_host,
                         float * residual_host);

/* IkTask::calcTangents (src/IkTask.cpp:33-47) batched: vertices (B,V,3) -> tangents (B,n,3,2) like IkTask::tangents_
 * (column 0 = normalize(v1 - v0), column 1 = normalize(normal x (v1 - v0))); face_idx_dev (B,n) int32 nullable = the
 * faces of the task set */
int smplpp_task_tangents(const smplpp_model_t * model, const smplpp_tasks_t * tasks, void * stream, int64_t batch,
                         const float * vertices_dev, const int32_t * face_idx_dev, float * tangents_dev);

/* Shared-beta stage (MoSh++ shape estimation over many frames; SURVEY §8e).  Frames couple only through the
 * 10 shape unknowns, so the step is split around ONE all-reduce of 111 doubles:
 *   (1) smplpp_ik_shared_beta_reduce: per-frame normal equations with the beta columns, Schur complement
 *       S_f = A_bb - A_bf A_ff^-1 A_fb, r_f = b_b - A_bf A_ff^-1 b_f, summed over the local frames into
 *       reduced_dev = [S (10x10) | r (10) | sum ||e||^2 (1)]  (fp64);
 *   (2) the caller all-reduces reduced_dev over ranks (NCCL sum; nothing to do on one GPU);
 *   (3) smplpp_ik_shared_beta_apply: every rank solves the same 10-dim box QP (|dbeta| <= limit), back-
 *       substitutes x_f = -A_ff^-1 (b_f + A_fb dbeta) and updates theta_state and the shared beta (10).
 * The per-frame factors are kept in `workspace` between (1) and (3). */
size_t smplpp_ik_shared_beta_workspace_bytes(const smplpp_tasks_t * tasks, const smplpp_ik_options * opt,
                                             int64_t batch);
int smplpp_ik_shared_beta_reduce(const smplpp_model_t * model, const smplpp_vposer_t * vposer,
                                 const smplpp_tasks_t * tasks, const smplpp_ik_options * opt, void * stream,
                                 int64_t batch, const float * theta_state_dev, const float * shared_beta_dev,
                                 float * vertex_weights_dev, const float * target_pos_dev,
                                 const float * pos_task_weight_dev, int32_t * status_dev, double * reduced_dev,
                                 void * workspace_dev, size_t workspace_bytes);
int smplpp_ik_shared_beta_apply(const smplpp_tasks_t * tasks, const smplpp_ik_options * opt, void * stream,
                                int64_t batch, float * theta_state_dev, float * shared_beta_dev,
                                const int32_t * status_dev, const double * reduced_dev, void * workspace_dev,
                                size_t workspace_bytes);

/* The three calls above as ONE, with the collective inside (SURVEY 8b: the shared-beta step taking an ncclComm_t):
 * reduce -> ncclAllReduce(sum) of the 111 doubles on `stream` over `nccl_comm` (an ncclComm_t passed as void*; NULL on a
 * single GPU) -> apply.  reduced_dev (111 doubles) is caller-owned scratch that also returns the summed message.  NCCL is
 * resolved at run time (the process's own ncclAllReduce when a framework loaded it, else libnccl.so.2, or the library
 * named by SMPLPP_NCCL_LIB): libsmplpp_b200.so itself links only the CUDA runtime. */
int smplpp_ik_shared_beta_step(const smplpp_model_t * model, const smplpp_vposer_t * vposer, const smplpp_tasks_t * tasks,
                               const smplpp_ik_options * opt, void * stream, int64_t batch, float * theta_state_dev,
                               float * shared_beta_dev, float * vertex_weights_dev, const float * target_pos_dev,
                               const float * pos_task_weight_dev, int32_t * status_dev, double * reduced_dev,
                               void * nccl_comm, void * workspace_dev, size_t workspace_bytes);

/* ---------------------------------------------------------------------------------------------------------
 * The motion stage of the mocap mode as one call (node/node.cpp:509-535 MocapBody.yaml, :571-595 label matching,
 * :667-691 targets, :785 skip rule, :1369-1407 loop, scripts/convertRosbagToText.py motion text).
 * The reference walks the frames serially with ONE iteration per frame, warm-started from the previous frame after 31
 * warm-up iterations on the first frame.  Here all frames are solved at once: `warmup_iterations` on the first frame of
 * the range give the common start (state, attachments), then every frame gets `iterations` steps; with reproject != 0
 * every step is the full loop body (projection onto the pre-update mesh, faces / weights re-seated per frame).
 *   opt                  enable_vposer, regularisation, normal_offset ...; the motion-stage settings (phi pinned, fixed
 *                        beta) are forced as the node does (node.cpp:558-560, 699)
 *   initial_state_host   (theta_dim) g_theta at start (node.cpp:377-410)
 *   first_frame, frame_count  range of C3D frames (frame_count 0 = to the end)
 *   theta75_out_host     (frames, 75)  theta of every frame, VPoser states decoded (node.cpp:1374-1391); nullable
 *   status_out_host      (frames)      0 solved, 1 skipped (fewer than half of the markers), 2 / 3 numerical; nullable
 *   residual_out_host    (frames)      mean |e_m| over the valid markers at the last linearisation point; nullable
 *   motion_text_path     nullable: 75 values per line and frame
 * ------------------------------------------------------------------------------------------------------- */
typedef struct smplpp_mocap_summary
{
  int64_t frames, markers, solved, skipped, failed;
  double mean_residual, max_residual; /* over the solved frames, metres */
} smplpp_mocap_summary;

int smplpp_solve_mocap_motion(const smplpp_model_t * model, const smplpp_vposer_t * vposer, const char * c3d_path,
                              const char * mocap_body_yaml_path, const smplpp_ik_options * opt, int32_t warmup_iterations,
                              int32_t iterations, int32_t reproject, const float * initial_state_host, int64_t first_frame,
                              int64_t frame_count, float * theta75_out_host, int32_t * status_out_host,
                              float * residual_out_host, const char * motion_text_path, smplpp_mocap_summary * summary);

/* ---------------------------------------------------------------------------------------------------------
 * Device memory for callers that link nothing but this C ABI (the header-only C++ facade has no CUDA headers).
 * smplpp_copy_to_host synchronises `stream`; smplpp_copy_to_device only enqueues (pageable sources are staged by the
 * runtime before it returns).
 * ------------------------------------------------------------------------------------------------------- */
int smplpp_device_alloc(void ** out_dev, size_t bytes);
void smplpp_device_free(void * ptr_dev);
int smplpp_copy_to_device(void * dst_dev, const void * src_host, size_t bytes, void * stream);
int smplpp_copy_to_host(void * dst_host, const void * src_dev, size_t bytes, void * stream);
int smplpp_stream_synchronize(void * stream);

/* ---------------------------------------------------------------------------------------------------------
 * Data formats on either side of the path (host only; SURVEY.md 8f ranks 2-3)
 * ------------------------------------------------------------------------------------------------------- */
/* A parameter file = one JSON object of nested numeric arrays (what nlohmann::json + xt::from_json read in
 * src/SMPL.cpp:566-611 and src/VPoser.cpp:173-237).  shape8 receives up to 8 extents, data points into the handle. */
int smplpp_json_open(const char * path, smplpp_json_t ** out);
void smplpp_json_close(smplpp_json_t * json);
int smplpp_json_array(const smplpp_json_t * json, const char * key, int32_t * ndim, int64_t * shape8,
                      const double ** data);
/* The .npz twin of a parameter file (np.savez of scripts/preprocess.py:98-117: a ZIP of stored .npy members, zip64 extra
 * fields, little-endian f4 / f8 / i4 / i8 / u4 / u8, C order); arrays are read with smplpp_json_array, closed with
 * smplpp_json_close. */
int smplpp_npz_open(const char * path, smplpp_json_t ** out);
int smplpp_model_load_npz(const char * path, smplpp_model_t ** out);
/* SMPL::setModelPath + SMPL::init (src/SMPL.cpp:560-643): keys face_indices, shape_blend_shapes, pose_blend_shapes,
 * vertices_template, joint_regressor, kinematic_tree, weights; the reference's messages ("Cannot initialize a SMPL
 * model!", "Shape parameter dimensions are invalid: 9 != 10", ...) come back through smplpp_last_error(). */
int smplpp_model_load_json(const char * path, smplpp_model_t ** out);
/* VPoserDecoderImpl::loadParamsFromJson (src/VPoser.cpp:169-238): keys decoder_net.{0,3,5}.{weight,bias} */
int smplpp_vposer_load_json(const char * path, smplpp_vposer_t ** out);

/* C3D motion capture file as the node reads it through ezc3d (node/node.cpp:572-595, 667-691) */
int smplpp_c3d_open(const char * path, smplpp_c3d_t ** out);
void smplpp_c3d_close(smplpp_c3d_t * c3d);
int64_t smplpp_c3d_frame_count(const smplpp_c3d_t * c3d);   /* header().nbFrames() */
int64_t smplpp_c3d_point_count(const smplpp_c3d_t * c3d);   /* POINT:USED */
double smplpp_c3d_frame_rate(const smplpp_c3d_t * c3d);     /* header().frameRate() */
const char * smplpp_c3d_label(const smplpp_c3d_t * c3d, int64_t point); /* POINT:LABELS[point] */
const char * smplpp_c3d_units(const smplpp_c3d_t * c3d);    /* POINT:UNITS */
/* index of the first POINT:LABELS value that ends with `name`; the length of that list when there is none
 * (std::find_if + std::distance over valuesAsString(), node.cpp:580-594) */
int64_t smplpp_c3d_find_label(const smplpp_c3d_t * c3d, const char * name);
/* frames [first, first + count) -> xyz_host (count, points, 3), valid_host (count, points): 0 = point.isEmpty(),
 * whose coordinates are returned as 0 (node.cpp:682-683 zeroes the target of a missing marker) */
int smplpp_c3d_read(const smplpp_c3d_t * c3d, int64_t first, int64_t count, float * xyz_host, uint8_t * valid_host);

/* Result files of the mocap modes.
 * MocapBody.yaml: written by the body stage (node/node.cpp:1425-1441: beta, then name / faceIdx / vertexWeights of every
 * IkTask) and loaded by the motion stage (node/node.cpp:509-535). */
int smplpp_write_mocap_body_yaml(const char * path, const float * beta10, int32_t n_tasks, const char * const * names,
                                 const int64_t * face_idx, const float * vertex_weights);
int smplpp_mocap_body_open(const char * path, smplpp_mocap_body_t ** out);
void smplpp_mocap_body_close(smplpp_mocap_body_t * body);
int32_t smplpp_mocap_body_task_count(const smplpp_mocap_body_t * body);
const char * smplpp_mocap_body_task_name(const smplpp_mocap_body_t * body, int32_t task);
int smplpp_mocap_body_get(const smplpp_mocap_body_t * body, float * beta10, int64_t * face_idx, float * vertex_weights);
/* SMPL::out (src/SMPL.cpp:757-790): Wavefront OBJ of one mesh (host arrays; faces 1-based as stored) */
int smplpp_write_obj(const char * path, int64_t n_vertices, const float * vertices_host, int64_t n_faces,
                     const int32_t * face_indices_1based);
/* Motion as text, one frame per line, 75 values of theta (scripts/convertRosbagToText.py:13-19) */
int smplpp_write_motion_text(const char * path, int64_t frames, const float * theta75_host);
int smplpp_read_motion_text(const char * path, int64_t max_frames, float * theta75_host, int64_t * frames_out);

#ifdef __cplusplus
}
#endif
#endif /* SMPLPP_B200_H */
