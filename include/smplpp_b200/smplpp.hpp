// smplpp_b200 — header-only C++ facade over the C ABI (include/smplpp_b200.h) that keeps the class and method names
// of the reference's libsmplpp (include/smplpp/SMPL.h:210-270, IkTask.h:13-85, VPoser.h:33-90,
// toolbox/Exception.h:49) so that a caller such as node/node.cpp keeps its shape once libtorch is removed from the
// path.  torch::Tensor is replaced by plain row-major host arrays (smplpp::Array) for the object-level API; callers
// that keep everything on the device use the C entry points directly.  Errors are rethrown as smplpp::Exception with
// the reference's message text ("<module> Error: <msg>", src/toolbox/Exception.cpp:77-91).
// There is NO CPU fallback: every call fails with "CUDA Error: ..." without a device.
#pragma once

#include <array>
#include <cstdint>
#include <cstdio>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../smplpp_b200.h"

namespace smplpp
{
constexpr int64_t VERTEX_NUM = SMPLPP_VERTEX_NUM;   // definition/def.h:8-14
constexpr int64_t JOINT_NUM = SMPLPP_JOINT_NUM;
constexpr int64_t SHAPE_BASIS_DIM = SMPLPP_SHAPE_DIM;
constexpr int64_t POSE_BASIS_DIM = SMPLPP_POSE_DIM;
constexpr int64_t FACE_INDEX_NUM = SMPLPP_FACE_NUM;
constexpr int64_t LATENT_DIM = SMPLPP_LATENT_DIM;

/// Counterpart of smplpp::Exception (toolbox/Exception.h:122): what() = "<module> Error: <text>".
class Exception : public std::runtime_error
{
public:
  explicit Exception(const std::string & what) : std::runtime_error(what) {}
};

inline void check(int rc)
{
  if(rc != SMPLPP_OK)
  {
    const char * msg = smplpp_last_error();
    throw Exception(msg && *msg ? msg : "SMPL Error: smplpp_b200 call failed");
  }
}

/// Dense row-major float array with a shape (the stand-in for the torch::Tensor values the reference returns).
struct Array
{
  std::vector<int64_t> shape;
  std::vector<float> data;
  Array() = default;
  explicit Array(std::vector<int64_t> s) : shape(std::move(s))
  {
    size_t n = 1;
    for(int64_t d : shape) n *= static_cast<size_t>(d);
    data.assign(n, 0.f);
  }
  int64_t size(size_t dim) const { return shape.at(dim); }
  float * ptr() { return data.data(); }
  const float * ptr() const { return data.data(); }
};

namespace detail
{
/// A device allocation behind the C ABI (the facade has no CUDA headers); grows on demand, freed on destruction.
class DeviceBuffer
{
public:
  DeviceBuffer() = default;
  DeviceBuffer(const DeviceBuffer &) = delete;
  DeviceBuffer & operator=(const DeviceBuffer &) = delete;
  ~DeviceBuffer() { smplpp_device_free(ptr_); }
  void * reserve(size_t bytes)
  {
    if(bytes > bytes_)
    {
      smplpp_device_free(ptr_);
      ptr_ = nullptr, bytes_ = 0;
      check(smplpp_device_alloc(&ptr_, bytes));
      bytes_ = bytes;
    }
    return ptr_;
  }
  template<typename T>
  T * upload(const T * host, size_t count)
  {
    reserve(count * sizeof(T));
    check(smplpp_copy_to_device(ptr_, host, count * sizeof(T), nullptr));
    return static_cast<T *>(ptr_);
  }
  float * upload(const Array & a) { return upload(a.ptr(), a.data.size()); }
  template<typename T>
  T * as() const
  {
    return static_cast<T *>(ptr_);
  }
  size_t bytes() const { return bytes_; }

private:
  void * ptr_ = nullptr;
  size_t bytes_ = 0;
};

inline Array download(const float * dev, std::vector<int64_t> shape)
{
  Array a(std::move(shape));
  if(!a.data.empty()) check(smplpp_copy_to_host(a.ptr(), dev, a.data.size() * sizeof(float), nullptr));
  return a;
}
inline void require(bool ok, const char * what)
{
  if(!ok) throw Exception(what);
}
} // namespace detail

/// The tensors of the model file (keys of src/SMPL.cpp:573-611).
struct ModelParams
{
  int64_t vertex_num = VERTEX_NUM;
  std::vector<int32_t> face_indices;      // (F,3) 1-based
  std::vector<float> shape_blend_shapes;  // (V,3,10)
  std::vector<float> pose_blend_shapes;   // (V,3,207)
  std::vector<float> vertices_template;   // (V,3)
  std::vector<float> joint_regressor;     // (24,V)
  std::vector<int64_t> kinematic_tree;    // (2,24)
  std::vector<float> weights;             // (V,24)
};

/// smplpp::SMPL (src/SMPL.cpp): init / launch / getters with host arrays.
class SMPL
{
public:
  SMPL() = default;
  explicit SMPL(const ModelParams & params) { init(params); }
  SMPL(const SMPL &) = delete;
  SMPL & operator=(const SMPL &) = delete;
  ~SMPL()
  {
    if(m__model) smplpp_model_destroy(m__model);
  }

  /// SMPL::setModelPath (SMPL.cpp:325-339) + SMPL::init() (SMPL.cpp:560-643): the model JSON is read by the library
  /// (smplpp_model_load_json); the messages are the reference's.
  void setModelPath(const std::string & modelPath)
  {
    if(FILE * f = fopen(modelPath.c_str(), "rb"))
      fclose(f);
    else
      throw Exception("SMPL Error: Failed to initialize model path!"); // SMPL.cpp:337
    m__modelPath = modelPath;
  }
  void init()
  {
    if(m__model) smplpp_model_destroy(m__model);
    m__model = nullptr;
    // the JSON of scripts/preprocess.py, or its np.savez twin (scripts/preprocess.py:98-117) when the path ends in .npz
    const bool npz = m__modelPath.size() > 4 && m__modelPath.compare(m__modelPath.size() - 4, 4, ".npz") == 0;
    check(npz ? smplpp_model_load_npz(m__modelPath.c_str(), &m__model) : smplpp_model_load_json(m__modelPath.c_str(), &m__model));
    m__vertexNum = smplpp_model_vertex_num(m__model);
    smplpp_json_t * j = nullptr;
    check(npz ? smplpp_npz_open(m__modelPath.c_str(), &j) : smplpp_json_open(m__modelPath.c_str(), &j));
    int32_t ndim = 0;
    int64_t shape[8];
    const double * data = nullptr;
    const int rc = smplpp_json_array(j, "face_indices", &ndim, shape, &data);
    if(rc == SMPLPP_OK && ndim == 2)
    {
      m__faceIndices.resize(static_cast<size_t>(shape[0] * shape[1]));
      for(size_t i = 0; i < m__faceIndices.size(); i++) m__faceIndices[i] = static_cast<int32_t>(data[i]);
    }
    smplpp_json_close(j);
    check(rc);
  }

  /// SMPL::init from already-parsed arrays
  void init(const ModelParams & p)
  {
    const size_t V = static_cast<size_t>(p.vertex_num);
    if(p.shape_blend_shapes.size() != V * 3 * SHAPE_BASIS_DIM)
      throw Exception("SMPL Error: Shape parameter dimensions are invalid!"); // SMPL.cpp:581
    if(p.pose_blend_shapes.size() != V * 3 * POSE_BASIS_DIM)
      throw Exception("SMPL Error: Pose parameter dimensions are invalid!"); // SMPL.cpp:588
    if(p.vertices_template.size() != V * 3 || p.joint_regressor.size() != JOINT_NUM * V
       || p.kinematic_tree.size() != 2 * JOINT_NUM || p.weights.size() != V * JOINT_NUM || p.face_indices.size() % 3)
      throw Exception("SMPL Error: Cannot initialize a SMPL model!"); // SMPL.cpp:616
    smplpp_model_desc d;
    d.vertex_num = p.vertex_num;
    d.face_num = static_cast<int64_t>(p.face_indices.size() / 3);
    d.face_indices = p.face_indices.data();
    d.shape_blend_shapes = p.shape_blend_shapes.data();
    d.pose_blend_shapes = p.pose_blend_shapes.data();
    d.vertices_template = p.vertices_template.data();
    d.joint_regressor = p.joint_regressor.data();
    d.kinematic_tree = p.kinematic_tree.data();
    d.weights = p.weights.data();
    if(m__model) smplpp_model_destroy(m__model);
    m__model = nullptr;
    check(smplpp_model_create(&d, &m__model));
    m__faceIndices = p.face_indices;
    m__vertexNum = p.vertex_num;
  }

  /// SMPL::launch (SMPL.cpp:671-737): beta (N,10) or (1,10) shared, theta (N,25,3) with row 0 = root translation.
  /// Inputs go to the device, the forward pass runs there (smplpp_forward) and the results STAY there: the getters
  /// download what they are asked for, IkTask and the normal getters read the device buffers.
  void launch(const Array & beta, const Array & theta)
  {
    if(!m__model || theta.shape.size() != 3 || theta.shape[1] != JOINT_NUM + 1 || theta.shape[2] != 3)
      throw Exception("SMPL Error: Cannot launch a SMPL model!"); // SMPL.cpp:676
    const int64_t n = theta.shape[0];
    if(beta.shape.size() != 2 || beta.shape[1] != SHAPE_BASIS_DIM || (beta.shape[0] != n && beta.shape[0] != 1))
      throw Exception("BlendShape Error: Failed to set beta!"); // BlendShape.cpp:340
    m__batch = n;
    m__betaStride = (beta.shape[0] == 1 && n > 1) ? 0 : SHAPE_BASIS_DIM;
    m__dBeta.upload(beta);
    m__dTheta.upload(theta);
    m__dVertices.reserve(static_cast<size_t>(n * m__vertexNum * 3) * sizeof(float));
    m__dJoints.reserve(static_cast<size_t>(n * JOINT_NUM * 3) * sizeof(float));
    const size_t ws = smplpp_forward_workspace_bytes(m__model, n);
    m__dWs.reserve(ws);
    check(smplpp_forward(m__model, nullptr, n, m__dBeta.as<float>(), m__betaStride, m__dTheta.as<float>(),
                         m__dVertices.as<float>(), m__dJoints.as<float>(), nullptr, nullptr, m__dWs.as<void>(), ws));
    check(smplpp_stream_synchronize(nullptr));
    m__launched = true;
    m__haveVertices = m__haveJoints = false;
  }
  /// The same through the host-buffer pipeline of the library (chunked, copies overlapped with compute): the fastest
  /// way to get ALL vertices of a large batch back to the host (bench.py's e2e call).
  void launchHost(const Array & beta, const Array & theta)
  {
    if(!m__model || theta.shape.size() != 3 || theta.shape[1] != JOINT_NUM + 1 || theta.shape[2] != 3)
      throw Exception("SMPL Error: Cannot launch a SMPL model!");
    const int64_t n = theta.shape[0];
    if(beta.shape.size() != 2 || beta.shape[1] != SHAPE_BASIS_DIM || (beta.shape[0] != n && beta.shape[0] != 1))
      throw Exception("BlendShape Error: Failed to set beta!");
    launch(slice0(beta), slice0(theta)); // device state for the raw getters: frame 0
    m__vertices = Array({n, m__vertexNum, 3});
    m__joints = Array({n, JOINT_NUM, 3});
    const int64_t stride = (beta.shape[0] == 1 && n > 1) ? 0 : SHAPE_BASIS_DIM;
    check(smplpp_forward_host(m__model, n, beta.ptr(), stride, theta.ptr(), m__vertices.ptr(), m__joints.ptr()));
    m__haveVertices = m__haveJoints = true;
  }

  /// SMPL::getVertex (SMPL.cpp:446-461): (N,V,3)
  const Array & getVertex()
  {
    if(!m__launched) throw Exception("LinearBlendSknning Error: Failed to get vertices of new pose!"); // LinearBlendSkinning.cpp:409
    if(!m__haveVertices)
    {
      m__vertices = detail::download(m__dVertices.as<float>(), {m__batch, m__vertexNum, 3});
      m__haveVertices = true;
    }
    return m__vertices;
  }
  /// SMPL::getRestJoint (SMPL.cpp:425-440): (N,24,3)
  const Array & getRestJoint()
  {
    if(!m__launched) throw Exception("JointRegression Error: Failed to get joints!");
    if(!m__haveJoints)
    {
      m__joints = detail::download(m__dJoints.as<float>(), {m__batch, JOINT_NUM, 3});
      m__haveJoints = true;
    }
    return m__joints;
  }
  /// SMPL::getRestShape (SMPL.cpp:386-405 -> JointRegression::getRestShape): (N,V,3) = template + shape + pose blend
  Array getRestShape()
  {
    if(!m__launched) throw Exception("JointRegression Error: Failed to get deformed shape in rest pose!");
    detail::DeviceBuffer rest;
    rest.reserve(static_cast<size_t>(m__batch * m__vertexNum * 3) * sizeof(float));
    check(smplpp_forward(m__model, nullptr, m__batch, m__dBeta.as<float>(), m__betaStride, m__dTheta.as<float>(), nullptr,
                         nullptr, nullptr, rest.as<float>(), m__dWs.as<void>(), m__dWs.bytes()));
    return detail::download(rest.as<float>(), {m__batch, m__vertexNum, 3});
  }
  /// SMPL::getVertexRaw (LinearBlendSkinning.cpp:419-427): vertices `idx` (0-based) of batch element 0
  Array getVertexRaw(const std::vector<int64_t> & idx)
  {
    if(!m__launched) throw Exception("LinearBlendSknning Error: Failed to get vertices of new pose!");
    Array out({static_cast<int64_t>(idx.size()), 3});
    for(size_t i = 0; i < idx.size(); i++)
    {
      detail::require(idx[i] >= 0 && idx[i] < m__vertexNum, "LinearBlendSknning Error: Failed to get vertices of new pose!");
      check(smplpp_copy_to_host(out.ptr() + 3 * i, m__dVertices.as<float>() + 3 * idx[i], 3 * sizeof(float), nullptr));
    }
    return out;
  }
  Array getVertexRaw(int64_t idx) { return getVertexRaw(std::vector<int64_t>{idx}); }
  /// SMPL::getFaceIndexRaw (SMPL.cpp:407-423): the three 1-BASED vertex ids of face `idx`
  std::array<int32_t, 3> getFaceIndexRaw(int64_t idx) const
  {
    detail::require(idx >= 0 && static_cast<size_t>(3 * idx + 2) < m__faceIndices.size(), "SMPL Error: Failed to get face indices!");
    return {m__faceIndices[3 * idx], m__faceIndices[3 * idx + 1], m__faceIndices[3 * idx + 2]};
  }
  /// SMPL::calcNormal (SMPL.cpp:518-525): unit normal of face `faceIdx` on batch element 0
  Array calcNormal(int64_t faceIdx) { return normals(&faceIdx, nullptr); }
  /// SMPL::calcVertexNormal (SMPL.cpp:527-535): normalised mean of the adjacent face normals
  Array calcVertexNormal(int64_t idx) { return normals(nullptr, &idx); }
  /// m__adjacentFacesList (SMPL.cpp:619-640): adjacent face (0-based row of face_indices) -> weight 1 / degree
  std::map<int32_t, float> getAdjacentFaces(int64_t vertexIdx) const
  {
    std::map<int32_t, float> out;
    for(size_t f = 0; f < m__faceIndices.size() / 3; f++)
      for(int k = 0; k < 3; k++)
        if(m__faceIndices[3 * f + k] - 1 == vertexIdx) out[static_cast<int32_t>(f)] = 0.f;
    for(auto & kv : out) kv.second = 1.f / static_cast<float>(out.size());
    return out;
  }
  /// device state of the last launch (for IkTask and callers of the device-pointer C entries)
  const float * deviceVertices() const { return m__dVertices.as<float>(); }
  int64_t batch() const { return m__batch; }
  /// SMPL::setVertPath + SMPL::out (SMPL.cpp:341-355, 757-790): mesh `index` of the batch as Wavefront OBJ
  void setVertPath(const std::string & vertexPath) { m__vertPath = vertexPath; }
  void out(int64_t index)
  {
    if(!m__launched || index < 0 || index >= m__batch || m__vertPath.empty())
      throw Exception("SMPL Error: Cannot export the deformed mesh!"); // SMPL.cpp:785
    getVertex();
    check(smplpp_write_obj(m__vertPath.c_str(), m__vertexNum, m__vertices.ptr() + index * m__vertexNum * 3,
                           static_cast<int64_t>(m__faceIndices.size() / 3), m__faceIndices.data()));
  }
  /// SMPL::getFaceIndex (SMPL.cpp:386-405): (F,3), 1-based like the stored tensor
  const std::vector<int32_t> & getFaceIndex() const { return m__faceIndices; }
  int64_t getVertexNum() const { return m__vertexNum; }
  /// the C handle, for device-pointer calls (smplpp_forward, smplpp_ik_step, ...)
  smplpp_model_t * handle() const { return m__model; }

private:
  static Array slice0(const Array & a)
  {
    std::vector<int64_t> shp = a.shape;
    shp[0] = 1;
    Array o(shp);
    std::copy(a.data.begin(), a.data.begin() + static_cast<std::ptrdiff_t>(o.data.size()), o.data.begin());
    return o;
  }
  Array normals(const int64_t * faceIdx, const int64_t * vertIdx)
  {
    if(!m__launched) throw Exception("LinearBlendSknning Error: Failed to get vertices of new pose!");
    detail::DeviceBuffer idx, out;
    const int64_t id = faceIdx ? *faceIdx : *vertIdx;
    detail::require(id >= 0 && id < (faceIdx ? static_cast<int64_t>(m__faceIndices.size() / 3) : m__vertexNum),
                    "SMPL Error: Failed to get face indices!");
    idx.upload(&id, 1);
    out.reserve(3 * sizeof(float));
    check(smplpp_normals(m__model, nullptr, 1, m__dVertices.as<float>(), faceIdx ? 1 : 0, faceIdx ? idx.as<int64_t>() : nullptr,
                         faceIdx ? out.as<float>() : nullptr, vertIdx ? 1 : 0, vertIdx ? idx.as<int64_t>() : nullptr,
                         vertIdx ? out.as<float>() : nullptr));
    return detail::download(out.as<float>(), {3});
  }
  smplpp_model_t * m__model = nullptr;
  std::string m__modelPath, m__vertPath;
  std::vector<int32_t> m__faceIndices;
  int64_t m__vertexNum = 0, m__batch = 0, m__betaStride = SHAPE_BASIS_DIM;
  Array m__vertices, m__joints;
  detail::DeviceBuffer m__dBeta, m__dTheta, m__dVertices, m__dJoints, m__dWs;
  bool m__launched = false, m__haveVertices = false, m__haveJoints = false;
};

/// smplpp::VPoserDecoder (src/VPoser.cpp:143-238): the six decoder_net tensors, row-major (out, in).
class VPoserDecoder
{
public:
  VPoserDecoder(const std::vector<float> & w0, const std::vector<float> & b0, const std::vector<float> & w3,
                const std::vector<float> & b3, const std::vector<float> & w5, const std::vector<float> & b5)
  {
    if(w0.size() != 512 * 32 || b0.size() != 512 || w3.size() != 512 * 512 || b3.size() != 512 || w5.size() != 126 * 512
       || b5.size() != 126)
      throw Exception("VPoser Error: invalid dimension of decoder parameters!"); // VPoser.cpp:190
    smplpp_vposer_desc d{w0.data(), b0.data(), w3.data(), b3.data(), w5.data(), b5.data()};
    check(smplpp_vposer_create(&d, &vposer_));
  }
  /// VPoserDecoderImpl::loadParamsFromJson (VPoser.cpp:169-238)
  VPoserDecoder() = default;
  void loadParamsFromJson(const std::string & jsonPath)
  {
    if(vposer_) smplpp_vposer_destroy(vposer_);
    vposer_ = nullptr;
    check(smplpp_vposer_load_json(jsonPath.c_str(), &vposer_));
  }
  VPoserDecoder(const VPoserDecoder &) = delete;
  VPoserDecoder & operator=(const VPoserDecoder &) = delete;
  ~VPoserDecoder()
  {
    if(vposer_) smplpp_vposer_destroy(vposer_);
  }
  /// VPoserDecoderImpl::forward (VPoser.cpp:163-167): latent (B,32) -> axis-angle (B,21,3)
  Array forward(const Array & latent)
  {
    if(!vposer_ || latent.shape.size() != 2 || latent.shape[1] != LATENT_DIM) throw Exception("VPoser Error: invalid latent tensor!");
    const int64_t b = latent.shape[0];
    in_.upload(latent);
    out_.reserve(static_cast<size_t>(b) * 63 * sizeof(float));
    check(smplpp_vposer_decode(vposer_, nullptr, b, in_.as<float>(), out_.as<float>(), nullptr));
    return detail::download(out_.as<float>(), {b, 21, 3});
  }
  /// d(axis-angle) / d(latent) (B,63,32): what the reference obtains from autograd through forward()
  Array jacobian(const Array & latent)
  {
    if(!vposer_ || latent.shape.size() != 2 || latent.shape[1] != LATENT_DIM) throw Exception("VPoser Error: invalid latent tensor!");
    const int64_t b = latent.shape[0];
    in_.upload(latent);
    out_.reserve(static_cast<size_t>(b) * 63 * sizeof(float));
    jac_.reserve(static_cast<size_t>(b) * 63 * 32 * sizeof(float));
    check(smplpp_vposer_decode(vposer_, nullptr, b, in_.as<float>(), out_.as<float>(), jac_.as<float>()));
    return detail::download(jac_.as<float>(), {b, 63, 32});
  }
  /// torch::nn::Module::eval / to: the kernels implement eval mode (Dropout = identity, VPoser.cpp:150) on the current device
  void eval() {}
  void to(int /*device*/) {}
  smplpp_vposer_t * handle() const { return vposer_; }

private:
  smplpp_vposer_t * vposer_ = nullptr;
  detail::DeviceBuffer in_, out_, jac_;
};

/// smplpp::convertRotMatToAxisAngle (src/VPoser.cpp:25-120): (N,3,3) -> (N,3)
inline Array convertRotMatToAxisAngle(const Array & rotMat)
{
  if(rotMat.shape.size() != 3 || rotMat.shape[1] != 3 || rotMat.shape[2] != 3) throw Exception("VPoser Error: invalid rotation tensor!");
  detail::DeviceBuffer in, out;
  in.upload(rotMat);
  out.reserve(static_cast<size_t>(rotMat.shape[0]) * 3 * sizeof(float));
  check(smplpp_rotmat_to_axis_angle(nullptr, rotMat.shape[0], in.as<float>(), out.as<float>()));
  return detail::download(out.as<float>(), {rotMat.shape[0], 3});
}

/// smplpp::calcTriangleVertexWeights (toolbox/GeometryUtils.h:42-52): pos (3), triangle (3,3) -> weights (3)
inline Array calcTriangleVertexWeights(const Array & pos, const Array & triangle)
{
  if(pos.data.size() != 3 || triangle.data.size() != 9) throw Exception("GeometryUtils Error: invalid triangle tensors!");
  detail::DeviceBuffer p, t, w;
  p.upload(pos);
  t.upload(triangle);
  w.reserve(3 * sizeof(float));
  check(smplpp_triangle_vertex_weights(nullptr, 1, p.as<float>(), t.as<float>(), w.as<float>()));
  return detail::download(w.as<float>(), {3});
}

// ---------------------------------------------------------------------------------------------------------------
// The four pipeline modules with the setter / compute / getter triples of the reference (BlendShape.h:221-244,
// JointRegression.h:183-204, WorldTransformation.h:174-191, LinearBlendSkinning.h:175-195).  Setters copy to the device
// (the reference deep-copies too), the compute call is one C entry, getters download.
// ---------------------------------------------------------------------------------------------------------------
class BlendShape
{
public:
  void setBeta(const Array & beta)
  {
    if(beta.shape.size() != 2 || beta.shape[1] != SHAPE_BASIS_DIM) throw Exception("BlendShape Error: Failed to set beta!"); // BlendShape.cpp:340
    batch_ = beta.shape[0];
    beta_.upload(beta);
  }
  void setTheta(const Array & theta)
  {
    if(theta.shape.size() != 3 || theta.shape[1] != JOINT_NUM || theta.shape[2] != 3)
      throw Exception("BlendShape Error: Failed to set theta!"); // BlendShape.cpp:394
    thetaBatch_ = theta.shape[0];
    theta_.upload(theta);
  }
  void setShapeBlendBasis(const Array & basis)
  {
    if(basis.shape.size() != 3 || basis.shape[1] != 3 || basis.shape[2] != SHAPE_BASIS_DIM)
      throw Exception("BlendShape Error: Failed to set shape blend basis!"); // BlendShape.cpp:367
    vertexNum_ = basis.shape[0];
    shapeBasis_.upload(basis);
  }
  void setPoseBlendBasis(const Array & basis)
  {
    if(basis.shape.size() != 3 || basis.shape[1] != 3 || basis.shape[2] != POSE_BASIS_DIM)
      throw Exception("BlendShape Error: Failed to set pose blend basis!"); // BlendShape.cpp:451
    poseVertexNum_ = basis.shape[0];
    poseBasis_.upload(basis);
  }
  /// BlendShape::blend (BlendShape.cpp:620-647)
  void blend()
  {
    if(batch_ < 1 || batch_ != thetaBatch_ || vertexNum_ < 1 || vertexNum_ != poseVertexNum_)
      throw Exception("BlendShape Error: Cannot blend shapes!");
    const size_t bv = static_cast<size_t>(batch_ * vertexNum_ * 3) * sizeof(float);
    shapeOut_.reserve(bv), poseOut_.reserve(bv), rot_.reserve(static_cast<size_t>(batch_ * JOINT_NUM * 9) * sizeof(float));
    check(smplpp_blend_shape(nullptr, batch_, vertexNum_, beta_.as<float>(), theta_.as<float>(), shapeBasis_.as<float>(),
                             poseBasis_.as<float>(), shapeOut_.as<float>(), poseOut_.as<float>(), rot_.as<float>()));
    done_ = true;
  }
  Array getShapeBlendShape() const { return get(shapeOut_, {batch_, vertexNum_, 3}, "BlendShape Error: Failed to get shape blend shape!"); }
  Array getPoseBlendShape() const { return get(poseOut_, {batch_, vertexNum_, 3}, "BlendShape Error: Failed to get pose blend shape!"); }
  Array getPoseRotation() const { return get(rot_, {batch_, JOINT_NUM, 3, 3}, "BlendShape Error: Failed to get pose rotation!"); }

private:
  Array get(const detail::DeviceBuffer & b, std::vector<int64_t> shape, const char * err) const
  {
    if(!done_) throw Exception(err);
    return detail::download(b.as<float>(), std::move(shape));
  }
  int64_t batch_ = 0, thetaBatch_ = 0, vertexNum_ = 0, poseVertexNum_ = 0;
  bool done_ = false;
  detail::DeviceBuffer beta_, theta_, shapeBasis_, poseBasis_, shapeOut_, poseOut_, rot_;
};

class JointRegression
{
public:
  void setShapeBlendShape(const Array & a) { set(shape_, a, 3, "JointRegression Error: Failed to set shape blend shape!"); }
  void setPoseBlendShape(const Array & a) { set(pose_, a, 3, "JointRegression Error: Failed to set pose blend shape!"); }
  void setTemplateRestShape(const Array & a)
  {
    if(a.shape.size() != 2 || a.shape[1] != 3) throw Exception("JointRegression Error: Failed to set template rest shape!");
    vertexNum_ = a.shape[0];
    templ_.upload(a);
  }
  void setJointRegressor(const Array & a)
  {
    if(a.shape.size() != 2 || a.shape[0] != JOINT_NUM) throw Exception("JointRegression Error: Failed to set joint regressor!");
    jreg_.upload(a);
  }
  /// JointRegression::regress (JointRegression.cpp:507-598)
  void regress()
  {
    if(batch_ < 1 || vertexNum_ < 1) throw Exception("JointRegression Error: Cannot regress joints!");
    rest_.reserve(static_cast<size_t>(batch_ * vertexNum_ * 3) * sizeof(float));
    joints_.reserve(static_cast<size_t>(batch_ * JOINT_NUM * 3) * sizeof(float));
    check(smplpp_joint_regression(nullptr, batch_, vertexNum_, templ_.as<float>(), jreg_.as<float>(), shape_.as<float>(),
                                  pose_.as<float>(), rest_.as<float>(), joints_.as<float>()));
    done_ = true;
  }
  Array getRestShape() const
  {
    if(!done_) throw Exception("JointRegression Error: Failed to get deformed shape in rest pose!");
    return detail::download(rest_.as<float>(), {batch_, vertexNum_, 3});
  }
  Array getJoint() const
  {
    if(!done_) throw Exception("JointRegression Error: Failed to get joints!");
    return detail::download(joints_.as<float>(), {batch_, JOINT_NUM, 3});
  }

private:
  void set(detail::DeviceBuffer & b, const Array & a, int64_t last, const char * err)
  {
    if(a.shape.size() != 3 || a.shape[2] != last) throw Exception(err);
    batch_ = a.shape[0];
    b.upload(a);
  }
  int64_t batch_ = 0, vertexNum_ = 0;
  bool done_ = false;
  detail::DeviceBuffer shape_, pose_, templ_, jreg_, rest_, joints_;
};

class WorldTransformation
{
public:
  void setJoint(const Array & a)
  {
    if(a.shape.size() != 3 || a.shape[1] != JOINT_NUM || a.shape[2] != 3) throw Exception("WorldTransformation Error: Failed to set joints!");
    batch_ = a.shape[0];
    joints_.upload(a);
  }
  void setPoseRotation(const Array & a)
  {
    if(a.shape.size() != 4 || a.shape[1] != JOINT_NUM || a.shape[2] != 3 || a.shape[3] != 3)
      throw Exception("WorldTransformation Error: Failed to set pose rotations!");
    rot_.upload(a);
  }
  void setKinematicTree(const std::vector<int64_t> & tree)
  {
    if(tree.size() != 2 * JOINT_NUM) throw Exception("WorldTransformation Error: Failed to set kinematic tree!");
    tree_.upload(tree.data(), tree.size());
  }
  /// WorldTransformation::transform (WorldTransformation.cpp:421-468)
  void transform()
  {
    if(batch_ < 1) throw Exception("WorldTransformation Error: Cannot transform bones!");
    out_.reserve(static_cast<size_t>(batch_ * JOINT_NUM * 16) * sizeof(float));
    check(smplpp_world_transformation(nullptr, batch_, tree_.as<int64_t>(), joints_.as<float>(), rot_.as<float>(), out_.as<float>()));
    done_ = true;
  }
  Array getTransformation() const
  {
    if(!done_) throw Exception("WorldTransformation Error: Failed to get transformations!");
    return detail::download(out_.as<float>(), {batch_, JOINT_NUM, 4, 4});
  }

private:
  int64_t batch_ = 0;
  bool done_ = false;
  detail::DeviceBuffer joints_, rot_, tree_, out_;
};

class LinearBlendSkinning
{
public:
  void setWeight(const Array & a)
  {
    if(a.shape.size() != 2 || a.shape[1] != JOINT_NUM) throw Exception("LinearBlendSkinning Error: Failed to set weights!");
    vertexNum_ = a.shape[0];
    weights_.upload(a);
  }
  void setRestShape(const Array & a)
  {
    if(a.shape.size() != 3 || a.shape[2] != 3) throw Exception("LinearBlendSkinning Error: Failed to set rest shape!");
    batch_ = a.shape[0];
    rest_.upload(a);
  }
  void setTransformation(const Array & a)
  {
    if(a.shape.size() != 4 || a.shape[1] != JOINT_NUM || a.shape[2] != 4 || a.shape[3] != 4)
      throw Exception("LinearBlendSkinning Error: Failed to set transformations!");
    xf_.upload(a);
  }
  void setRootPos(const Array & a)
  {
    root_.upload(a);
    haveRoot_ = true;
  }
  /// LinearBlendSkinning::skinning (LinearBlendSkinning.cpp:445-483)
  void skinning()
  {
    if(batch_ < 1 || vertexNum_ < 1) throw Exception("LinearBlendSkinning Error: Cannot skin the model!");
    out_.reserve(static_cast<size_t>(batch_ * vertexNum_ * 3) * sizeof(float));
    check(smplpp_linear_blend_skinning(nullptr, batch_, vertexNum_, weights_.as<float>(), rest_.as<float>(), xf_.as<float>(),
                                       haveRoot_ ? root_.as<float>() : nullptr, out_.as<float>()));
    done_ = true;
  }
  Array getVertex() const
  {
    if(!done_) throw Exception("LinearBlendSknning Error: Failed to get vertices of new pose!"); // sic, LinearBlendSkinning.cpp:409
    return detail::download(out_.as<float>(), {batch_, vertexNum_, 3});
  }

private:
  int64_t batch_ = 0, vertexNum_ = 0;
  bool done_ = false, haveRoot_ = false;
  detail::DeviceBuffer weights_, rest_, xf_, root_, out_;
};

/// The C3D file of the mocap modes as node/node.cpp:572-595, 667-691 uses it (there: ezc3d::c3d).
class C3d
{
public:
  explicit C3d(const std::string & path) { check(smplpp_c3d_open(path.c_str(), &c3d_)); }
  C3d(const C3d &) = delete;
  C3d & operator=(const C3d &) = delete;
  ~C3d()
  {
    if(c3d_) smplpp_c3d_close(c3d_);
  }
  int64_t nbFrames() const { return smplpp_c3d_frame_count(c3d_); }
  int64_t nbPoints() const { return smplpp_c3d_point_count(c3d_); }
  double frameRate() const { return smplpp_c3d_frame_rate(c3d_); }
  std::string label(int64_t i) const { return smplpp_c3d_label(c3d_, i); }
  /// first label ending with the task name (node.cpp:580-594); nbPoints() when there is none
  int64_t findLabel(const std::string & taskName) const { return smplpp_c3d_find_label(c3d_, taskName.c_str()); }
  /// frames [first, first + count): xyz (count, points, 3), valid (count, points); a missing point is zero / 0
  void read(int64_t first, int64_t count, std::vector<float> & xyz, std::vector<uint8_t> & valid) const
  {
    xyz.resize(static_cast<size_t>(count * nbPoints() * 3));
    valid.resize(static_cast<size_t>(count * nbPoints()));
    check(smplpp_c3d_read(c3d_, first, count, xyz.data(), valid.data()));
  }

private:
  smplpp_c3d_t * c3d_ = nullptr;
};

/// n smplpp::IkTask objects (IkTask.h:13-85) handled as one batch: the attachment faces are fixed here, the per-frame
/// fields (targetPos_, posTaskWeight_, vertexWeights_) are device arrays passed to smplpp_ik_step.
class IkTaskSet
{
public:
  IkTaskSet(const SMPL & smpl, const std::vector<int64_t> & faceIdx)
  {
    check(smplpp_tasks_create(smpl.handle(), static_cast<int32_t>(faceIdx.size()), faceIdx.data(), &tasks_));
  }
  IkTaskSet(const IkTaskSet &) = delete;
  IkTaskSet & operator=(const IkTaskSet &) = delete;
  ~IkTaskSet()
  {
    if(tasks_) smplpp_tasks_destroy(tasks_);
  }
  int32_t size() const { return smplpp_tasks_count(tasks_); }
  smplpp_tasks_t * handle() const { return tasks_; }

  /// One IK iteration for B frames with host arrays (the loop body of node/node.cpp:753-968 per frame): theta (B, 75 | 44),
  /// beta (B,10) or (1,10) shared, vertexWeights (B,n,3), targetPos (B,n,3), posTaskWeight (B,n) or empty.  theta, beta
  /// (with optimize_beta) and vertexWeights are updated in place; the residual, the Jacobian rows the reference harvests
  /// from Tensor::backward (node.cpp:823-873), A, b and the step are kept for the getters below.
  std::vector<int32_t> step(const SMPL & smpl, const VPoserDecoder * vposer, const smplpp_ik_options & opt, Array & theta,
                            Array & beta, Array & vertexWeights, const Array & targetPos, const Array & posTaskWeight = Array())
  {
    const int64_t b = theta.shape.at(0);
    const int32_t n = size();
    const int32_t thetaDim = smplpp_ik_theta_dim(&opt), dim = smplpp_ik_dim(&opt, n);
    if(theta.shape.size() != 2 || theta.shape[1] != thetaDim) throw Exception("IkTask Error: invalid IK step arguments!");
    if(vertexWeights.data.size() != static_cast<size_t>(b * n * 3) || targetPos.data.size() != static_cast<size_t>(b * n * 3))
      throw Exception("IkTask Error: invalid task tensors!");
    const int64_t stride = (beta.shape.at(0) == 1 && b > 1) ? 0 : SHAPE_BASIS_DIM;
    dTheta_.upload(theta), dBeta_.upload(beta), dVw_.upload(vertexWeights), dTgt_.upload(targetPos);
    const bool havePw = !posTaskWeight.data.empty();
    if(havePw) dPw_.upload(posTaskWeight);
    dStatus_.reserve(static_cast<size_t>(b) * sizeof(int32_t));
    dE_.reserve(static_cast<size_t>(b * 4 * n) * sizeof(float));
    dJ_.reserve(static_cast<size_t>(b * 4 * n * dim) * sizeof(float));
    dA_.reserve(static_cast<size_t>(b * dim * dim) * sizeof(double));
    dB_.reserve(static_cast<size_t>(b * dim) * sizeof(double));
    dDelta_.reserve(static_cast<size_t>(b * dim) * sizeof(double));
    const size_t ws = smplpp_ik_workspace_bytes(tasks_, &opt, b);
    dWs_.reserve(ws + 256);
    check(smplpp_ik_step(smpl.handle(), vposer ? vposer->handle() : nullptr, tasks_, &opt, nullptr, b, dTheta_.as<float>(),
                         dBeta_.as<float>(), stride, dVw_.as<float>(), dTgt_.as<float>(), nullptr,
                         havePw ? dPw_.as<float>() : nullptr, dStatus_.as<int32_t>(), dE_.as<float>(), dJ_.as<float>(),
                         dA_.as<double>(), dB_.as<double>(), dDelta_.as<double>(), dWs_.as<void>(), ws + 256));
    std::vector<int32_t> status(static_cast<size_t>(b));
    check(smplpp_copy_to_host(status.data(), dStatus_.as<int32_t>(), status.size() * sizeof(int32_t), nullptr));
    check(smplpp_copy_to_host(theta.ptr(), dTheta_.as<float>(), theta.data.size() * sizeof(float), nullptr));
    check(smplpp_copy_to_host(beta.ptr(), dBeta_.as<float>(), beta.data.size() * sizeof(float), nullptr));
    check(smplpp_copy_to_host(vertexWeights.ptr(), dVw_.as<float>(), vertexWeights.data.size() * sizeof(float), nullptr));
    batch_ = b, dim_ = dim;
    return status;
  }
  /// The linearisation alone (smplpp_ik_jacobian): what the reference obtains with one Tensor::backward per residual row
  /// (node.cpp:823-873), without the solve.  theta and beta are not modified; vertexWeights receives the re-weighting of
  /// node.cpp:803-804; getError() / getJacobian() return the result.
  void linearize(const SMPL & smpl, const VPoserDecoder * vposer, const smplpp_ik_options & opt, const Array & theta,
                 const Array & beta, Array & vertexWeights, const Array & targetPos, const Array & posTaskWeight = Array())
  {
    const int64_t b = theta.shape.at(0);
    const int32_t n = size();
    const int32_t thetaDim = smplpp_ik_theta_dim(&opt), dim = smplpp_ik_dim(&opt, n);
    if(theta.shape.size() != 2 || theta.shape[1] != thetaDim) throw Exception("IkTask Error: invalid IK step arguments!");
    if(vertexWeights.data.size() != static_cast<size_t>(b * n * 3) || targetPos.data.size() != static_cast<size_t>(b * n * 3))
      throw Exception("IkTask Error: invalid task tensors!");
    const int64_t stride = (beta.shape.at(0) == 1 && b > 1) ? 0 : SHAPE_BASIS_DIM;
    dTheta_.upload(theta), dBeta_.upload(beta), dVw_.upload(vertexWeights), dTgt_.upload(targetPos);
    const bool havePw = !posTaskWeight.data.empty();
    if(havePw) dPw_.upload(posTaskWeight);
    dE_.reserve(static_cast<size_t>(b * 4 * n) * sizeof(float));
    dJ_.reserve(static_cast<size_t>(b * 4 * n * dim) * sizeof(float));
    const size_t ws = smplpp_ik_workspace_bytes(tasks_, &opt, b);
    dWs_.reserve(ws + 256);
    check(smplpp_ik_jacobian(smpl.handle(), vposer ? vposer->handle() : nullptr, tasks_, &opt, nullptr, b, dTheta_.as<float>(),
                             dBeta_.as<float>(), stride, dVw_.as<float>(), dTgt_.as<float>(), nullptr,
                             havePw ? dPw_.as<float>() : nullptr, dE_.as<float>(), dJ_.as<float>(), dWs_.as<void>(), ws + 256));
    check(smplpp_copy_to_host(vertexWeights.ptr(), dVw_.as<float>(), vertexWeights.data.size() * sizeof(float), nullptr));
    batch_ = b, dim_ = dim;
  }
  /// IkTask::calcActualPos (+ calcActualNormal) of every task after SMPL::launch (src/SMPL.cpp:671-737,
  /// src/IkTask.cpp:59-86) for B poses WITHOUT the mesh (smplpp_task_forward_host): beta (B,10) or (1,10) shared,
  /// theta (B,25,3), vertexWeights (B,n,3) or (1,n,3) shared.  Returns the positions (B,n,3); normals (nullable) receives
  /// the task normals (B,n,3).
  Array calcActualPositions(const SMPL & smpl, const Array & beta, const Array & theta, const Array & vertexWeights,
                            double normalOffset, Array * normals = nullptr)
  {
    const int32_t n = size();
    if(theta.shape.size() != 3 || theta.shape[1] != JOINT_NUM + 1 || theta.shape[2] != 3)
      throw Exception("IkTask Error: invalid IK step arguments!");
    const int64_t b = theta.shape[0];
    if(beta.shape.size() != 2 || beta.shape[1] != SHAPE_BASIS_DIM || (beta.shape[0] != b && beta.shape[0] != 1))
      throw Exception("BlendShape Error: Failed to set beta!");
    if(vertexWeights.shape.size() != 3 || vertexWeights.shape[1] != n || vertexWeights.shape[2] != 3
       || (vertexWeights.shape[0] != b && vertexWeights.shape[0] != 1))
      throw Exception("IkTask Error: invalid task tensors!");
    const int64_t betaStride = (beta.shape[0] == 1 && b > 1) ? 0 : SHAPE_BASIS_DIM;
    const int64_t vwStride = (vertexWeights.shape[0] == 1 && b > 1) ? 0 : 3 * static_cast<int64_t>(n);
    Array pos({b, n, 3});
    if(normals) *normals = Array({b, n, 3});
    check(smplpp_task_forward_host(smpl.handle(), tasks_, b, beta.ptr(), betaStride, theta.ptr(), vertexWeights.ptr(),
                                   vwStride, static_cast<float>(normalOffset), pos.ptr(), normals ? normals->ptr() : nullptr));
    return pos;
  }
  /// e (B, 4n): rows 4m..4m+2 = posTaskWeight (actualPos - targetPos), row 4m+3 = the normal task (node.cpp:807-820)
  Array getError() const { return detail::download(dE_.as<float>(), {batch_, 4 * size()}); }
  /// J (B, 4n, dim) in the reference's column layout [theta | phi (2n) | beta] (node.cpp:787-877)
  Array getJacobian() const { return detail::download(dJ_.as<float>(), {batch_, 4 * size(), dim_}); }
  /// the step deltaConfig (B, dim) (node.cpp:907-939), float64 on the device, narrowed here
  std::vector<double> getDelta() const
  {
    std::vector<double> d(static_cast<size_t>(batch_ * dim_));
    if(!d.empty()) check(smplpp_copy_to_host(d.data(), dDelta_.as<double>(), d.size() * sizeof(double), nullptr));
    return d;
  }
  /// IkTask defaults (IkTask.h:59-84) + the constants of node/node.cpp:884-929
  static smplpp_ik_options defaultOptions()
  {
    smplpp_ik_options o;
    smplpp_ik_options_default(&o);
    return o;
  }

private:
  smplpp_tasks_t * tasks_ = nullptr;
  int64_t batch_ = 0;
  int32_t dim_ = 0;
  detail::DeviceBuffer dTheta_, dBeta_, dVw_, dTgt_, dPw_, dStatus_, dE_, dJ_, dA_, dB_, dDelta_, dWs_;
};

/// smplpp::IkTask (include/smplpp/IkTask.h:13-85, src/IkTask.cpp): ONE attachment face on batch element 0 of the last
/// SMPL::launch, with the reference's public fields and methods.  (Batched work goes through IkTaskSet.)
class IkTask
{
public:
  IkTask(const std::shared_ptr<SMPL> & smpl, int64_t faceIdx) : smpl_(smpl), faceIdx_(faceIdx)
  {
    targetPos_ = Array({3});
    targetNormal_ = Array({3});
    targetNormal_.data = {0.f, 0.f, 1.f}; // IkTask.cpp:13-16
    vertexWeights_ = Array({3});
    vertexWeights_.data = {1.f / 3.f, 1.f / 3.f, 1.f / 3.f}; // IkTask.h:74-78
    tangents_ = Array({3, 2});
    phi_ = Array({2});
  }
  /// IkTask::calcTangents (IkTask.cpp:33-47)
  void calcTangents()
  {
    detail::DeviceBuffer out;
    out.reserve(6 * sizeof(float));
    check(smplpp_task_tangents(smpl_->handle(), tasks(), nullptr, 1, smpl_->deviceVertices(), nullptr, out.as<float>()));
    tangents_ = detail::download(out.as<float>(), {3, 2});
  }
  /// IkTask::calcVertexWeights (IkTask.cpp:49-57): weights of actualPos + tangents * phi in the attachment triangle
  void calcVertexWeights(const Array & actualPos)
  {
    Array pos({3});
    for(int r = 0; r < 3; r++)
      pos.data[r] = actualPos.data.at(r) + tangents_.data[2 * r] * phi_.data[0] + tangents_.data[2 * r + 1] * phi_.data[1];
    const std::array<int32_t, 3> f = smpl_->getFaceIndexRaw(faceIdx_);
    const Array tri = smpl_->getVertexRaw(std::vector<int64_t>{f[0] - 1, f[1] - 1, f[2] - 1});
    vertexWeights_ = calcTriangleVertexWeights(pos, tri);
  }
  /// IkTask::calcActualPos (IkTask.cpp:59-72): sum_i w_i v_i (+ normalOffset_ * actual normal)
  Array calcActualPos() const { return positions(static_cast<float>(normalOffset_), false); }
  /// IkTask::calcActualNormal (IkTask.cpp:74-86)
  Array calcActualNormal() const { return positions(0.f, true); }

  std::shared_ptr<SMPL> smpl_;
  int64_t faceIdx_;
  Array targetPos_, targetNormal_;
  double posTaskWeight_ = 1.0, normalTaskWeight_ = 1.0, phiLimit_ = 0.04, normalOffset_ = 0.0; // IkTask.h:59-72
  Array vertexWeights_, tangents_, phi_;

private:
  smplpp_tasks_t * tasks() const
  {
    if(!set_ || setFace_ != faceIdx_)
    {
      set_.reset(new IkTaskSet(*smpl_, std::vector<int64_t>{faceIdx_}));
      setFace_ = faceIdx_;
    }
    return set_->handle();
  }
  Array positions(float offset, bool normal) const
  {
    detail::DeviceBuffer w, pos, nrm;
    w.upload(vertexWeights_);
    pos.reserve(3 * sizeof(float)), nrm.reserve(3 * sizeof(float));
    check(smplpp_task_positions(smpl_->handle(), tasks(), nullptr, 1, smpl_->deviceVertices(), w.as<float>(), offset,
                                pos.as<float>(), nrm.as<float>()));
    return detail::download(normal ? nrm.as<float>() : pos.as<float>(), {3});
  }
  mutable std::unique_ptr<IkTaskSet> set_;
  mutable int64_t setFace_ = -1;
};
} // namespace smplpp
