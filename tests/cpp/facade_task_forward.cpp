// smplpp::IkTaskSet::calcActualPositions (the markers-only forward pass through the header-only facade) against the
// compiled reference's IkTask::calcActualPos after SMPL::launch (tests/golden/ref_ik.npz, motion mode: re-weighted
// attachments of node.cpp:803-804, 15 mm normal offset), dumped as raw files by tests/test_task_forward_gpu.py.
// Also: shared vs per-frame inputs give the same bytes, normals are unit length, shape errors carry the reference texts.
// usage: facade_task_forward <dir>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>

#include "smplpp_b200/smplpp.hpp"

using namespace smplpp;

static std::string g_dir;
static std::vector<char> load_bytes(const std::string & name)
{
  std::ifstream f(g_dir + "/" + name, std::ios::binary | std::ios::ate);
  if(!f) throw Exception("facade_task_forward: cannot open " + name);
  std::vector<char> v(static_cast<size_t>(f.tellg()));
  f.seekg(0);
  f.read(v.data(), static_cast<std::streamsize>(v.size()));
  return v;
}
template<typename T>
static std::vector<T> load(const std::string & name)
{
  const std::vector<char> b = load_bytes(name);
  std::vector<T> v(b.size() / sizeof(T));
  std::memcpy(v.data(), b.data(), v.size() * sizeof(T));
  return v;
}
static Array arr(const std::string & name, std::vector<int64_t> shape)
{
  Array a(std::move(shape));
  const std::vector<float> v = load<float>(name);
  if(v.size() != a.data.size()) throw Exception("facade_task_forward: unexpected size of " + name);
  a.data = v;
  return a;
}
static int g_failed = 0;
static void expect(const char * what, double got, double tol)
{
  std::printf("  %-58s %.3g (tol %.1g) %s\n", what, got, tol, got <= tol ? "ok" : "FAIL");
  if(!(got <= tol)) g_failed++;
}

int main(int argc, char ** argv)
{
  if(argc < 2) return 2;
  g_dir = argv[1];
  try
  {
    SMPL smpl;
    smpl.setModelPath(g_dir + "/model.npz");
    smpl.init();
    const std::vector<int64_t> faces = load<int64_t>("ik_face_idx.i64");
    const int64_t n = static_cast<int64_t>(faces.size());
    const Array theta = arr("ik_theta_in.f32", {1, 25, 3}), beta = arr("ik_beta_in.f32", {1, 10});
    const Array vw = arr("ik_motion_vertex_weights_out.f32", {1, n, 3}), actual = arr("ik_motion_actual_pos.f32", {n, 3});
    IkTaskSet set(smpl, faces);
    std::puts("IkTaskSet::calcActualPositions (motion mode: re-weighted attachments, 15 mm normal offset)");
    Array normals;
    const Array pos = set.calcActualPositions(smpl, beta, theta, vw, 0.015, &normals);
    double mp = 0, ml = 0;
    for(int64_t m = 0; m < n; m++)
    {
      for(int k = 0; k < 3; k++) mp = std::fmax(mp, std::fabs(double(pos.data[3 * m + k]) - actual.data[3 * m + k]));
      const float * q = normals.ptr() + 3 * m;
      ml = std::fmax(ml, std::fabs(std::sqrt(double(q[0]) * q[0] + double(q[1]) * q[1] + double(q[2]) * q[2]) - 1.0));
    }
    expect("positions vs reference calcActualPos [m]", mp, 1e-5);
    expect("normals unit length", ml, 1e-5);
    // three copies of the frame: shared beta / weights (stride 0) and per-frame rows give the same bytes as one frame
    const int64_t B = 3;
    Array theta3({B, 25, 3}), beta3({B, 10}), vw3({B, n, 3});
    for(int64_t b = 0; b < B; b++)
    {
      std::copy(theta.data.begin(), theta.data.end(), theta3.data.begin() + b * 75);
      std::copy(beta.data.begin(), beta.data.end(), beta3.data.begin() + b * 10);
      std::copy(vw.data.begin(), vw.data.end(), vw3.data.begin() + b * n * 3);
    }
    const Array shared = set.calcActualPositions(smpl, beta, theta3, vw, 0.015);
    const Array perFrame = set.calcActualPositions(smpl, beta3, theta3, vw3, 0.015);
    bool same = true;
    for(int64_t b = 0; b < B; b++)
      same &= std::memcmp(shared.ptr() + b * n * 3, pos.ptr(), n * 3 * sizeof(float)) == 0
              && std::memcmp(perFrame.ptr() + b * n * 3, pos.ptr(), n * 3 * sizeof(float)) == 0;
    expect("shared and per-frame inputs: bitwise the single frame", same ? 0.0 : 1.0, 0.0);
    try
    {
      set.calcActualPositions(smpl, Array({B, 9}), theta3, vw, 0.0);
      g_failed++;
    }
    catch(const Exception & e)
    {
      expect("beta (B,9) throws the reference's text", std::strstr(e.what(), "BlendShape Error: Failed to set beta!") ? 0 : 1, 0);
    }
    try
    {
      set.calcActualPositions(smpl, beta, theta3, Array({2, n, 3}), 0.0);
      g_failed++;
    }
    catch(const Exception & e)
    {
      expect("weights (2,n,3) for B = 3 throws", std::strstr(e.what(), "IkTask Error: invalid task tensors!") ? 0 : 1, 0);
    }
  }
  catch(const Exception & e)
  {
    std::printf("FAIL: %s\n", e.what());
    return 1;
  }
  if(g_failed)
  {
    std::printf("facade task forward: %d FAIL\n", g_failed);
    return 1;
  }
  std::puts("facade task forward: OK");
  return 0;
}
