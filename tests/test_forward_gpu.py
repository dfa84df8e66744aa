"""GPU parity tests of the forward path (K1 pose chain, K2 fused blend + skinning, K3 skinning, module kernels,
normals) against the oracle and the reference golden vectors.  Everything goes through the C-ABI library."""
import numpy as np
import pytest
import torch

from conftest import TOL_VERTEX_M

pytestmark = pytest.mark.gpu

f32 = np.float32


def dev(a):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=f32), device="cuda:0")


# ---- known-answer vectors of src/toolbox/Tester.cpp through the module-level API ----

def test_kat_blend_shape(kat):
    from smplpp_b200 import api
    i, e = kat["blendShape"]["inputs"], kat["blendShape"]["expected"]
    m = api.BlendShape()
    m.setBeta(np.asarray(i["beta"]))
    m.setTheta(np.asarray(i["theta"]))
    m.setShapeBlendBasis(np.asarray(i["shapeBlendBasis"]))
    m.setPoseBlendBasis(np.asarray(i["poseBlendBasis"]))
    m.blend()
    assert np.allclose(m.getShapeBlendShape().cpu().numpy().reshape(-1), np.asarray(e["shapeBlendShape"]).reshape(-1),
                       atol=2e-6)
    assert np.allclose(m.getPoseBlendShape().cpu().numpy().reshape(-1), np.asarray(e["poseBlendShape"]).reshape(-1),
                       atol=5e-6)
    assert np.allclose(m.getPoseRotation().cpu().numpy()[0, :5], np.asarray(e["poseRotation"]), atol=1.5e-6)


def test_kat_joint_regression(kat):
    from smplpp_b200 import api
    i, e = kat["jointRegression"]["inputs"], kat["jointRegression"]["expected"]
    m = api.JointRegression()
    m.setShapeBlendShape(np.asarray(i["shapeBlendShape"]))
    m.setPoseBlendShape(np.asarray(i["poseBlendShape"]))
    m.setTemplateRestShape(np.asarray(i["templateShape"]))
    m.setJointRegressor(np.asarray(i["jointRegressor"]))
    m.regress()
    assert np.allclose(m.getRestShape().cpu().numpy(), np.asarray(e["restShape"]), atol=1.5e-6)
    assert np.allclose(m.getJoint().cpu().numpy()[0], np.asarray(e["joints"]), atol=2e-6)


def test_kat_world_transformation(kat):
    from smplpp_b200 import api
    i, e = kat["worldTransformation"]["inputs"], kat["worldTransformation"]["expected"]
    m = api.WorldTransformation()
    m.setKinematicTree(np.asarray(i["kineTree"], dtype=np.int64))
    m.setJoint(np.asarray(i["joints"]))
    m.setPoseRotation(np.asarray(i["poseRotation"]))
    m.transform()
    got = m.getTransformation().cpu().numpy()[0, :5]
    assert np.allclose(got, np.asarray(e["transformations"]), atol=2e-6, rtol=2e-6)


def test_kat_linear_blend_skinning(kat):
    from smplpp_b200 import api
    i, e = kat["linearBlendSkinning"]["inputs"], kat["linearBlendSkinning"]["expected"]
    m = api.LinearBlendSkinning()
    m.setWeight(np.asarray(i["weights"]))
    m.setRestShape(np.asarray(i["restShape"]))
    m.setTransformation(np.asarray(i["transformations"]))
    m.skinning()
    assert np.allclose(m.getVertex().cpu().numpy().reshape(-1), np.asarray(e["vertices"]).reshape(-1), atol=1.5e-6)


# ---- full model: golden vectors of the compiled reference ----

@pytest.mark.parametrize("variant", [1, 3, 6])
def test_forward_vs_reference_golden(smpl_gpu, golden_forward, variant):
    from smplpp_b200 import capi
    g = golden_forward
    capi.check(capi.lib().smplpp_set_forward_variant(variant))
    try:
        smpl_gpu.launch(g["beta"], g["theta"])
        v = smpl_gpu.getVertex().cpu().numpy()
        j = smpl_gpu.getRestJoint().cpu().numpy()
        rest = smpl_gpu.getRestShape().cpu().numpy()
    finally:
        capi.check(capi.lib().smplpp_set_forward_variant(0))
    assert np.abs(v - g["vertices"]).max() <= TOL_VERTEX_M
    assert np.abs(j - g["joints"]).max() <= TOL_VERTEX_M
    assert np.abs(rest - g["rest_shape"]).max() <= TOL_VERTEX_M
    # in practice the fp32 FFMA path and the tcgen05 fp16 split-precision path sit well below the stated tolerance
    assert np.abs(v - g["vertices"]).max() < 2e-6


@pytest.mark.parametrize("variant", [6])
@pytest.mark.parametrize("batch", [1, 2, 8, 9, 95, 96, 97, 127, 191, 192, 193, 300])
def test_forward_tensor_core_variants_match_ffma(smpl_gpu, variant, batch):
    """Ragged frame counts through the tcgen05 kernel (96-frame blocks, 8-frame transform sub-batches, frame pairs
    per epilogue warp) against the FFMA kernel on the same inputs, every frame and vertex."""
    from smplpp_b200 import capi, synth
    beta, theta = synth.make_forward_inputs(batch, 77 + batch)
    out = {}
    for var in (1, variant):
        capi.check(capi.lib().smplpp_set_forward_variant(var))
        try:
            smpl_gpu.launch(beta, theta)
            out[var] = smpl_gpu.getVertex().cpu().numpy()
        finally:
            capi.check(capi.lib().smplpp_set_forward_variant(0))
    assert np.isfinite(out[variant]).all()
    assert np.abs(out[variant] - out[1]).max() < 1e-6


@pytest.mark.parametrize("batch", [2000, 4096 + 37])
def test_forward_pipelined_kernel_many_items_per_cta(smpl_gpu, batch):
    """The persistent tcgen05 kernel (variant 6, skin_tc3.cu) with many work items per CTA: ring wrap-around, vertex-tile
    changes inside a CTA's range and a ragged last frame block, against the FFMA kernel on every frame and vertex."""
    from smplpp_b200 import capi, synth
    beta, theta = synth.make_forward_inputs(batch, 5 + batch)
    out = {}
    for var in (1, 6):
        capi.check(capi.lib().smplpp_set_forward_variant(var))
        try:
            smpl_gpu.launch(beta, theta)
            out[var] = smpl_gpu.getVertex()
        finally:
            capi.check(capi.lib().smplpp_set_forward_variant(0))
    assert bool(torch.isfinite(out[6]).all())
    assert float((out[6] - out[1]).abs().max()) < 1e-6


def test_normals_vs_reference_golden(smpl_gpu, golden_forward, oracle_model):
    """calcNormal / calcVertexNormal (SMPL.cpp:518-535).  A normal amplifies a vertex error by 1 / edge length
    (edges of the synthetic mesh go down to a few mm), so the comparison has two parts: (1) the kernel against the
    oracle's formula on the SAME (GPU) vertices, tight; (2) against the compiled reference's golden normals within
    the vertex tolerance amplified by the mesh's edge scale (1e-5 m / ~5 cm typical edge => 2e-4)."""
    import torch
    from oracle import smpl_oracle as so
    g = golden_forward
    smpl_gpu.launch(g["beta"][:1], g["theta"][:1])
    fn, vn = smpl_gpu.normals(g["normal_face_idx"], g["normal_vert_idx"])
    fn, vn = fn.cpu().numpy()[0], vn.cpu().numpy()[0]
    v0 = smpl_gpu.getVertex()[0].cpu()
    fn_o = np.stack([so.calc_normal(oracle_model, v0, int(f)).numpy() for f in g["normal_face_idx"]])
    vn_o = np.stack([so.calc_vertex_normal(oracle_model, v0, int(i)).numpy() for i in g["normal_vert_idx"]])
    assert np.abs(fn - fn_o).max() < 2e-6 and np.abs(vn - vn_o).max() < 2e-6
    assert np.abs(fn - g["face_normals"]).max() < 2e-4
    assert np.abs(vn - g["vertex_normals"]).max() < 2e-4
    assert np.abs(smpl_gpu.calcNormal(int(g["normal_face_idx"][3])).cpu().numpy() - g["face_normals"][3]).max() < 2e-4


# ---- full model vs the oracle on seeded inputs (ragged batch sizes cross every tile boundary) ----

@pytest.mark.parametrize("batch,seed,shared_beta", [(1, 10, False), (70, 11, False), (129, 12, True)])
def test_forward_vs_oracle(smpl_gpu, oracle_model, batch, seed, shared_beta):
    from oracle import smpl_oracle as so
    from smplpp_b200 import synth
    beta, theta = synth.make_forward_inputs(batch, seed)
    if shared_beta:
        beta = np.repeat(beta[:1], batch, axis=0)
    v_o, j_o, rest_o, xf_o = so.forward_numpy(oracle_model, beta, theta)
    smpl_gpu.launch(beta[:1] if shared_beta else beta, theta, want_transforms=True)
    v = smpl_gpu.getVertex().cpu().numpy()
    assert np.abs(v - v_o).max() <= TOL_VERTEX_M
    assert np.abs(smpl_gpu.getRestJoint().cpu().numpy() - j_o).max() <= TOL_VERTEX_M
    assert np.abs(smpl_gpu.getRestShape().cpu().numpy() - rest_o).max() <= TOL_VERTEX_M
    assert np.abs(smpl_gpu.getTransformation().cpu().numpy() - xf_o).max() <= TOL_VERTEX_M


def test_edge_poses_vs_oracle(smpl_gpu, oracle_model):
    """theta = 0 (Rodrigues with a = sqrt(3) 1e-8), tiny angles, angles near pi and 2 pi."""
    from oracle import smpl_oracle as so
    rng = np.random.default_rng(3)
    theta = np.zeros((6, 25, 3), f32)
    theta[1, 1:] = 1e-7
    theta[2, 1:] = rng.normal(size=(24, 3)) * 1e-4
    axis = rng.normal(size=(24, 3))
    axis /= np.linalg.norm(axis, axis=1, keepdims=True)
    theta[3, 1:] = axis * np.pi
    theta[4, 1:] = axis * (2 * np.pi - 1e-3)
    theta[5, 1:] = axis * 5.0
    theta[:, 0] = rng.uniform(-1, 1, size=(6, 3))
    beta = rng.normal(size=(6, 10)).astype(f32) * 2
    v_o, j_o, _, _ = so.forward_numpy(oracle_model, beta, theta)
    smpl_gpu.launch(beta, theta)
    assert np.abs(smpl_gpu.getVertex().cpu().numpy() - v_o).max() <= TOL_VERTEX_M
    assert np.isfinite(smpl_gpu.getVertex().cpu().numpy()).all()


def test_model_skinning_vs_oracle(smpl_gpu, oracle_model, params):
    """K3 standalone (packed sparse weights, 4x4 transforms incl. homogeneous row) vs LinearBlendSkinning."""
    import ctypes as C
    from oracle import smpl_oracle as so
    from smplpp_b200 import api, capi, synth
    beta, theta = synth.make_forward_inputs(19, 13)
    with torch.no_grad():
        r = so.smpl_launch(oracle_model, torch.as_tensor(beta), torch.as_tensor(theta))
    rest, xf = dev(r.rest_shape.numpy()), dev(r.transforms.numpy())
    root = dev(theta[:, 0])
    out = torch.empty_like(rest)
    capi.check(capi.lib().smplpp_model_skinning(smpl_gpu.handle, None, C.c_int64(19), api._ptr(rest), api._ptr(xf),
                                                api._ptr(root), api._ptr(out)))
    torch.cuda.synchronize()
    assert np.abs(out.cpu().numpy() - r.vertices.numpy()).max() <= TOL_VERTEX_M
    xf34 = xf[:, :, :3, :].contiguous()
    out34 = torch.empty_like(rest)
    capi.check(capi.lib().smplpp_model_skinning34(smpl_gpu.handle, None, C.c_int64(19), api._ptr(rest), api._ptr(xf34),
                                                  api._ptr(root), api._ptr(out34)))
    torch.cuda.synchronize()
    assert np.abs(out34.cpu().numpy() - r.vertices.numpy()).max() <= TOL_VERTEX_M


@pytest.mark.parametrize("batch", [1, 2, 19, 50, 700])
def test_skinning_tma_pipeline(smpl_gpu, oracle_model, batch):
    """K3' (per-warp TMA pipelines, lbs_tma.cu) against LinearBlendSkinning (oracle) and against the
    register-pipelined kernel bit for bit: odd frames start 8 bytes off a 16-byte boundary, the last slice is short
    (6890 = 53 x 128 + 106), the last chunk ends exactly at the end of the allocation, 16-frame CTAs are ragged."""
    import ctypes as C
    from oracle import smpl_oracle as so
    from smplpp_b200 import api, capi, synth
    beta, theta = synth.make_forward_inputs(batch, 31 + batch)
    with torch.no_grad():
        r = so.smpl_launch(oracle_model, torch.as_tensor(beta), torch.as_tensor(theta))
    V = r.rest_shape.shape[1]
    xf34 = dev(r.transforms.numpy()[:, :, :3, :].copy())
    root = dev(theta[:, 0])
    # exact-size allocations (torch rounds to 512 B; the tail guard words make an overrun visible)
    rest = dev(r.rest_shape.numpy())
    guard = torch.full((batch * V * 3 + 64,), 7.0, dtype=torch.float32, device="cuda:0")
    outs = {}
    for var in (201, 200, 202):  # FFMA register kernel, FFMA TMA pipeline, tcgen05 skinning matrices
        capi.check(capi.lib().smplpp_set_forward_variant(var))
        guard.fill_(7.0)
        out = guard[:batch * V * 3].view(batch, V, 3)
        try:
            capi.check(capi.lib().smplpp_model_skinning34(smpl_gpu.handle, None, C.c_int64(batch), api._ptr(rest),
                                                          api._ptr(xf34), api._ptr(root), api._ptr(out)))
            torch.cuda.synchronize()
        finally:
            capi.check(capi.lib().smplpp_set_forward_variant(202))
        assert (guard[batch * V * 3:] == 7.0).all()
        outs[var] = out.cpu().numpy().copy()
    for var in outs:
        assert np.abs(outs[var] - r.vertices.numpy()).max() <= TOL_VERTEX_M
    assert np.array_equal(outs[200], outs[201])
    assert np.abs(outs[202] - outs[201]).max() < 1.5e-6  # fp16x3 split of W and G' (2^-22 relative on ~1 m terms)
    # no root translation
    out = torch.empty_like(rest)
    capi.check(capi.lib().smplpp_model_skinning34(smpl_gpu.handle, None, C.c_int64(batch), api._ptr(rest), api._ptr(xf34),
                                                  None, api._ptr(out)))
    torch.cuda.synchronize()
    assert np.abs(out.cpu().numpy() + theta[:, :1] - r.vertices.numpy()).max() <= TOL_VERTEX_M


def test_dense_weights_small_model():
    """A model whose skinning rows are dense (24 non-zeros, sums != 1) and V not a multiple of the tile."""
    from oracle import smpl_oracle as so
    from smplpp_b200 import api, synth
    rng = np.random.default_rng(7)
    V = 77
    tree = np.stack([synth.PARENTS.copy(), np.arange(24)])
    tree[0, 0] = 4294967295
    faces = np.stack([rng.permutation(V)[:3] for _ in range(40)]).astype(np.int32) + 1
    p = synth.SmplParams(
        face_indices=faces, shape_blend_shapes=rng.normal(size=(V, 3, 10)).astype(f32) * 0.01,
        pose_blend_shapes=rng.normal(size=(V, 3, 207)).astype(f32) * 0.002,
        vertices_template=rng.normal(size=(V, 3)).astype(f32) * 0.3,
        joint_regressor=rng.dirichlet(np.ones(V), size=24).astype(f32), kinematic_tree=tree,
        weights=rng.uniform(0.1, 1.0, size=(V, 24)).astype(f32))
    m = api.SMPL(p)
    assert m.vertex_num == V
    beta, theta = synth.make_forward_inputs(5, 14)
    om = so.SmplModel.from_params(p)
    v_o, j_o, rest_o, _ = so.forward_numpy(om, beta, theta)
    m.launch(beta, theta)
    assert np.abs(m.getVertex().cpu().numpy() - v_o).max() <= TOL_VERTEX_M
    assert np.abs(m.getRestShape().cpu().numpy() - rest_o).max() <= TOL_VERTEX_M
    assert np.abs(m.getRestJoint().cpu().numpy() - j_o).max() <= TOL_VERTEX_M


# ---- BASELINE config 2 (B = 4096): size-independent properties ----

def test_full_batch_properties(smpl_gpu, oracle_model):
    from oracle import smpl_oracle as so
    from smplpp_b200 import synth
    B = 4096
    beta, theta = synth.make_forward_inputs(B, 11)
    smpl_gpu.launch(beta, theta)
    v = smpl_gpu.getVertex()
    assert torch.isfinite(v).all()
    # (a) batch invariance: any frame of the big batch equals the same frame launched alone
    pick = [0, 63, 64, 1000, 4095]
    smpl_gpu.launch(beta[pick], theta[pick])
    assert (smpl_gpu.getVertex() - v[pick]).abs().max().item() == 0.0
    # (b) spot-check against the oracle
    v_o, _, _, _ = so.forward_numpy(oracle_model, beta[pick], theta[pick])
    assert np.abs(v[pick].cpu().numpy() - v_o).max() <= TOL_VERTEX_M
    # (c) translation equivariance: moving theta row 0 moves every vertex by the same vector
    shift = np.array([0.25, -1.5, 3.0], f32)
    theta2 = theta.copy()
    theta2[:, 0] += shift
    smpl_gpu.launch(beta, theta2)
    d = smpl_gpu.getVertex() - v
    assert (d - torch.as_tensor(shift, device=d.device)).abs().max().item() < 2e-6
    # (d) rest pose: theta = 0 gives T + S beta (+ translation)
    theta0 = np.zeros_like(theta[:8])
    theta0[:, 0] = theta[:8, 0]
    smpl_gpu.launch(beta[:8], theta0)
    rest = smpl_gpu.getRestShape()
    assert (smpl_gpu.getVertex() - (rest + torch.as_tensor(theta0[:, :1], device=rest.device))).abs().max().item() < 2e-6


def test_launch_host_matches_device(smpl_gpu):
    from smplpp_b200 import synth
    beta, theta = synth.make_forward_inputs(33, 15)
    smpl_gpu.launch(beta, theta)
    v = smpl_gpu.getVertex().cpu().numpy()
    j = smpl_gpu.getRestJoint().cpu().numpy()
    vh, jh = smpl_gpu.launch_host(beta, theta)
    assert np.array_equal(v, vh) and np.array_equal(j, jh)


@pytest.mark.parametrize("n,shared_beta", [(700, False), (513, True), (256, False)])
def test_launch_host_chunked_pipeline(smpl_gpu, n, shared_beta):
    """smplpp_forward_host runs the batch in 256-frame chunks on two streams: ragged last chunk, page-locked
    and pageable destinations, shared beta (stride 0) must all equal the one-shot device launch bit for bit."""
    from smplpp_b200 import api, synth
    beta, theta = synth.make_forward_inputs(n, 16)
    if shared_beta:
        beta = beta[:1]
    smpl_gpu.launch(beta, theta)
    v = smpl_gpu.getVertex().cpu().numpy()
    j = smpl_gpu.getRestJoint().cpu().numpy()
    # pageable destinations (staged through pinned chunk buffers, host threads copy out)
    vh, jh = smpl_gpu.launch_host(beta, theta)
    assert np.array_equal(v, vh) and np.array_equal(j, jh)
    # page-locked sources and destinations (DMA straight into the caller's arrays), called twice (buffer reuse)
    pb, pt = api.pinned_empty(beta.shape), api.pinned_empty(theta.shape)
    pb[...], pt[...] = beta, theta
    pv, pj = api.pinned_empty(v.shape), api.pinned_empty(j.shape)
    for _ in range(2):
        pv.fill(np.nan)
        smpl_gpu.launch_host(pb, pt, out_vertices=pv, out_joints=pj)
        assert np.array_equal(v, pv) and np.array_equal(j, pj)
    # vertices only
    pv.fill(np.nan)
    smpl_gpu.launch_host(pb, pt, want_joints=False, out_vertices=pv)
    assert np.array_equal(v, pv)


def test_error_messages(smpl_gpu):
    """Shape violations raise with the reference's message text (smpl_error, Exception.cpp:77-91)."""
    from smplpp_b200 import api
    with pytest.raises(api.SmplppError, match="Cannot launch a SMPL model!"):
        smpl_gpu.launch(np.zeros((2, 10), f32), np.zeros((2, 24, 3), f32))
    with pytest.raises(api.SmplppError, match="BlendShape Error: Failed to set beta!"):
        smpl_gpu.launch(np.zeros((2, 9), f32), np.zeros((2, 25, 3), f32))
    m = api.BlendShape()
    with pytest.raises(api.SmplppError, match="Failed to set theta!"):
        m.setTheta(np.zeros((1, 23, 3), f32))
    fresh = api.SMPL()
    with pytest.raises(api.SmplppError, match="Failed to initialize model path!"):
        fresh.setModelPath("/nonexistent/smpl_male.json")
    with pytest.raises(api.SmplppError, match="Cannot initialize a SMPL model!"):
        fresh.init()


def test_cpp_facade_smoke(tmp_path, params, vposer_params):
    """The header-only C++ facade (smplpp::SMPL / VPoserDecoder / C3d over the C ABI) end to end on the GPU:
    tests/cpp/facade_smoke.cpp, including setModelPath + init() and loadParamsFromJson on JSON files and the C3D reader."""
    import os
    import subprocess
    import sys
    from smplpp_b200 import synth
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, "tests"))
    from c3d_writer import write_c3d
    exe = os.path.join(root, "tests", "cpp", "facade_smoke")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-s", "-C", os.path.join(root, "tests", "cpp")])
    mpath, vpath, cpath = str(tmp_path / "model.json"), str(tmp_path / "vposer.json"), str(tmp_path / "walk.c3d")
    params.to_json(mpath)
    synth.vposer_to_json(vposer_params, vpath)
    rng = np.random.default_rng(0)
    write_c3d(cpath, rng.normal(size=(12, 5, 3)).astype(np.float32), rng.random((12, 5)) > 0.2, ["A", "B", "C", "D", "E"])
    r = subprocess.run([exe, mpath, vpath, cpath], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "facade smoke: OK" in r.stdout, r.stdout + r.stderr
    assert "c3d 12 frames x 5 points at 120 Hz, first label A" in r.stdout
    assert "V=6890, 13776 faces" in r.stdout


def test_native_json_loaders_match_python_loaders(tmp_path, params, vposer_params):
    """smplpp_model_load_json / smplpp_vposer_load_json (SMPL::init, VPoserDecoder::loadParamsFromJson through the
    C-ABI JSON reader) build the same device models as the arrays handed over by the Python mirror."""
    from smplpp_b200 import api, synth
    mpath, vpath = str(tmp_path / "model.json"), str(tmp_path / "vposer.json")
    params.to_json(mpath)
    synth.vposer_to_json(vposer_params, vpath)
    a = api.SMPL(params, device="cuda:0")
    b = api.SMPL.from_json_native(mpath, device="cuda:0")
    beta, theta = synth.make_forward_inputs(7, 3)
    a.launch(beta, theta)
    b.launch(beta, theta)
    assert torch.equal(a.getVertex(), b.getVertex()) and torch.equal(a.getRestJoint(), b.getRestJoint())
    assert torch.equal(a.getFaceIndex(), b.getFaceIndex())
    # the .npz twin (np.savez, scripts/preprocess.py:98-117) through smplpp_model_load_npz
    npath = str(tmp_path / "model.npz")
    np.savez(npath, vertices_template=params.vertices_template, face_indices=params.face_indices, weights=params.weights,
             shape_blend_shapes=params.shape_blend_shapes, pose_blend_shapes=params.pose_blend_shapes,
             joint_regressor=params.joint_regressor, kinematic_tree=params.kinematic_tree)
    c = api.SMPL.from_json_native(npath, device="cuda:0")
    c.launch(beta, theta)
    assert torch.equal(a.getVertex(), c.getVertex()) and torch.equal(a.getFaceIndex(), c.getFaceIndex())
    va = api.VPoserDecoder(vposer_params, device="cuda:0")
    vb = api.VPoserDecoder(device="cuda:0")
    vb.loadParamsFromJsonNative(vpath)
    z = np.random.default_rng(0).normal(size=(5, 32)).astype(np.float32)
    assert torch.equal(va.forward(z), vb.forward(z))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs in one process")
def test_two_devices_in_one_process(params, vposer_params):
    """One process driving two devices (function attributes, memory pools and model constants are per device): the same
    forward pass, projection and VPoser Jacobian on cuda:0 and cuda:1 give identical results."""
    from smplpp_b200 import api, synth
    beta, theta = synth.make_forward_inputs(200, 5)
    z = np.random.default_rng(1).normal(size=(9, 32)).astype(np.float32)
    res = []
    for dev in ("cuda:0", "cuda:1"):
        smpl = api.SMPL(params, device=dev)
        smpl.launch(beta, theta)
        v = smpl.getVertex()
        face, closest, sq, w = smpl.projectPoints(v[:, ::200][:, :30].contiguous() + 0.01)
        vp = api.VPoserDecoder(vposer_params, device=dev)
        aa, jac = vp.forward(z, jacobian=True)
        res.append([t.cpu() for t in (v, face, closest, aa, jac)])
    for a, b in zip(*res):
        assert torch.equal(a, b)
