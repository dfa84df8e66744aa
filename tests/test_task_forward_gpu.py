"""Markers-only forward pass (smplpp_task_forward / smplpp_task_forward_host; IkTaskSet.forward_positions[_host];
smplpp::IkTaskSet::calcActualPositions): IkTask::calcActualPos / calcActualNormal for a batch of poses without the mesh,
against the compiled reference's golden, the oracle and the existing route smplpp_forward + smplpp_task_positions."""
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import TOL_VERTEX_M

pytestmark = pytest.mark.gpu
f32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FACADE_SRC = os.path.join(ROOT, "tests", "cpp", "facade_task_forward.cpp")
BATCH = 4096 + 37  # ragged: not a multiple of the 128-frame tile of the rest-shape kernel
NORMAL_TOL_RAD = 1e-3  # estimate: a normal amplifies a vertex difference by 1 / edge length


@pytest.fixture(params=[420, 421], ids=["restshape_tc", "restshape_ffma"])
def rest_variant(request):
    """Rest rows of the task vertices on tcgen05 (420, the default) or by the FFMA blend kernel (421)."""
    from smplpp_b200 import capi
    try:
        capi.check(capi.lib().smplpp_set_forward_variant(request.param))
        yield request.param
    finally:
        capi.check(capi.lib().smplpp_set_forward_variant(420))


@pytest.fixture(scope="module")
def marker_set(smpl_gpu, marker_tasks):
    from smplpp_b200 import api
    _, face_idx, _ = marker_tasks
    return api.IkTaskSet(smpl_gpu, face_idx)


@pytest.fixture(scope="module")
def poses():
    from smplpp_b200 import synth
    return synth.make_forward_inputs(BATCH, 31)


def _weights(n, batch, seed):
    rng = np.random.default_rng(seed)
    w = rng.dirichlet(np.ones(3), size=(batch, n)).astype(f32)
    return w


def _old_route(smpl, tset, beta, theta, w, offset):
    """smplpp_forward (full mesh) + smplpp_task_positions: what the library offered before."""
    smpl.launch(beta, theta)
    wb = np.broadcast_to(w.reshape(-1, tset.n, 3), (theta.shape[0], tset.n, 3))
    pos, nrm = tset.positions(smpl.getVertex(), np.ascontiguousarray(wb), offset, want_normals=True)
    return pos.cpu().numpy(), nrm.cpu().numpy()


def _angle(a, b):
    c = np.clip(np.sum(a.astype(np.float64) * b, axis=-1) / (np.linalg.norm(a, axis=-1) * np.linalg.norm(b, axis=-1)), -1, 1)
    return np.arccos(c)


def test_reference_golden(smpl_gpu, golden_ik, rest_variant):
    """Motion mode of the compiled reference: calcActualPos after the re-weighting of node.cpp:803-804, 15 mm offset."""
    from smplpp_b200 import api
    g = golden_ik
    tset = api.IkTaskSet(smpl_gpu, g["face_idx"])
    theta, beta, w = g["theta_in"].reshape(1, 25, 3), g["beta_in"].reshape(1, 10), g["motion_vertex_weights_out"]
    pos = tset.forward_positions(beta, theta, w, 0.015).cpu().numpy()[0]
    pos_h = tset.forward_positions_host(beta, theta, w, 0.015)[0]
    err = np.abs(pos - g["motion_actual_pos"]).max()
    print("golden: max |pos - reference calcActualPos| = %.3g m" % err)
    assert err <= TOL_VERTEX_M
    assert np.array_equal(pos, pos_h)


@pytest.mark.parametrize("offset", [0.0, 0.015])
@pytest.mark.parametrize("shared_weights", [False, True], ids=["weights_per_frame", "weights_shared"])
@pytest.mark.parametrize("shared_beta", [False, True], ids=["beta_per_frame", "beta_shared"])
def test_against_old_route_and_oracle(smpl_gpu, marker_set, oracle_model, poses, rest_variant, shared_beta, shared_weights,
                                      offset):
    from oracle import smpl_oracle as so
    beta, theta = poses
    if shared_beta:
        beta = beta[:1]
    n = marker_set.n
    w = _weights(n, 1 if shared_weights else BATCH, 5)
    pos, nrm = marker_set.forward_positions(beta, theta, w[0] if shared_weights else w, offset, want_normals=True)
    pos, nrm = pos.cpu().numpy(), nrm.cpu().numpy()
    assert pos.shape == (BATCH, n, 3) and np.isfinite(pos).all()
    pos_old, nrm_old = _old_route(smpl_gpu, marker_set, beta, theta, w, offset)
    # every frame against the full-mesh route.  The offset term moves the point along the task normal, and a normal
    # amplifies a vertex difference by 1 / edge length: the two routes' meshes differ by ~1e-7..5e-7 m, which on the
    # sub-millimetre edges of some posed ring faces turns the normals by a few mrad, and 0.015 m x mrad is above 1e-5 m.
    # So the point on the face (calcActualPos without the offset term) is compared on every frame; the full position
    # and the normal are compared with the oracle on fixed frames, and on the frames where the two routes disagree most
    # the new route must be at least as close to the oracle as the old one.
    err_old = np.abs(pos - pos_old).max()
    err_face = np.abs((pos - offset * nrm) - (pos_old - offset * nrm_old)).max()
    assert err_face <= TOL_VERTEX_M
    # unit normals
    assert np.abs(np.linalg.norm(nrm.astype(np.float64), axis=-1) - 1).max() <= 1e-5
    d = np.abs(pos - pos_old).max(axis=2)
    fixed = [0, 127, 128, 2049, BATCH - 1]
    worst = [int(f) for f in np.argsort(d.max(axis=1))[-3:] if int(f) not in fixed]
    frames = fixed + worst
    bsel = np.repeat(beta, len(frames), axis=0) if shared_beta else beta[frames]
    v_o, _, _, _ = so.forward_numpy(oracle_model, bsel, theta[frames])
    face_idx = marker_set.face_idx
    stats = {k: np.zeros(4) for k in ("fixed", "worst")}  # |pos - oracle|, angle, same for the old route
    err_face_o = 0.0
    with torch.no_grad():
        for i, f in enumerate(frames):
            vt = torch.as_tensor(v_o[i])
            st = stats["fixed" if f in fixed else "worst"]
            for m in sorted(set([0, 7, 19, 33, n - 1, int(np.argmax(d[f]))])):
                wm = w[0 if shared_weights else f, m]
                t = so.IkTask(int(face_idx[m]), normal_offset=offset, vertex_weights=torch.as_tensor(wm))
                ref_p = t.calc_actual_pos(oracle_model, vt).numpy()
                ref_n = t.calc_actual_normal(oracle_model, vt).numpy()
                st[:] = np.maximum(st, [np.abs(pos[f, m] - ref_p).max(), _angle(nrm[f, m], ref_n),
                                        np.abs(pos_old[f, m] - ref_p).max(), _angle(nrm_old[f, m], ref_n)])
                err_face_o = max(err_face_o, float(np.abs(pos[f, m] - offset * nrm[f, m] - (ref_p - offset * ref_n)).max()))
    print("offset %.3f: every frame: max |pos - old route| %.3g m (point on the face %.3g m), normal angle %.3g rad; "
          "oracle, fixed frames: |pos| %.3g m, normal %.3g rad (old route %.3g m, %.3g rad); frames of largest "
          "disagreement: |pos| %.3g m, normal %.3g rad (old route %.3g m, %.3g rad)"
          % ((offset, err_old, err_face, _angle(nrm, nrm_old).max()) + tuple(stats["fixed"]) + tuple(stats["worst"])))
    assert err_face_o <= TOL_VERTEX_M
    assert stats["fixed"][0] <= TOL_VERTEX_M
    assert stats["fixed"][1] <= NORMAL_TOL_RAD
    assert stats["worst"][0] <= max(TOL_VERTEX_M, stats["worst"][2])
    assert stats["worst"][1] <= max(NORMAL_TOL_RAD, stats["worst"][3])


def _grid_model(seed=11, side=9):
    """Small height-field mesh with DENSE skinning rows (24 non-zeros per vertex, sums != 1)."""
    from smplpp_b200 import synth
    rng = np.random.default_rng(seed)
    V = side * side
    ij = np.stack(np.meshgrid(np.arange(side), np.arange(side), indexing="ij"), -1).reshape(-1, 2)
    x, y = ij[:, 0] / (side - 1) - 0.5, ij[:, 1] / (side - 1) - 0.5
    templ = np.stack([0.6 * x, 0.6 * y, 0.05 * np.sin(3 * x) * np.cos(2 * y)], -1).astype(f32)
    faces = []
    for i in range(side - 1):
        for j in range(side - 1):
            a, b, c, d = i * side + j, (i + 1) * side + j, (i + 1) * side + j + 1, i * side + j + 1
            faces += [(a, b, c), (a, c, d)]
    tree = np.stack([synth.PARENTS.copy(), np.arange(24)])
    tree[0, 0] = 4294967295
    p = synth.SmplParams(
        face_indices=np.asarray(faces, np.int32) + 1, shape_blend_shapes=rng.normal(size=(V, 3, 10)).astype(f32) * 0.005,
        pose_blend_shapes=rng.normal(size=(V, 3, 207)).astype(f32) * 0.001, vertices_template=templ,
        joint_regressor=rng.dirichlet(np.ones(V), size=24).astype(f32), kinematic_tree=tree,
        weights=rng.uniform(0.1, 1.0, size=(V, 24)).astype(f32))
    return p, len(faces)


def test_dense_skinning_rows(rest_variant):
    """More than 4 influences per vertex: the compact rows of the task set carry all 24."""
    from smplpp_b200 import api, capi, synth
    p, nf = _grid_model()
    m = api.SMPL(p)
    assert capi.lib().smplpp_model_max_influences(m.handle) == 24
    face_idx = np.array([9, 20, 33, 47, 58, 64, 71, 90, 101], np.int64)
    assert face_idx.max() < nf
    tset = api.IkTaskSet(m, face_idx)
    beta, theta = synth.make_forward_inputs(300, 17)
    theta[:, 1:] *= 0.3
    w = _weights(len(face_idx), 300, 3)
    for offset in (0.0, 0.015):
        pos, nrm = tset.forward_positions(beta, theta, w, offset, want_normals=True)
        pos_old, nrm_old = _old_route(m, tset, beta, theta, w, offset)
        err = np.abs(pos.cpu().numpy() - pos_old).max()
        ang = _angle(nrm.cpu().numpy(), nrm_old).max()
        print("dense rows, offset %.3f: max |pos - old route| %.3g m, normal angle %.3g rad" % (offset, err, ang))
        assert err <= TOL_VERTEX_M
        assert ang <= NORMAL_TOL_RAD


@pytest.mark.parametrize("offset", [0.0, 0.015])
def test_host_entry_bitwise_and_batch_invariance(marker_set, poses, monkeypatch, offset):
    from smplpp_b200 import api
    beta, theta = poses
    n = marker_set.n
    w = _weights(n, BATCH, 9)
    pos_d, nrm_d = [a.cpu().numpy() for a in marker_set.forward_positions(beta, theta, w, offset, want_normals=True)]
    # bitwise batch invariance of the device entry: a frame alone gives the bytes it gets inside the batch
    for f in (0, 127, 128, 1000, BATCH - 1):
        p1, n1 = marker_set.forward_positions(beta[f:f + 1], theta[f:f + 1], w[f:f + 1], offset, want_normals=True)
        assert np.array_equal(p1.cpu().numpy()[0], pos_d[f]) and np.array_equal(n1.cpu().numpy()[0], nrm_d[f])
    # host entry: one chunk, then 1000-frame chunks (ragged last chunk), pageable and page-locked arrays
    for chunk in (None, "1000"):
        if chunk:
            monkeypatch.setenv("SMPLPP_TASK_CHUNK", chunk)
        ph, nh = marker_set.forward_positions_host(beta, theta, w, offset, want_normals=True)
        assert np.array_equal(ph, pos_d) and np.array_equal(nh, nrm_d)
        pb, pt, pw = api.pinned_empty(beta.shape), api.pinned_empty(theta.shape), api.pinned_empty(w.shape)
        pb[...], pt[...], pw[...] = beta, theta, w
        pp, pn = api.pinned_empty(pos_d.shape), api.pinned_empty(pos_d.shape)
        for _ in range(2):  # buffer reuse
            pp.fill(np.nan)
            pn.fill(np.nan)
            marker_set.forward_positions_host(pb, pt, pw, offset, want_normals=True, out_positions=pp, out_normals=pn)
            assert np.array_equal(pp, pos_d) and np.array_equal(pn, nrm_d)
        # positions only
        pp.fill(np.nan)
        marker_set.forward_positions_host(pb, pt, pw, offset, out_positions=pp)
        assert np.array_equal(pp, pos_d)
    # batch 1
    p1 = marker_set.forward_positions_host(beta[5:6], theta[5:6], w[5:6], offset)
    assert np.array_equal(p1[0], pos_d[5])
    # shared beta and shared weights (stride 0) against the device entry on the same inputs
    d_sh = marker_set.forward_positions(beta[:1], theta, w[0], offset).cpu().numpy()
    h_sh = marker_set.forward_positions_host(beta[:1], theta, w[0], offset)
    assert np.array_equal(d_sh, h_sh)
    assert np.array_equal(d_sh[3], marker_set.forward_positions(beta[0], theta[3:4], w[0], offset).cpu().numpy()[0])


def test_error_codes_and_texts(smpl_gpu, marker_set):
    from smplpp_b200 import api, capi
    L = capi.lib()
    dev = smpl_gpu.m__device
    n = marker_set.n
    B = 4
    beta = torch.zeros((B, 10), device=dev)
    theta = torch.zeros((B, 25, 3), device=dev)
    w = torch.full((B, n, 3), 1 / 3, device=dev)
    pos = torch.empty((B, n, 3), device=dev)
    need = L.smplpp_task_forward_workspace_bytes(marker_set._h, B)
    assert need > 0 and L.smplpp_task_forward_workspace_bytes(marker_set._h, 0) == 0
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    p = api._ptr
    stream = api._stream(dev)

    def call(batch=B, beta_p=p(beta), bstride=10, theta_p=p(theta), w_p=p(w), wstride=3 * n, pos_p=p(pos), nbytes=need):
        with torch.cuda.device(dev):
            return L.smplpp_task_forward(smpl_gpu.handle, marker_set._h, stream, batch, beta_p, bstride, theta_p, w_p,
                                         wstride, 0.015, pos_p, None, p(ws), nbytes)

    def expect(rc, text):
        assert rc == -1  # SMPLPP_ERR_INVALID
        assert text in L.smplpp_last_error().decode()

    assert call() == 0
    torch.cuda.synchronize()
    expect(call(pos_p=None), "IkTask Error: invalid task tensors!")
    expect(call(theta_p=None), "IkTask Error: invalid task tensors!")
    expect(call(beta_p=None), "IkTask Error: invalid task tensors!")
    expect(call(w_p=None), "IkTask Error: invalid task tensors!")
    expect(call(batch=0), "IkTask Error: invalid task tensors!")
    expect(call(bstride=5), "BlendShape Error: Failed to set beta!")
    expect(call(wstride=3), "vertex weights stride must be 0 or 3n")
    expect(call(nbytes=need - 1), "workspace too small")
    hb, ht, hw = np.zeros((B, 10), f32), np.zeros((B, 25, 3), f32), np.full((B, n, 3), 1 / 3, f32)
    hp = np.empty((B, n, 3), f32)

    def host(batch=B, theta_p=ht.ctypes.data, wstride=3 * n, pos_p=hp.ctypes.data):
        return L.smplpp_task_forward_host(smpl_gpu.handle, marker_set._h, batch, hb.ctypes.data, 10, theta_p,
                                          hw.ctypes.data, wstride, 0.0, pos_p, None)

    assert host() == 0
    expect(host(theta_p=None), "IkTask Error: invalid task tensors!")
    expect(host(pos_p=None), "IkTask Error: invalid task tensors!")
    expect(host(batch=0), "IkTask Error: invalid task tensors!")
    expect(host(wstride=3 * n + 3), "vertex weights stride must be 0 or 3n")
    # Python-level shape checks
    with pytest.raises(api.SmplppError, match="BlendShape Error: Failed to set beta!"):
        marker_set.forward_positions(np.zeros((B, 9), f32), ht, hw)
    with pytest.raises(api.SmplppError, match="IkTask Error: invalid task tensors!"):
        marker_set.forward_positions(hb, ht, np.zeros((2, n, 3), f32))


def _build_facade(out_dir):
    """g++ alone (the facade sits above the C ABI) into a scratch directory, so the tree can stay read-only."""
    exe = os.path.join(str(out_dir), "facade_task_forward")
    lib_dir = os.path.join(ROOT, "smplpp_b200")
    subprocess.check_call([os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-Wall", "-I" + os.path.join(ROOT, "include"),
                           FACADE_SRC, "-o", exe, "-L" + lib_dir, "-lsmplpp_b200", "-Wl,-rpath," + lib_dir])
    return exe


def test_cpp_facade_calc_actual_positions(tmp_path, params, golden_ik):
    """tests/cpp/facade_task_forward.cpp: smplpp::IkTaskSet::calcActualPositions against the reference golden."""
    exe = _build_facade(tmp_path)
    d = str(tmp_path)
    np.savez(os.path.join(d, "model.npz"), face_indices=params.face_indices, shape_blend_shapes=params.shape_blend_shapes,
             pose_blend_shapes=params.pose_blend_shapes, vertices_template=params.vertices_template,
             joint_regressor=params.joint_regressor, kinematic_tree=params.kinematic_tree, weights=params.weights)
    k = golden_ik
    np.ascontiguousarray(k["face_idx"], dtype=np.int64).tofile(os.path.join(d, "ik_face_idx.i64"))
    for key in ("theta_in", "beta_in", "motion_vertex_weights_out", "motion_actual_pos"):
        np.ascontiguousarray(k[key], dtype=f32).tofile(os.path.join(d, "ik_%s.f32" % key))
    r = subprocess.run([exe, d], capture_output=True, text=True, timeout=600)
    print(r.stdout)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "facade task forward: OK" in r.stdout and "FAIL" not in r.stdout
