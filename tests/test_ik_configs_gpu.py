"""GPU parity of the IK path at the BASELINE configs against multi-frame, multi-iteration goldens of the compiled
reference (tests/golden/ref_ik_configs.npz, made by tests/golden/make_ref_golden_ik_configs.py):

  configs[2]  MoSh direct: 8 frames x 30 iterations (node.cpp:753-968 looped), residual trajectory + final theta
  configs[3]  MoSh++ VPoser: 4 frames x 10 iterations
  shared-beta stage with 16 frames (direct and VPoser) against the stored dense float64 solve of the block-arrow system
  built from the reference's per-frame Jacobians
  the host-buffer call smplpp_ik_solve_host against the device loop
"""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, TOL_RESIDUAL_M

pytestmark = pytest.mark.gpu
f32 = np.float32
MOTION = dict(normal_task_weight=0.0, phi_limit=0.0, normal_offset=0.015, optimize_beta=0, enable_qp=1, enable_phi=0)


def cu(a, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device="cuda:0").contiguous()


@pytest.fixture(scope="module")
def gc():
    return dict(np.load(os.path.join(GOLDEN, "ref_ik_configs.npz")))


@pytest.fixture(scope="module")
def task_set(smpl_gpu, marker_tasks, vposer_params):
    from smplpp_b200 import api
    _, face_idx, _ = marker_tasks
    return api.IkTaskSet(smpl_gpu, face_idx, vposer=api.VPoserDecoder(vposer_params))


def marker_residual(e, valid):
    r = np.linalg.norm(e.reshape(e.shape[0], -1, 4)[:, :, :3], axis=2)
    return (r * valid).sum(1) / valid.sum(1)


def run_trajectory(task_set, opt, x0, beta, vw0, target, valid, iters):
    F = target.shape[0]
    theta = cu(np.repeat(x0[None], F, axis=0))
    vw = cu(np.repeat(vw0[None], F, axis=0))
    beta_d, tgt, pw = cu(beta), cu(target), cu(valid)
    res, traj = [], []
    for _ in range(iters):
        status, out = task_set.step(opt, theta, beta_d, vw, tgt, pos_task_weight=pw, outputs=True)
        assert (status == 0).all()
        res.append(marker_residual(out["e"].cpu().numpy(), valid))
        traj.append(theta.cpu().numpy().copy())
    return np.stack(res, 1), np.stack(traj, 1), vw.cpu().numpy()


def teacher_forced(task_set, opt, gc, prefix, theta_dim):
    """Every (frame, iteration) of the golden trajectory as ONE batch element: iteration k starts from the compiled
    reference's own state after iteration k-1, so each step is an independent parity check along the real trajectory."""
    th, vw, res = gc[prefix + "_theta_traj"], gc[prefix + "_vertex_weights_traj"], gc[prefix + "_residual"]
    F, K = res.shape
    n = vw.shape[2]
    th_in = np.concatenate([np.repeat(gc[prefix + "_theta_in"][None, None], F, axis=0), th[:, :-1]], axis=1)
    vw_in = np.concatenate([np.repeat(gc["vertex_weights_in"][None, None], F, axis=0), vw[:, :-1]], axis=1)
    theta, w = cu(th_in.reshape(F * K, theta_dim)), cu(vw_in.reshape(F * K, n, 3))
    tgt = cu(np.repeat(gc[prefix + "_target"][:, None], K, axis=1).reshape(F * K, n, 3))
    valid = np.repeat(gc[prefix + "_valid"][:, None], K, axis=1).reshape(F * K, n)
    status, out = task_set.step(opt, theta, cu(gc["beta"]), w, tgt, pos_task_weight=cu(valid), outputs=True)
    assert (status == 0).all()
    r = marker_residual(out["e"].cpu().numpy(), valid).reshape(F, K)
    th_out = theta.cpu().numpy().reshape(F, K, theta_dim)
    # the two updates compared where the markers can see them: J (theta_gpu - theta_ref) in metres.  (theta itself is
    # only determined up to the weakly observed directions, where rounding in b is amplified by 1 / (1e-3 + |e|^2).)
    J = out["J"].cpu().numpy().astype(np.float64)[:, :, :theta_dim]
    dth = (th_out - th).reshape(F * K, theta_dim).astype(np.float64)
    marker_space = np.abs(np.einsum("brc,bc->br", J, dth)).max()
    return r, th_out, w.cpu().numpy().reshape(F, K, n, 3), marker_space


def test_config3_every_iteration_vs_reference(task_set, gc, ik_variant):
    """BASELINE configs[2], 8 frames x 30 iterations of the compiled reference, teacher-forced: the residual of every
    (frame, iteration) within 1e-5 m, the updated theta and re-weighted attachments of every step."""
    from smplpp_b200 import api
    res, th, vw, marker_space = teacher_forced(task_set, api.ik_options(**MOTION), gc, "c3", 75)
    assert np.abs(res - gc["c3_residual"]).max() < 1e-5
    assert marker_space < TOL_RESIDUAL_M                         # the two updates agree to 0.1 mm at the markers
    assert np.abs(th - gc["c3_theta_traj"]).max() < 1e-3
    assert np.abs(vw - gc["c3_vertex_weights_traj"]).max() < 2e-4


def test_config3_free_running_30_iterations(task_set, gc):
    """The same 30 iterations free-running on the GPU.  The iteration is not contractive along weakly observed joints
    (damping 1e-3 only): two runs of the COMPILED REFERENCE that differ only in the libtorch thread count drift apart by
    up to `band` (2e-4 m of residual, 0.08 rad; golden c3_alt_*).  Frame 4 shows what that means: its residual bounces
    between 1.49 and 1.67 mm from iteration 8 on before it drops into the converged 1.46 mm, and rounding decides when -
    iteration 19 in the reference run, 27 in its other-thread-count twin, 19 / 30 in the two GPU variants of the pose-blend
    columns (scripts/diag_pb.py).  The GPU run must stay inside the band during the 30 iterations, track the reference to
    1e-5 m while the trajectories still coincide, and - run on until every frame has settled - reach the reference's
    converged residual within 1e-4 m."""
    from smplpp_b200 import api
    opt = api.ik_options(**MOTION)
    K = gc["c3_residual"].shape[1]
    res, traj, vw = run_trajectory(task_set, opt, gc["c3_theta_in"], gc["beta"], gc["vertex_weights_in"], gc["c3_target"],
                                   gc["c3_valid"], 2 * K)
    alt = gc["c3_alt_frames"]
    band = np.abs(gc["c3_alt_residual"] - gc["c3_residual"][alt]).max()
    dev = np.abs(res[:, :K] - gc["c3_residual"])
    conv = np.abs(res[:, -1] - gc["c3_residual"][:, -1])
    print("free-running residual deviation %.2e m (reference vs itself: %.2e m), converged residual deviation %.2e m"
          % (dev.max(), band, conv.max()))
    assert dev[:, :3].max() < 1e-5
    assert dev.max() < max(TOL_RESIDUAL_M, 1.5 * band)
    assert conv.max() < TOL_RESIDUAL_M                            # converged marker residual within 1e-4 m
    assert np.abs(res[:, -1] - res[:, -5]).max() < TOL_RESIDUAL_M # ... and stays there
    assert np.abs(traj[:, 0] - gc["c3_theta_traj"][:, 0]).max() < 2e-4
    assert res[:, -1].max() < 0.25 * res[:, 0].min()


def test_config4_vposer_every_iteration_vs_reference(task_set, gc, ik_variant):
    """BASELINE configs[3] (per-frame part), 4 frames x 10 iterations, teacher-forced: VPoser latent state, decoder and
    its Jacobian inside the step."""
    from smplpp_b200 import api
    res, th, vw, marker_space = teacher_forced(task_set, api.ik_options(enable_vposer=1, **MOTION), gc, "c4", 44)
    assert np.abs(res - gc["c4_residual"]).max() < 2e-5
    # steps of 0.1 .. 0.5 in the latent at residuals of 3 .. 40 cm, through a decoder Jacobian that is accurate to 2e-4
    # where a decoded joint angle comes close to pi (tests/test_vposer_gpu.py): 0.3 mm at the markers
    assert marker_space < 3e-4
    assert np.abs(th - gc["c4_theta_traj"]).max() < 1e-3
    assert np.abs(vw - gc["c4_vertex_weights_traj"]).max() < 5e-4


def test_config4_vposer_free_running(task_set, gc):
    from smplpp_b200 import api
    opt = api.ik_options(enable_vposer=1, **MOTION)
    K = gc["c4_residual"].shape[1]
    res, traj, _ = run_trajectory(task_set, opt, gc["c4_theta_in"], gc["beta"], gc["vertex_weights_in"], gc["c4_target"],
                                  gc["c4_valid"], K)
    dev = np.abs(res - gc["c4_residual"])
    # The same loop of the compiled reference with ONE libtorch thread instead of eight (c4_alt_*,
    # tests/golden/make_ref_golden_c4_alt.py): far from convergence (residual of centimetres after 10 heavily damped steps
    # through a random decoder) rounding is amplified from iteration to iteration, and the reference's own two runs end
    # 3 cm (88 %) apart on frame 2.  The GPU trajectory has to coincide with the reference while rounding has not been
    # amplified yet and stay inside that band afterwards; parity of every single step is test_config4_*_every_iteration.
    band = np.abs(gc["c4_alt_residual"] - gc["c4_residual"])
    print("VPoser free-running residual deviation %.2e m (residual level %.3f m; reference vs itself %.2e m, relative %.2f)"
          % (dev.max(), gc["c4_residual"][:, -1].max(), band.max(), (band / gc["c4_residual"]).max()))
    assert dev[:, :4].max() < 5e-5
    assert dev.max() < 1.5 * band.max()
    assert (dev / gc["c4_residual"]).max() < max(0.25, 1.5 * (band / gc["c4_residual"]).max())
    assert np.abs(traj[:, 0] - gc["c4_theta_traj"][:, 0]).max() < 5e-4


def test_solve_host_equals_device_loop(task_set, gc):
    """smplpp_ik_solve_host (host arrays in / out, K iterations inside) == K calls of smplpp_ik_step."""
    from smplpp_b200 import api
    opt = api.ik_options(**MOTION)
    K = 5
    F = gc["c3_target"].shape[0]
    res, traj, vw = run_trajectory(task_set, opt, gc["c3_theta_in"], gc["beta"], gc["vertex_weights_in"], gc["c3_target"],
                                   gc["c3_valid"], K)
    theta_h = np.repeat(gc["c3_theta_in"][None], F, axis=0).astype(f32)
    vw_h = np.repeat(gc["vertex_weights_in"][None], F, axis=0).astype(f32)
    status, r = task_set.solve_host(opt, K, theta_h, gc["beta"].astype(f32), vw_h, gc["c3_target"].astype(f32),
                                    pos_task_weight=gc["c3_valid"].astype(f32))
    assert (status == 0).all()
    assert np.array_equal(theta_h, traj[:, -1])
    assert np.array_equal(vw_h, vw)
    assert np.abs(r - res[:, -1]).max() < 1e-6


@pytest.fixture(params=[(401, 410, 420), (401, 411, 421), (402, 410, 420)], ids=["two_kernels", "two_kernels_ffma_variants", "fused_kernel"])
def ik_variant(request):
    from smplpp_b200 import capi
    # 401 / 402: ik_jacobian_kernel + solve kernel / fused kernel; 410 / 411: ik_solve_mma_kernel (fp64 tensor cores, the
    # default where the problem shape allows) / the scalar ik_solve_kernel; 420 / 421: pose-blend columns of J by
    # ik_poseblend_tc_kernel (tcgen05, the default) / by the FFMA phase of ik_jacobian_kernel
    for v in request.param:
        capi.check(capi.lib().smplpp_set_forward_variant(v))
    yield request.param[0]
    for v in (400, 410, 420):
        capi.check(capi.lib().smplpp_set_forward_variant(v))


@pytest.mark.parametrize("mode", ["direct", "vposer"])
def test_shared_beta_16_frames_vs_dense_solve(task_set, gc, mode, ik_variant):
    """One shared-beta step over 16 frames against the float64 box-QP solution of the dense block-arrow system built
    from the reference's per-frame e and J (stored as sb_x / sb_x_vposer by make_ref_golden_ik_configs.py)."""
    from smplpp_b200 import api
    vposer = mode == "vposer"
    x = gc["sb_x_vposer" if vposer else "sb_x"]
    x_in = gc["sb_state_in" if vposer else "sb_theta_in"].astype(f32)
    F, D = x_in.shape
    opt = api.ik_options(enable_vposer=int(vposer), **MOTION)
    theta = cu(x_in)
    sbeta = cu(np.zeros(10, f32))
    vw = cu(np.repeat(gc["vertex_weights_in"][None], F, axis=0))
    status = task_set.shared_beta_step(opt, theta, sbeta, vw, cu(gc["sb_target"]), pos_task_weight=cu(gc["sb_valid"]))
    assert (status == 0).all()
    dbeta = sbeta.cpu().numpy().astype(np.float64)
    dtheta = (theta.cpu().numpy() - x_in).astype(np.float64)
    assert np.abs(dbeta - x[F * D:]).max() < 2e-4
    assert np.abs(dtheta - x[:F * D].reshape(F, D)).max() < 5e-4
    assert (np.abs(dbeta) <= 0.5 + 1e-6).all()


def test_even_task_vertex_count_vs_oracle(smpl_gpu, oracle_model, marker_tasks):
    """A task set whose vertex count is EVEN and >= 128: the compact sub-model must never reach the tensor-core
    skinning kernel (which indexes the full model's dense weights)."""
    from oracle import smpl_oracle as so
    from smplpp_b200 import api, synth
    _, face_idx, vw0 = marker_tasks
    ts = None
    for k in range(11, len(face_idx) + 1):
        cand = api.IkTaskSet(smpl_gpu, face_idx[:k])
        if cand.vertex_count >= 128 and cand.vertex_count % 2 == 0:
            ts = cand
            break
    assert ts is not None, "no prefix of the marker list has an even vertex count >= 128"
    n = ts.n
    gt = synth.make_motion(12, 20)
    beta = (np.random.default_rng(5).normal(size=10) * 0.5).astype(f32)
    smpl_gpu.launch(beta, gt[9:10])
    w0 = cu(vw0[None, :n])
    target = ts.positions(smpl_gpu.getVertex(), w0, 0.015).contiguous()
    opt = api.ik_options(skip_if_too_few=0, **MOTION)
    theta, vw = cu(gt[:1].reshape(1, 75)), w0.clone()
    status, out = ts.step(opt, theta, cu(beta), vw, target, outputs=True)
    assert int(status[0]) == 0
    tgt_h = target.cpu().numpy()[0]
    tasks = [so.IkTask(int(face_idx[i]), target_pos=torch.as_tensor(tgt_h[i]), normal_task_weight=0.0, phi_limit=0.0,
                       normal_offset=0.015, vertex_weights=torch.as_tensor(vw0[i])) for i in range(n)]
    r = so.ik_iteration(oracle_model, tasks, gt[0].reshape(-1), beta)
    assert np.abs(out["e"][0].cpu().numpy() - r.e).max() < 1e-5
    J = out["J"][0].cpu().numpy()
    assert np.abs(J - r.J).max() / np.abs(r.J).max() < 1e-4
    assert np.abs(theta[0].cpu().numpy() - r.theta_state).max() < 2e-4


# ----------------------------------------------------------------------------------------------------------------
# body stage (node.cpp:652-656, 695-700, 1349): 51 iterations of ONE frame, VPoser state, beta and phi from iteration 25,
# the attachment re-seated after every iteration (faces change on this mesh in almost every iteration)
# ----------------------------------------------------------------------------------------------------------------
def body_options(api, late):
    return api.ik_options(enable_vposer=1, skip_if_too_few=0, normal_task_weight=0.0, normal_offset=0.015,
                          phi_limit=0.04 if late else 0.0, enable_phi=1 if late else 0, optimize_beta=1 if late else 0, enable_qp=1)


def test_body_stage_every_iteration_vs_reference(task_set, gc, smpl_gpu):
    """Teacher-forced: iteration k starts from the compiled reference's state after iteration k-1 (theta, beta, faces,
    weights), so each of the 51 iterations is an independent parity check of the COMPLETE loop body - step on per-frame
    attachments, projection onto the pre-update mesh, re-seated faces and weights - including all the face changes."""
    from smplpp_b200 import api
    n = task_set.n
    K = gc["body_theta"].shape[0]
    th_in = np.concatenate([gc["body_theta_in"][None], gc["body_theta"][:-1]]).astype(f32)
    be_in = np.concatenate([np.zeros((1, 10), f32), gc["body_beta"][:-1]]).astype(f32)
    fa_in = np.concatenate([gc["face_idx"][None], gc["body_face"][:-1]]).astype(np.int32)
    vw_in = np.concatenate([np.full((1, n, 3), 1.0 / 3.0, f32), gc["body_vw"][:-1]]).astype(f32)
    changed = 0
    for lo, hi, late in ((0, 25, False), (25, K, True)):
        B = hi - lo
        opt = body_options(api, late)
        theta, beta = cu(th_in[lo:hi]), cu(be_in[lo:hi])
        vw, face = cu(vw_in[lo:hi]), cu(fa_in[lo:hi], torch.int32)
        tgt = cu(np.repeat(gc["body_target"][None], B, axis=0))
        status, out = task_set.iterate(opt, theta, beta, vw, face, tgt, outputs=True)
        assert (status == 0).all()
        res = marker_residual(out["e"].cpu().numpy(), np.ones((B, n), f32))
        assert np.abs(res - gc["body_res"][lo:hi]).max() < 1e-5          # same state in, same residual
        assert np.abs(theta.cpu().numpy() - gc["body_theta"][lo:hi]).max() < 5e-4
        assert np.abs(beta.cpu().numpy() - gc["body_beta"][lo:hi]).max() < 5e-4
        # re-seated attachment: same face (ties between neighbouring faces aside) and the same point on the mesh
        f_gpu, f_ref = face.cpu().numpy(), gc["body_face"][lo:hi]
        agree = f_gpu == f_ref
        assert agree.mean() >= 0.97
        changed += int((f_ref != fa_in[lo:hi]).sum())
        # the point the weights reproduce on the pre-update mesh against the reference's closest point; where the two
        # picked different faces (a point above a ridge is equally far from both) the DISTANCE must agree instead
        smpl_gpu.launch(be_in[lo:hi], task_set.assemble_theta(cu(th_in[lo:hi])))
        verts = smpl_gpu.getVertex().cpu().numpy().astype(np.float64)
        faces0 = smpl_gpu._faces_host.astype(np.int64) - 1
        tri = verts[np.arange(B)[:, None, None], faces0[f_gpu]]           # (B, n, 3, 3)
        pt = (vw.cpu().numpy()[..., None].astype(np.float64) * tri).sum(2)
        ref_pt, src = gc["body_closest"][lo:hi], gc["body_point"][lo:hi].astype(np.float64)
        # (from iteration 25 on the projected point itself moves by tangents * dphi, so the step's own tolerance of
        # 2e-4 applies to it; typical deviations are micrometres)
        err = np.linalg.norm(pt - ref_pt, axis=2)[agree]
        assert np.quantile(err, 0.95) < 2e-5 and err.max() < 2.5e-4
        d_gpu, d_ref = np.linalg.norm(pt - src, axis=2), np.linalg.norm(ref_pt - src, axis=2)
        assert np.abs(d_gpu - d_ref).max() < 2.5e-4
        assert np.abs(vw.cpu().numpy()[agree] - gc["body_vw"][lo:hi][agree]).max() < 2e-3
    assert changed > 200  # the golden trajectory really exercises re-seated faces


def test_body_stage_free_running(task_set, gc):
    """The same 51 iterations free-running on the GPU: beta and phi switch on at iteration 25, attachments wander over
    the mesh."""
    from smplpp_b200 import api
    n = task_set.n
    K = gc["body_theta"].shape[0]
    theta, beta = cu(gc["body_theta_in"][None]), cu(np.zeros((1, 10), f32))
    vw, face = cu(np.full((1, n, 3), 1.0 / 3.0, f32)), cu(gc["face_idx"][None], torch.int32)
    tgt = cu(gc["body_target"][None])
    res = []
    for k in range(K):
        status, out = task_set.iterate(body_options(api, k >= 25), theta, beta, vw, face, tgt, outputs=True)
        assert int(status[0]) == 0
        res.append(marker_residual(out["e"].cpu().numpy(), np.ones((1, n), f32))[0])
    res = np.asarray(res)
    print("body stage residual: gpu %.5f -> %.5f m, reference %.5f -> %.5f m, max deviation %.2e m, faces equal at the end: %d / %d"
          % (res[0], res[-1], gc["body_res"][0], gc["body_res"][-1], np.abs(res - gc["body_res"]).max(),
             int((face.cpu().numpy()[0] == gc["body_face"][-1]).sum()), n))
    # this synthetic body stage (random decoder, |e|^2 damping of ~2.5) does not settle in 51 iterations in the compiled
    # reference either (0.25 -> 0.11 -> 0.17 -> 0.13 m): per-iteration parity is the teacher-forced test above, here the
    # whole loop must run through (status 0 everywhere), stay bounded and end at the reference's residual level
    assert np.isfinite(res).all() and abs(res[0] - gc["body_res"][0]) < 1e-5
    assert abs(res[1] - gc["body_res"][1]) < 1e-2
    assert 0.5 * gc["body_res"].min() < res.min() and res.max() < 1.5 * gc["body_res"].max()
    assert abs(res[-1] - gc["body_res"][-1]) < 0.05
    assert np.abs(beta.cpu().numpy()[0]).max() <= 0.5 * 26 + 1e-3 and np.isfinite(theta.cpu().numpy()).all()
