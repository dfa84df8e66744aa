"""The bounded solve of the IK step against a float64 KKT certificate, and the shared-beta stage against the block-arrow
system it reduces.

Every bounded IK step solves min 1/2 d'Ad + b'd over a box (|phi| <= phi_limit, |dbeta| <= delta_beta_limit) with a primal
active-set iteration written three times: ik_solve_kernel (two-kernel path; every bounded configuration, the fp64
tensor-core solve declines a QP), the QP phase of the fused kernel (variant 402 and smplpp_ik_step_faces) and
shared_beta_qp_kernel (the 10-unknown shared-beta QP).  The tests judge each result on the GPU's own float64 A and b (the
step's outputs), so the linearisation, which tests/test_ik_linearisation_gpu.py checks, is not measured again:

  - every frame: status 0, and tests/box_qp_ref.py's kkt_certificate holds on (A, b, delta);
  - frames 0, 31, 32, 127, 128, 129: f(delta) exceeds the objective of scipy's bvls (an independent solver) by at most
    1e-12 (|f| + s ||delta||);
  - the update is the one the kernels define: theta_out == f32(theta_in + f32(delta_theta)) bitwise, the same for
    per-frame beta, and dphi_out == f32(delta_phi) on the per-frame-faces path;
  - the paths that share their inputs agree on every bound whose multiplier exceeds 1e-8 s.

130 frames give partial blocks to the 32-frame CTAs, the 128-frame tiles and the fused kernel's padding teams.  Paths (the
variants of smplpp_set_forward_variant):
  default 400 410 420 | ffma 401 411 421 | fused 402 410 420 | faces: smplpp_ik_step_faces, per-frame random faces
"""
from __future__ import annotations

import numpy as np
import pytest
import torch

import box_qp_ref as q
import test_ik_linearisation_gpu as lin

pytestmark = pytest.mark.gpu
f32 = np.float32
B = lin.B  # 130
FRAMES6 = lin.FRAMES6
PATHS = ("default", "ffma", "fused", "faces")
MOTION = lin.MOTION
BODY = dict(MOTION, enable_vposer=1, enable_phi=1, phi_limit=0.004, optimize_beta=1, delta_beta_limit=0.05,
            normal_task_weight=1.0, normal_offset=0.0)

# name: (options, seed, pos_task_weight scale, beta state / target: None, or the sigma of beta_true with beta_0 = 0)
CONFIGS = {
    "phi_all": (dict(MOTION, enable_phi=1, phi_limit=1e-4), 31, 1.0, None),
    "phi_none": (dict(MOTION, enable_phi=1, phi_limit=1.0), 32, 1.0, None),
    "phi_degenerate": (dict(MOTION, enable_phi=1), 32, 1.0, None),  # phi_limit from phi_none (same inputs)
    # the ||e||^2 damping keeps |dbeta| of the unbounded step small on these inputs: 1e-4 binds nearly every component
    "beta_tight": (dict(MOTION, optimize_beta=1, delta_beta_limit=1e-4), 34, 1.0, 1.5),
    "beta_pinned": (dict(MOTION, optimize_beta=1, delta_beta_limit=0.0), 35, 1.0, 1.5),
    "body_mixed": (BODY, 36, 1.0, None),  # D = 44 + 82 + 10 = 136 with the normal rows
    "scaled_up": (BODY, 36, 1e3, None),
    "scaled_down": (BODY, 36, 1e-3, None),
}
CASES = [(c, p) for c in CONFIGS for p in PATHS]
TABLE = []
RESULTS = {}


def theta_dim(opts):
    return 44 if opts.get("enable_vposer") else 75


@pytest.fixture(scope="module")
def handles(params, vposer_params, smpl_gpu):
    from smplpp_b200 import api
    yield params, smpl_gpu, api.VPoserDecoder(vposer_params)
    print("\n%-15s %-8s %22s %14s %14s" % ("configuration", "path", "active min/med/max", "worst KKT", "worst gap/tol"))
    for row in TABLE:
        print("%-15s %-8s %22s %14.3g %14.3g" % row)


def _targets(smpl, ts, faces, beta, pose, vw, rng):
    """Markers of (beta, pose) on the shared task set, or on every frame's own faces (faces (B, n)), plus 5 mm noise."""
    if faces.ndim == 2:
        tgt = np.empty(vw.shape, f32)
        for b in range(vw.shape[0]):
            tgt[b] = lin._task_set(smpl, faces[b]).forward_positions(beta[b:b + 1], pose[b:b + 1], vw[b:b + 1],
                                                                     0.015)[0].cpu().numpy()
    else:
        tgt = ts.forward_positions(beta, pose, vw, 0.015).cpu().numpy()
    return tgt + rng.normal(scale=0.005, size=tgt.shape).astype(f32)


_PREP = {}


def prepared(name, handles, faces_path):
    """(opts, task set, inputs) of one configuration; the faces path gets its own inputs with per-frame faces."""
    key = (name, faces_path)
    if key in _PREP:
        return _PREP[key]
    from smplpp_b200 import synth
    params, smpl, vposer = handles
    opts, seed, pw_scale, beta_sigma = CONFIGS[name]
    opts = dict(opts)
    if name == "phi_degenerate":
        # the float32 median |phi| of phi_none's frame 0: about half of the phi bounds bind, and the median component's
        # unconstrained optimum sits on its bound
        o, ts0, inp0 = prepared("phi_none", handles, faces_path)
        d = run(o, ts0, inp0, "faces" if faces_path else "default")["delta"][0]
        phi = np.sort(np.abs(d[75:75 + 2 * ts0.n]))
        opts["phi_limit"] = float(f32(phi[len(phi) // 2]))
    cfg = lin.Cfg("random", opts, seed=seed, per_frame_faces=faces_path)
    rng = np.random.default_rng(cfg.seed)
    ts = lin._task_set(smpl, lin.task_faces(cfg, params, rng), vposer if cfg.vposer else None)
    inp = lin.make_inputs(cfg, params, smpl, ts)
    if beta_sigma is not None:
        # beta_0 = 0 against targets of beta_true ~ N(0, sigma^2) on the target pose of make_inputs
        r = np.random.default_rng(500 + seed)
        beta_true = (r.normal(size=(B, 10)) * beta_sigma).astype(f32)
        pose = synth.make_motion(B, 20 + cfg.seed).astype(f32)
        inp.tgt = _targets(smpl, ts, inp.faces, beta_true, pose, inp.vw, r)
        inp.beta = np.zeros((B, 10), f32)
    if pw_scale != 1.0:
        inp.pw = np.full((B, ts.n), pw_scale, f32)
    _PREP[key] = (opts, ts, inp)
    return _PREP[key]


def run(opts, ts, inp, path):
    """One step of all frames on `path`; host copies of status, A, b, delta, the updated state and dphi_out (faces)."""
    from smplpp_b200 import api
    opt = api.ik_options(skip_if_too_few=0, **opts)
    theta, beta, vw = lin.cu(inp.theta), lin.cu(inp.beta), lin.cu(inp.vw)
    face = dphi = None
    if path == "faces":
        face = lin.cu(inp.faces, torch.int32)
        dphi = torch.full((B, ts.n, 2), float("nan"), dtype=torch.float32, device="cuda:0")
    lin.set_variant(lin.VARIANTS[path])
    try:
        status, out = ts.step(opt, theta, beta, vw, lin.cu(inp.tgt),
                              pos_task_weight=lin.cu(inp.pw) if inp.pw is not None else None,
                              target_normal=lin.cu(inp.tn) if inp.tn is not None else None, outputs=True, face_idx=face,
                              dphi_out=dphi)
    finally:
        lin.set_variant(lin.DEFAULT_VARIANT)
    res = {k: out[k].cpu().numpy() for k in ("A", "b", "delta")}
    res.update(status=status.cpu().numpy(), theta=theta.cpu().numpy(), beta=beta.cpu().numpy(),
               dphi=None if dphi is None else dphi.cpu().numpy())
    return res


def check_update(opts, n, inp, out):
    """theta_out == f32(theta_in + f32(delta_theta)) bitwise (ik.cu / ik2.cu, node.cpp:946-968), the same for per-frame
    beta; beta is untouched without beta columns."""
    td = theta_dim(opts)
    d = out["delta"]
    assert np.array_equal(out["theta"], inp.theta + d[:, :td].astype(f32))
    if opts.get("optimize_beta"):
        assert np.array_equal(out["beta"], inp.beta + d[:, td + 2 * n:].astype(f32))
    else:
        assert np.array_equal(out["beta"], inp.beta)
    if out["dphi"] is not None:
        assert np.array_equal(out["dphi"].reshape(B, 2 * n), d[:, td:td + 2 * n].astype(f32))


@pytest.mark.parametrize("config,path", CASES, ids=["%s-%s" % c for c in CASES])
def test_bounded_step_is_optimal(handles, config, path):
    opts, ts, inp = prepared(config, handles, path == "faces")
    n, td = ts.n, theta_dim(opts)
    out = run(opts, ts, inp, path)
    if path != "faces":  # the cross-path comparison below takes the paths that share their inputs
        RESULTS[(config, path)] = out
    assert (out["status"] == 0).all(), np.unique(out["status"], return_counts=True)  # 3 (iteration cap) is a failure
    dim = out["A"].shape[1]
    lo, hi = q.ik_bounds(opts, n, dim, td)
    blocks = q.ik_blocks(td, n, dim)
    fails, ratios, active = [], [], []
    for f in range(B):
        A, b, d = out["A"][f], out["b"][f], out["delta"][f]
        ok, rep = q.kkt_certificate(A, b, d, lo, hi, blocks)
        ratios.append(rep["worst_ratio"])
        active.append(rep["n_upper"] + rep["n_lower"])
        if not ok:
            fails.append("frame %d: %s" % (f, rep["worst"]))
    gaps = []
    for f in FRAMES6:
        A, b, d = out["A"][f], out["b"][f], out["delta"][f]
        x_ref = q.reference_box_qp(A, b, lo, hi)
        gap = q.objective(A, b, d) - q.objective(A, b, x_ref)
        gaps.append(gap / q.objective_gap_tol(A, b, d))
        if gap > q.objective_gap_tol(A, b, d):
            fails.append("frame %d: f(delta) - f(bvls) = %.3g, allowed %.3g" % (f, gap, q.objective_gap_tol(A, b, d)))
    active = np.array(active)
    TABLE.append((config, path, "%d/%d/%d" % (active.min(), np.median(active), active.max()), max(ratios), max(gaps)))
    print("%s %s: active %d/%d/%d, worst KKT ratio %.3g, worst objective gap / tol %.3g"
          % (config, path, active.min(), np.median(active), active.max(), max(ratios), max(gaps)))
    assert not fails, fails[:10]
    check_update(opts, n, inp, out)
    # what each configuration is there for
    phi = out["delta"][:, td:td + 2 * n]
    nphi_act = (np.abs(phi) >= float(f32(opts.get("phi_limit", 0.0)))).sum(1) if opts.get("enable_phi") else None
    if config == "phi_all":
        assert np.median(nphi_act) >= 0.9 * 2 * n, nphi_act
    elif config == "phi_none":
        assert active.max() == 0
        for f in range(B):
            d_chk = -np.linalg.solve(out["A"][f], out["b"][f])
            assert np.abs(out["delta"][f] - d_chk).max() <= 1e-9 * np.abs(d_chk).max(), f
    elif config == "phi_degenerate":
        assert 0.2 * 2 * n <= nphi_act[0] <= 0.8 * 2 * n, nphi_act[0]
    elif config == "beta_tight":
        nb = (np.abs(out["delta"][:, td + 2 * n:]) == float(f32(opts["delta_beta_limit"]))).sum(1)
        assert np.median(nb) >= 9 and nb.min() >= 5, nb
    elif config == "beta_pinned":
        assert (out["delta"][:, td + 2 * n:] == 0.0).all() and np.array_equal(out["beta"], inp.beta)
        th = slice(0, td)
        for f in range(B):
            d_chk = -np.linalg.solve(out["A"][f][th, th], out["b"][f][th])
            assert np.abs(out["delta"][f][th] - d_chk).max() <= 1e-9 * np.abs(d_chk).max(), f
    elif config in ("body_mixed", "scaled_up", "scaled_down"):
        assert np.median(active) >= 1


@pytest.mark.parametrize("config", list(CONFIGS))
def test_active_sets_agree_across_paths(handles, config):
    """default, ffma and fused run on the same inputs: wherever a bound's multiplier exceeds 1e-8 s on either path, both
    have that unknown at the same bound (A and b differ between the paths in the last bits only)."""
    opts, ts, inp = prepared(config, handles, False)
    n, td = ts.n, theta_dim(opts)
    outs = {p: RESULTS.get((config, p)) or run(opts, ts, inp, p) for p in ("default", "ffma", "fused")}
    dim = outs["default"]["A"].shape[1]
    lo, hi = q.ik_bounds(opts, n, dim, td)
    bad = []
    for f in range(B):
        sides, strong = {}, {}
        for p, o in outs.items():
            A, b, d = o["A"][f], o["b"][f], o["delta"][f]
            sides[p] = q.active_set(d, lo, hi)
            strong[p] = q.multipliers(A, b, d, lo, hi) > 1e-8 * q.problem_scale(A, b, d)
        for p in ("ffma", "fused"):
            m = strong["default"] | strong[p]
            diff = np.nonzero(m & (sides["default"] != sides[p]))[0]
            if diff.size:
                bad.append("frame %d, %s vs default: unknowns %s" % (f, p, diff[:8].tolist()))
    assert not bad, bad[:10]


def test_largest_task_set_bounded(handles):
    """phi and beta bounds on the largest random task set the two-kernel step accepts (bisection on its return code):
    one face more is refused with SMPLPP_ERR_INVALID and one of the documented texts, the largest one's bounded solve
    passes the certificate, and a normal step runs afterwards."""
    from smplpp_b200 import api, capi, synth
    params, smpl, _ = handles
    opts = dict(MOTION, enable_phi=1, phi_limit=0.004, optimize_beta=1, delta_beta_limit=0.05)
    opt = api.ik_options(skip_if_too_few=0, **opts)
    order = np.random.default_rng(78).permutation(params.face_indices.shape[0]).astype(np.int64)
    nf = 3

    def attempt(n, outputs=False):
        ts = lin._task_set(smpl, order[:n])
        rng = np.random.default_rng(n)
        theta = synth.make_motion(nf, 56).reshape(nf, 75).astype(f32)
        theta[:, 3:] += rng.normal(scale=0.05, size=(nf, 72)).astype(f32)
        vw = rng.dirichlet(np.ones(3), size=(nf, n)).astype(f32)
        beta = np.zeros((nf, 10), f32)
        tgt = ts.forward_positions((rng.normal(size=(nf, 10)) * 0.5).astype(f32), synth.make_motion(nf, 56), vw,
                                   0.015).cpu().numpy()
        tgt += rng.normal(scale=0.005, size=tgt.shape).astype(f32)
        if outputs:
            status, out = ts.step(opt, lin.cu(theta), lin.cu(beta), lin.cu(vw), lin.cu(tgt), outputs=True)
            return status.cpu().numpy(), {k: v.cpu().numpy() for k, v in out.items()}
        return lin._raw_step(ts, opt, lin.cu(theta), lin.cu(beta), lin.cu(vw), lin.cu(tgt))[0]

    lo, hi = 41, 82
    while attempt(hi) == 0:
        lo, hi = hi, 2 * hi
        assert hi < 4096
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if attempt(mid) == 0:
            lo = mid
        else:
            hi = mid
    assert attempt(hi) == -1  # SMPLPP_ERR_INVALID
    msg = capi.lib().smplpp_last_error().decode()
    assert msg in ("IkTask Error: task set too large for one CTA per frame",
                   "IkTask Error: IK problem too large for one CTA per frame"), msg
    status, out = attempt(lo, outputs=True)
    assert (status == 0).all()
    dim = out["A"].shape[1]
    lb, ub = q.ik_bounds(opts, lo, dim, 75)
    worst, active = 0.0, []
    for f in range(nf):
        A, b, d = out["A"][f], out["b"][f], out["delta"][f]
        ok, rep = q.kkt_certificate(A, b, d, lb, ub, q.ik_blocks(75, lo, dim))
        assert ok, (f, rep)
        worst, active = max(worst, rep["worst_ratio"]), active + [rep["n_upper"] + rep["n_lower"]]
        x_ref = q.reference_box_qp(A, b, lb, ub)
        assert q.objective(A, b, d) - q.objective(A, b, x_ref) <= q.objective_gap_tol(A, b, d)
    TABLE.append(("largest_n%d" % lo, "default", "%d/%d/%d" % (min(active), np.median(active), max(active)), worst, 0.0))
    print("largest bounded task set: n = %d (D = %d); n = %d: %s" % (lo, dim, hi, msg))
    assert (attempt(41) == 0)


# ----------------------------------------------------------------------------------------------------------------
# shared-beta stage
# ----------------------------------------------------------------------------------------------------------------
SB_FRAMES = 300
SB_SKIPPED = (0, 31, 32, 127, 128, 200, 299)  # fewer than n/2 valid markers: status 1
# the two Schur implementations on the same J (tcgen05 pose-blend columns for both), and the fused kernel
SB_PATHS = {"tc_schur": (401, 410, 420), "scalar": (401, 411, 420), "fused": (402, 410, 420)}
# |dbeta| of the unbounded reduced QP is a few 1e-3 here (the summed ||e||^2 damps it), so 1e-4 binds all ten
SB_CASES = [(m, lim) for m in ("direct", "vposer") for lim in (0.5, 0.01, 1e-4, 0.0)]


def _sb_inputs(handles, vposer_mode):
    from smplpp_b200 import synth
    params, smpl, vposer = handles
    rng = np.random.default_rng(900 + vposer_mode)
    faces = rng.choice(params.face_indices.shape[0], size=41, replace=False).astype(np.int64)
    ts = lin._task_set(smpl, faces, vposer if vposer_mode else None)
    n, F = ts.n, SB_FRAMES
    gt = synth.make_motion(F, 60 + vposer_mode).astype(f32)
    theta75 = gt.reshape(F, 75).copy()
    theta75[:, 3:] += rng.normal(scale=0.05, size=(F, 72)).astype(f32)
    theta = theta75
    if vposer_mode:
        theta = np.concatenate([theta75[:, :6], rng.normal(scale=0.7, size=(F, 32)), theta75[:, 69:75]], 1).astype(f32)
    beta_true = (rng.normal(size=10) * 2.0).astype(f32)
    vw = rng.dirichlet(np.ones(3), size=(F, n)).astype(f32)
    tgt = ts.forward_positions(beta_true, gt, vw, 0.015).cpu().numpy() + rng.normal(scale=0.005, size=(F, n, 3)).astype(f32)
    pw = np.ones((F, n), f32)
    for f in SB_SKIPPED:
        pw[f, rng.choice(n, size=n - n // 2 + 1, replace=False)] = 0.0
    return ts, theta, vw, tgt.astype(f32), pw


def _sb_run(ts, opts, theta, vw, tgt, pw, variants):
    """The shared-beta step and, on the same inputs, the per-frame step with the beta columns (update_state = 0)."""
    from smplpp_b200 import api
    F = theta.shape[0]
    lin.set_variant(variants)
    try:
        th, sb = lin.cu(theta), torch.zeros(10, dtype=torch.float32, device="cuda:0")
        status, red = ts.shared_beta_step(api.ik_options(**opts), th, sb, lin.cu(vw), lin.cu(tgt),
                                          pos_task_weight=lin.cu(pw), return_reduced=True)
        pf = api.ik_options(**dict(opts, optimize_beta=1, update_state=0))
        pstatus, out = ts.step(pf, lin.cu(theta), torch.zeros((F, 10), dtype=torch.float32, device="cuda:0"), lin.cu(vw),
                               lin.cu(tgt), pos_task_weight=lin.cu(pw), outputs=True)
    finally:
        lin.set_variant(lin.DEFAULT_VARIANT)
    return dict(status=status.cpu().numpy(), reduced=red.cpu().numpy(), theta=th.cpu().numpy(), beta=sb.cpu().numpy(),
                pstatus=pstatus.cpu().numpy(), A=out["A"].cpu().numpy(), b=out["b"].cpu().numpy(),
                e=out["e"].cpu().numpy())


@pytest.mark.parametrize("mode,limit", SB_CASES, ids=["%s-limit%g" % c for c in SB_CASES])
def test_shared_beta_stage_block_arrow(handles, mode, limit):
    """The shared-beta stage on 300 frames, 7 of them skipped, against the block-arrow system built from the per-frame
    blocks (DESIGN.md; tests/golden/make_ref_golden_ik_configs.py) in float64:
      reduced == [sum S_f | sum r_f | sum ||e_f||^2] over the status-0 frames, S_f = A_bb - A_bt A_tt^-1 A_tb (the beta
          block without its damping, which the QP adds once), r_f = b_b - A_bt A_tt^-1 b_t;
      the 10-unknown QP's dbeta (returned as float32 in the shared beta, beta_0 = 0) is optimal: its active set is the
          GPU's, its free entries are the float64 solution on that active set to float32 rounding, and that point passes
          the certificate and matches bvls' objective;
      theta_f of every status-0 frame moved by -A_tt^-1 (b_t + A_tb dbeta) to float32 rounding; status-1 frames unchanged;
      the three paths reach the same active set, and the two Schur paths the same dbeta within 1e-7 of the limit."""
    ts, theta, vw, tgt, pw = _sb_inputs(handles, mode == "vposer")
    opts = dict(MOTION, enable_vposer=int(mode == "vposer"), delta_beta_limit=limit, skip_if_too_few=1)
    td = theta_dim(opts)
    n = ts.n
    reg_b = float(f32(1e-3))
    lim = float(f32(limit))
    dbetas = {}
    for path, variants in SB_PATHS.items():
        r = _sb_run(ts, opts, theta, vw, tgt, pw, variants)
        skipped = np.zeros(SB_FRAMES, bool)
        skipped[list(SB_SKIPPED)] = True
        assert np.array_equal(r["status"], np.where(skipped, 1, 0)), (path, np.nonzero(r["status"])[0])
        assert np.array_equal(r["pstatus"], r["status"])
        bs = slice(td + 2 * n, td + 2 * n + 10)
        th = slice(0, td)
        S, rr, e2 = np.zeros((10, 10)), np.zeros(10), 0.0
        S_scale = r_scale = 0.0
        solves = {}
        for f in np.nonzero(~skipped)[0]:
            A, b = r["A"][f], r["b"][f]
            esq = float(r["e"][f].astype(np.float64) @ r["e"][f].astype(np.float64))
            Att, Atb = A[th, th], A[th, bs]
            Y = np.linalg.solve(Att, np.concatenate([Atb, b[th, None]], 1))
            solves[f] = Y
            Abb = A[bs, bs] - (reg_b + esq) * np.eye(10)
            S += Abb - Atb.T @ Y[:, :10]
            rr += b[bs] - Atb.T @ Y[:, 10]
            e2 += esq
            S_scale += np.abs(Abb).max()
            r_scale += np.abs(b[bs]).max() + np.abs(Atb.T @ Y[:, 10]).max()
        red = r["reduced"]
        assert np.abs(red[:100].reshape(10, 10) - S).max() <= 1e-9 * S_scale, path
        assert np.abs(red[100:110] - rr).max() <= 1e-9 * r_scale, path
        assert abs(red[110] - e2) <= 1e-9 * e2, path
        # the reduced QP and the GPU's dbeta
        H = red[:100].reshape(10, 10) + (reg_b + red[110]) * np.eye(10)
        g0 = red[100:110]
        lo, hi = np.full(10, -lim), np.full(10, lim)
        db32 = r["beta"]
        if lim == 0.0:
            assert (db32 == 0.0).all()
            x = np.zeros(10)
        else:
            side = np.where(db32 == f32(lim), 1, np.where(db32 == -f32(lim), -1, 0))
            x = side * lim
            fr = side == 0
            if fr.any():
                x[fr] = -np.linalg.solve(H[np.ix_(fr, fr)], g0[fr] + H[np.ix_(fr, ~fr)] @ x[~fr])
                assert (np.abs(db32[fr] - x[fr]) <= 2.0 ** -23 * np.abs(x[fr])).all(), (path, db32, x)
        ok, rep = q.kkt_certificate(H, g0, x, lo, hi)
        assert ok, (path, rep)
        x_ref = q.reference_box_qp(H, g0, lo, hi)
        assert q.objective(H, g0, x) - q.objective(H, g0, x_ref) <= q.objective_gap_tol(H, g0, x), path
        # back-substitution of every status-0 frame with that dbeta
        worst = 0.0
        for f, Y in solves.items():
            dth = -(Y[:, 10] + Y[:, :10] @ x)
            err = np.abs(r["theta"][f].astype(np.float64) - (theta[f].astype(np.float64) + dth))
            tol = 2.0 ** -23 * (np.abs(dth) + np.abs(r["theta"][f])) + 1e-9 * np.abs(dth).max()
            worst = max(worst, float((err / tol).max()))
            assert (err <= tol).all(), (path, f, int(np.argmax(err - tol)))
        assert np.array_equal(r["theta"][skipped], theta[skipped])
        dbetas[path] = db32
        TABLE.append(("sb_%s_%g" % (mode, limit), path, "%d/10" % int((np.abs(db32) == f32(lim)).sum()) if lim else "pinned",
                      rep["worst_ratio"], worst))
    # tc_schur and scalar reduce the same J: dbeta within 1e-7 of the limit (plus the float32 rounding of the output).
    # The fused kernel linearises with its own arithmetic (J differs from the two-kernel one in the last bits,
    # tests/test_ik_linearisation_gpu.py), which perturbs the reduced system as a whole: it must reach the same active
    # set (its dbeta is the exact solution of its own reduced QP, checked above), and its free entries may differ by
    # 1e-4 of the largest |dbeta| (measured on a B200: up to 4e-5, on a free entry 30 times smaller than the others)
    ref = dbetas["tc_schur"]
    side = lambda d: np.where(d == f32(lim), 1, np.where(d == -f32(lim), -1, 0)) if lim else np.zeros(10)  # noqa: E731
    for p, d in dbetas.items():
        assert np.array_equal(side(d), side(ref)), (p, d, ref)
        tol = 2.0 ** -23 * np.abs(ref) if p != "fused" else 1e-4 * np.abs(ref).max()
        assert (np.abs(d - ref) <= 1e-7 * lim + tol).all(), (p, d, ref)
