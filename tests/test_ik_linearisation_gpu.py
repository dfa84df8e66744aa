"""The linearisation of the IK step (e, J, re-weighted attachments) and what follows directly from it (A, b, delta) against
a float64 run of the oracle, on task sets, models and kernel paths beyond the 41 golden markers.

The float32 oracle is the reference's own arithmetic, and that is ill-conditioned on a few rows (up to 6e-4 of max |J|
where face normals nearly cancel, against a median row of 1e-8).  So the GPU is measured against the float64 oracle, and
each row may miss it by at most ten times what the float32 reference misses it by on the same row (floor 1e-4 of the
frame's max |J|); every column block (theta, phi, beta) is checked the same way with its own scale.  The comparator is
shown to catch a 1e-3 relative change of a single Jacobian column.

Every configuration runs 130 frames (per-frame poses, beta, targets and Dirichlet vertex weights) through each kernel path
that can take it, and compares frames 0, 31, 32, 127, 128 and 129 (the edges of the 32-frame CTAs of the pose-blend kernel
and of the 128-frame tiles of the rest-shape kernel) with the oracle, or three of them where the oracle is slow.

Kernel paths (smplpp_set_forward_variant):
  default   400 410 420  two kernels; tcgen05 rest shape and pose-blend columns; fp64 tensor-core solve where it fits
  ffma      401 411 421  two kernels; FFMA rest shape and pose-blend columns; scalar solve
  tc_pb     401 410 422  two kernels; FFMA rest shape, tcgen05 pose-blend columns
  fused     402 410 420  one fused kernel on the task set's shared attachment records
  faces     smplpp_ik_step_faces with every frame's faces given (the fused kernel on per-frame records)

The tcgen05 pose-blend columns are dropped for a task set in which a task has more than 21 vertex pairs (corners plus
1-ring vertices, ik.cu where pair_off is built).  The synthetic mesh has no such face: its largest pair count is exactly 21
(three faces), so that fallback cannot be reached here; `ring21` puts those three faces, the last ones the tcgen05 path
takes, into a task set instead.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
f32 = np.float32
F64 = torch.float64
B = 130
FRAMES6 = (0, 31, 32, 127, 128, 129)
FRAMES3 = (0, 32, 129)
REST_TC_MAX_VERTICES = 597  # 8 tiles of 224 coordinates (ik_poseblend_tc.cu, rstc::MAX_TILES)

VARIANTS = {"default": (400, 410, 420), "ffma": (401, 411, 421), "tc_pb": (401, 410, 422), "fused": (402, 410, 420),
            "faces": (400, 410, 420)}
DEFAULT_VARIANT = (400, 410, 420)


def cu(a, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device="cuda:0").contiguous()


def set_variant(vs):
    from smplpp_b200 import capi
    for v in vs:
        capi.check(capi.lib().smplpp_set_forward_variant(v))


# ----------------------------------------------------------------------------------------------------------------
# task sets and configurations
# ----------------------------------------------------------------------------------------------------------------
def _adjacency(params):
    faces0 = np.asarray(params.face_indices, np.int64) - 1
    adj = [[] for _ in range(params.vertices_template.shape[0])]
    for f, tri in enumerate(faces0.tolist()):
        for v in tri:
            adj[v].append(f)
    return faces0, adj


def ring_vertices(faces0, adj, f):
    """Corners and 1-ring vertices of face f: the vertex pairs of its task (ik.cu, pair_off)."""
    return set(int(v) for c in faces0[f] for g in adj[c] for v in faces0[g])


def rest_limit_faces(params, seed):
    """The longest prefix of a random face order whose task vertices (corners + rings) number <= 597, and the prefix one
    face longer (> 597)."""
    faces0, adj = _adjacency(params)
    order = np.random.default_rng(seed).permutation(len(faces0))
    used = set()
    for k, f in enumerate(order):
        grown = used | ring_vertices(faces0, adj, f)
        if len(grown) > REST_TC_MAX_VERTICES:
            return order[:k].astype(np.int64), order[:k + 1].astype(np.int64), len(used), len(grown)
        used = grown
    raise AssertionError("the mesh has fewer than 598 vertices")


def grid_params(seed=11, side=9):
    """Small height-field mesh with DENSE skinning rows (24 non-zeros per vertex, sums != 1); the helper of
    tests/test_task_forward_gpu.py."""
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
    return synth.SmplParams(
        face_indices=np.asarray(faces, np.int32) + 1, shape_blend_shapes=rng.normal(size=(V, 3, 10)).astype(f32) * 0.005,
        pose_blend_shapes=rng.normal(size=(V, 3, 207)).astype(f32) * 0.001, vertices_template=templ,
        joint_regressor=rng.dirichlet(np.ones(V), size=24).astype(f32), kinematic_tree=tree,
        weights=rng.uniform(0.1, 1.0, size=(V, 24)).astype(f32))


MOTION = dict(normal_task_weight=0.0, phi_limit=0.0, normal_offset=0.015, optimize_beta=0, enable_qp=1, enable_phi=0)
PHI = dict(phi_limit=0.04, enable_phi=1)


@dataclass
class Cfg:
    faces: str                      # how the task faces are chosen (see task_faces)
    opts: dict
    n: int = 41
    seed: int = 1
    noise: float = 0.05             # rad of pose noise on top of synth.make_motion
    frames: tuple = FRAMES3
    model: str = "smpl"             # "smpl" (synthetic SMPL) or "grid" (dense skinning rows)
    pos_weights: bool = False       # per-frame pos_task_weight with zeros and fractions
    per_frame_faces: bool = False   # every frame carries its own random faces (smplpp_ik_step_faces only)
    variants: tuple = tuple(VARIANTS)

    @property
    def vposer(self):
        return bool(self.opts.get("enable_vposer"))


CONFIGS = {
    # D = 75: tcgen05 rest shape and pose-blend columns, NB = 10 tensor-core solve
    "motion": Cfg("random", dict(MOTION), frames=FRAMES6),
    "llt": Cfg("random", dict(MOTION, normal_offset=0.0, enable_qp=0), seed=2),
    # rows_per_task = 4, at the 0.2 rad pose noise where the float32 reference is worst conditioned
    "normal_rows": Cfg("random", dict(MOTION, normal_task_weight=1.0, normal_offset=0.0), seed=3, noise=0.2),
    # phi columns: FFMA pose-blend phase and the scalar box-QP kernel
    "body": Cfg("random", dict(MOTION, optimize_beta=1, **PHI), seed=4, frames=FRAMES6),
    "beta_llt": Cfg("random", dict(MOTION, optimize_beta=1, enable_qp=0), seed=5),           # D = 85, NB = 11
    "beta_qp": Cfg("random", dict(MOTION, optimize_beta=1), seed=6),                         # beta bounds: scalar QP
    "vposer": Cfg("random", dict(MOTION, enable_vposer=1), seed=7, frames=FRAMES6),          # D = 44, NB = 6
    "vposer_beta_llt": Cfg("random", dict(MOTION, enable_vposer=1, optimize_beta=1, enable_qp=0), seed=8),  # D = 54, NB = 7
    "rest_le597": Cfg("rest_le", dict(MOTION), seed=9),
    "rest_gt597": Cfg("rest_gt", dict(MOTION), seed=9),
    "ring21": Cfg("ring21", dict(MOTION), n=20, seed=10),
    "n1": Cfg("random", dict(MOTION), n=1, seed=11),
    "face_twice": Cfg("twice", dict(MOTION), n=10, seed=12),
    "adjacent": Cfg("adjacent", dict(MOTION, normal_task_weight=1.0), seed=13),
    "pos_weights": Cfg("random", dict(MOTION), seed=14, pos_weights=True),
    "dense_skinning": Cfg("grid", dict(MOTION), n=9, seed=15, model="grid"),
    "per_frame_motion": Cfg("random", dict(MOTION), n=30, seed=16, per_frame_faces=True, variants=("faces",)),
    "per_frame_body": Cfg("random", dict(MOTION, enable_vposer=1, optimize_beta=1, **PHI), n=30, seed=17,
                          per_frame_faces=True, variants=("faces",)),
}


def task_faces(cfg: Cfg, params, rng):
    faces0, adj = _adjacency(params)
    nf = len(faces0)
    if cfg.faces == "random":
        return rng.choice(nf, size=cfg.n, replace=False).astype(np.int64)
    if cfg.faces in ("rest_le", "rest_gt"):
        le, gt, _, _ = rest_limit_faces(params, cfg.seed)
        return le if cfg.faces == "rest_le" else gt
    if cfg.faces == "ring21":
        pairs = np.array([len(ring_vertices(faces0, adj, f)) for f in range(nf)])
        assert pairs.max() == 21
        top = np.nonzero(pairs == 21)[0]
        rest = rng.choice(np.setdiff1d(np.arange(nf), top), size=cfg.n - len(top), replace=False)
        return rng.permutation(np.concatenate([top, rest])).astype(np.int64)
    if cfg.faces == "twice":
        f = rng.choice(nf, size=cfg.n - 1, replace=False)
        return np.concatenate([f[:4], f[2:3], f[4:]]).astype(np.int64)
    if cfg.faces == "adjacent":
        # one face and every face that shares a vertex with it (14 on this mesh, capped at 41)
        f0 = int(rng.integers(nf))
        near = sorted({g for c in faces0[f0] for g in adj[c]} - {f0})
        return np.asarray([f0] + near[:40], np.int64)
    if cfg.faces == "grid":
        return np.array([9, 20, 33, 47, 58, 64, 71, 90, 101], np.int64)
    raise ValueError(cfg.faces)


@dataclass
class Inputs:
    faces: np.ndarray               # (n,) shared, or (B, n) per frame
    theta: np.ndarray               # (B, theta_dim) state
    beta: np.ndarray                # (B, 10)
    vw: np.ndarray                  # (B, n, 3)
    tgt: np.ndarray                 # (B, n, 3)
    tn: Optional[np.ndarray]        # (B, n, 3) unit target normals, normal rows only
    pw: Optional[np.ndarray]        # (B, n)


def make_inputs(cfg: Cfg, params, smpl, ts):
    from smplpp_b200 import synth
    rng = np.random.default_rng(100 + cfg.seed)
    n = ts.n
    if cfg.model == "grid":
        beta, th = synth.make_forward_inputs(B, cfg.seed)
        th[:, 1:] *= 0.3
        theta75 = th.reshape(B, 75)
        tgt_theta = th.copy()
        tgt_theta[:, 1:] += rng.normal(scale=0.05, size=(B, 24, 3)).astype(f32)
    else:
        gt = synth.make_motion(B, 20 + cfg.seed)
        theta75 = gt.reshape(B, 75).astype(f32).copy()
        theta75[:, 3:] += rng.normal(scale=cfg.noise, size=(B, 72)).astype(f32)
        tgt_theta = gt.astype(f32)
        beta = (rng.normal(size=(B, 10)) * 0.5).astype(f32)
    vw = rng.dirichlet(np.ones(3), size=(B, n)).astype(f32)
    faces = ts.face_idx
    if cfg.per_frame_faces:
        nf = params.face_indices.shape[0]
        faces = np.stack([rng.choice(nf, size=n, replace=False) for _ in range(B)]).astype(np.int64)
        tgt = np.empty((B, n, 3), f32)
        for b in range(B):  # markers of the target pose on this frame's own faces
            tsb = _task_set(smpl, faces[b])
            tgt[b] = tsb.forward_positions(beta[b:b + 1], tgt_theta[b:b + 1], vw[b:b + 1], 0.015)[0].cpu().numpy()
    else:
        tgt = ts.forward_positions(beta, tgt_theta, vw, 0.015).cpu().numpy()
    tgt += rng.normal(scale=0.005, size=tgt.shape).astype(f32)
    tn = None
    if cfg.opts.get("normal_task_weight", 0.0) > 0:
        tn = rng.normal(size=(B, n, 3)).astype(f32)
        tn /= np.linalg.norm(tn, axis=2, keepdims=True)
    pw = None
    if cfg.pos_weights:
        pw = rng.choice(np.array([0.0, 0.25, 0.5, 1.0], f32), size=(B, n), p=[0.2, 0.2, 0.2, 0.4]).astype(f32)
    theta = theta75
    if cfg.vposer:
        theta = np.concatenate([theta75[:, :6], rng.normal(scale=0.7, size=(B, 32)), theta75[:, 69:75]], 1).astype(f32)
    return Inputs(faces, theta, beta, vw, tgt, tn, pw)


def _task_set(smpl, faces, vposer=None):
    from smplpp_b200 import api
    return api.IkTaskSet(smpl, np.asarray(faces, np.int64), vposer=vposer)


# ----------------------------------------------------------------------------------------------------------------
# oracle
# ----------------------------------------------------------------------------------------------------------------
def oracle_frame(models, cfg: Cfg, inp: Inputs, b: int, dtype, opts=None):
    from oracle import smpl_oracle as so
    o = cfg.opts if opts is None else opts
    model, vposer = models[dtype]
    faces = inp.faces[b] if inp.faces.ndim == 2 else inp.faces
    phi_limit = o.get("phi_limit", 0.0) if o.get("enable_phi") else 0.0
    tasks = []
    for i in range(len(faces)):
        kw = dict(target_normal=torch.as_tensor(inp.tn[b, i])) if inp.tn is not None else {}
        tasks.append(so.IkTask(int(faces[i]), target_pos=torch.as_tensor(inp.tgt[b, i]),
                               pos_task_weight=float(inp.pw[b, i]) if inp.pw is not None else 1.0,
                               normal_task_weight=o.get("normal_task_weight", 0.0), phi_limit=phi_limit,
                               normal_offset=o.get("normal_offset", 0.0), vertex_weights=torch.as_tensor(inp.vw[b, i]), **kw))
    return so.ik_iteration(model, tasks, inp.theta[b], inp.beta[b], vposer=vposer if o.get("enable_vposer") else None,
                           optimize_beta=bool(o.get("optimize_beta")), enable_qp=bool(o.get("enable_qp", 1)),
                           skip_if_too_few=False, dtype=dtype)


# ----------------------------------------------------------------------------------------------------------------
# the acceptance rule
# ----------------------------------------------------------------------------------------------------------------
def column_blocks(theta_dim, n, dim):
    return {"theta": (0, theta_dim), "phi": (theta_dim, theta_dim + 2 * n), "beta": (theta_dim + 2 * n, dim)}


def compare_linearisation(Jg, eg, J32, e32, J64, e64, blocks):
    """The rule for one frame.  Returns (failures, gpu error, float32 reference error), errors as max over rows of
    max_c |dJ| / max |J64| of the whole frame."""
    fails = []
    s = np.abs(J64).max()
    gpu_err = np.abs(Jg - J64).max(1) / s
    ref_err = np.abs(J32 - J64).max(1) / s
    for name, (lo, hi) in [("all", (0, J64.shape[1]))] + list(blocks.items()):
        if hi <= lo:
            continue
        sb = np.abs(J64[:, lo:hi]).max()
        if sb == 0.0:  # a block the configuration does not use is zero (phi columns without phi)
            if np.abs(Jg[:, lo:hi]).max() != 0.0:
                fails.append("J block %s should be zero" % name)
            continue
        g = np.abs(Jg[:, lo:hi] - J64[:, lo:hi]).max(1) / sb
        r = np.abs(J32[:, lo:hi] - J64[:, lo:hi]).max(1) / sb
        bad = np.nonzero(g > np.maximum(1e-4, 10.0 * r))[0]
        if bad.size:
            k = bad[np.argmax(g[bad])]
            fails.append("J block %s: %d rows fail, worst row %d: gpu %.3g, fp32 reference %.3g" % (name, bad.size, k, g[k], r[k]))
    de = np.abs(eg - e64)
    bad = np.nonzero(de > np.maximum(1e-5, 10.0 * np.abs(e32 - e64)))[0]
    if bad.size:
        fails.append("e: %d entries fail, worst %.3g m" % (bad.size, de[bad].max()))
    return fails, float(gpu_err.max()), float(ref_err.max())


def check_normal_equations(cfg: Cfg, n, J, e, A, b, delta, theta_state):
    """A and b from the GPU's own J and e in float64 (node.cpp:884-904), and delta as the fp64 solve of the GPU's own
    (A, b) where nothing is bounded, or within its bounds."""
    o = cfg.opts
    theta_dim = 44 if cfg.vposer else 75
    dim = J.shape[1]
    J64, e64 = J.astype(np.float64), e.astype(np.float64)
    reg = np.concatenate([np.full(theta_dim, 1e-3), np.full(2 * n, 1e-1), np.full(dim - theta_dim - 2 * n, 1e-3)])
    A_chk = J64.T @ J64
    b_chk = J64.T @ e64
    A_chk[np.diag_indices(dim)] += reg.astype(f32).astype(np.float64) + float(e64 @ e64)
    if cfg.vposer:  # latent and hand prior (node.cpp:895-904)
        wv = np.concatenate([np.zeros(6), np.full(32, 1e-5), np.full(6, 1e3)]).astype(f32).astype(np.float64)
        A_chk[np.arange(theta_dim), np.arange(theta_dim)] += wv
        b_chk[:theta_dim] += wv * theta_state.astype(np.float64)
    assert np.abs(A - A_chk).max() <= 1e-9 * max(1.0, np.abs(A_chk).max())
    assert np.abs(b - b_chk).max() <= 1e-9 * max(1.0, np.abs(b_chk).max())
    bounded = o.get("enable_qp", 1) and ((o.get("enable_phi") and o.get("phi_limit", 0) > 0) or o.get("optimize_beta"))
    if not bounded:
        d_chk = -np.linalg.solve(A, b)
        assert np.abs(delta - d_chk).max() <= 1e-6 * np.abs(d_chk).max()
    else:
        phi = delta[theta_dim:theta_dim + 2 * n]
        assert np.abs(phi).max(initial=0.0) <= o.get("phi_limit", 0.0) * (1 + 1e-6) + 1e-12
        if o.get("optimize_beta"):
            assert np.abs(delta[theta_dim + 2 * n:]).max() <= 0.5 * (1 + 1e-6)


# ----------------------------------------------------------------------------------------------------------------
# fixtures
# ----------------------------------------------------------------------------------------------------------------
TABLE = []


@pytest.fixture(scope="module")
def models(params, vposer_params, smpl_gpu):
    """GPU handles and float32 / float64 oracle models per model kind."""
    from oracle import smpl_oracle as so
    from smplpp_b200 import api
    out = {}
    vp32 = so.VPoserDecoder.from_params(vposer_params)
    m32 = so.SmplModel.from_params(params)
    out["smpl"] = (params, smpl_gpu, api.VPoserDecoder(vposer_params),
                   {torch.float32: (m32, vp32), F64: (m32.to(F64), vp32.to(F64))})
    gp = grid_params()
    g32 = so.SmplModel.from_params(gp)
    out["grid"] = (gp, api.SMPL(gp), None, {torch.float32: (g32, None), F64: (g32.to(F64), None)})
    yield out
    print("\n%-18s %-8s %12s %12s %10s" % ("configuration", "variant", "max GPU err", "max fp32 err", "max |de| m"))
    for row in TABLE:
        print("%-18s %-8s %12.3g %12.3g %10.3g" % row)


@pytest.fixture(scope="module")
def oracle_cache():
    return {}


def prepared(name, models, oracle_cache):
    """Task set, inputs and the float32 / float64 oracle results of the compared frames of one configuration, computed
    once for all kernel paths."""
    if name not in oracle_cache:
        cfg = CONFIGS[name]
        params, smpl, vposer, om = models[cfg.model]
        rng = np.random.default_rng(cfg.seed)
        ts = _task_set(smpl, task_faces(cfg, params, rng), vposer if cfg.vposer else None)
        inp = make_inputs(cfg, params, smpl, ts)
        ref = {b: (oracle_frame(om, cfg, inp, b, torch.float32), oracle_frame(om, cfg, inp, b, F64)) for b in cfg.frames}
        oracle_cache[name] = (cfg, ts, inp, ref)
    return oracle_cache[name]


def run_step(cfg: Cfg, ts, inp: Inputs, variant: str, frames=None):
    """One step on the GPU; frames=None: the whole batch, else the listed frames only.  Returns status and host copies of
    the outputs and the updated state."""
    from smplpp_b200 import api
    sel = slice(None) if frames is None else list(frames)
    opt = api.ik_options(skip_if_too_few=0, **cfg.opts)
    theta, beta, vw = cu(inp.theta[sel]), cu(inp.beta[sel]), cu(inp.vw[sel])
    face = None
    if variant == "faces":
        fa = inp.faces if inp.faces.ndim == 2 else np.broadcast_to(inp.faces, (B, ts.n))
        face = cu(fa[sel], torch.int32)
    set_variant(VARIANTS[variant])
    try:
        status, out = ts.step(opt, theta, beta, vw, cu(inp.tgt[sel]),
                              pos_task_weight=cu(inp.pw[sel]) if inp.pw is not None else None,
                              target_normal=cu(inp.tn[sel]) if inp.tn is not None else None, outputs=True, face_idx=face)
    finally:
        set_variant(DEFAULT_VARIANT)
    res = {k: v.cpu().numpy() for k, v in out.items()}
    res.update(status=status.cpu().numpy(), theta=theta.cpu().numpy(), beta=beta.cpu().numpy(), vw=vw.cpu().numpy())
    return res


CASES = [(c, v) for c, cfg in CONFIGS.items() for v in cfg.variants]


# ----------------------------------------------------------------------------------------------------------------
# tests
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("config,variant", CASES, ids=["%s-%s" % cv for cv in CASES])
def test_linearisation_vs_f64_oracle(models, oracle_cache, config, variant):
    cfg, ts, inp, ref = prepared(config, models, oracle_cache)
    n = ts.n
    if config == "dense_skinning":
        from smplpp_b200 import capi
        assert capi.lib().smplpp_model_max_influences(models["grid"][1].handle) == 24
    out = run_step(cfg, ts, inp, variant)
    assert (out["status"] == 0).all()
    theta_dim = 44 if cfg.vposer else 75
    worst = [0.0, 0.0, 0.0]
    failures = []
    for b in cfg.frames:
        r32, r64 = ref[b]
        J = out["J"][b]
        blocks = column_blocks(theta_dim, n, J.shape[1])
        fails, g, r = compare_linearisation(J, out["e"][b], r32.J, r32.e, r64.J, r64.e, blocks)
        failures += ["frame %d: %s" % (b, f) for f in fails]
        worst = [max(worst[0], g), max(worst[1], r), max(worst[2], float(np.abs(out["e"][b] - r64.e).max()))]
        assert np.abs(out["vw"][b] - r64.vertex_weights).max() < 1e-4
        check_normal_equations(cfg, n, J, out["e"][b], out["A"][b], out["b"][b], out["delta"][b], inp.theta[b])
    TABLE.append((config, variant, worst[0], worst[1], worst[2]))
    print("%s %s: max GPU error %.3g, max fp32 reference error %.3g (of max |J|), max |de| %.3g m"
          % (config, variant, worst[0], worst[1], worst[2]))
    assert not failures, failures
    # batch invariance: the compared frames run alone return the bytes they get inside the 130-frame batch
    alone = run_step(cfg, ts, inp, variant, frames=cfg.frames)
    for i, b in enumerate(cfg.frames):
        for k in ("e", "J", "A", "b", "delta", "theta", "beta", "vw", "status"):
            assert np.array_equal(alone[k][i], out[k][b]), (b, k)


def test_comparator_detects_one_column_off_by_1e3(models, oracle_cache):
    """The rule catches a subtle kernel bug: the GPU's own J with one joint-rotation column (one of those the pose-blend
    stage writes) scaled by 1 + 1e-3 fails it, while the unmodified J passes."""
    cfg, ts, inp, ref = prepared("motion", models, oracle_cache)
    out = run_step(cfg, ts, inp, "default", frames=(0,))
    r32, r64 = ref[0]
    J = out["J"][0]
    blocks = column_blocks(75, ts.n, J.shape[1])
    assert not compare_linearisation(J, out["e"][0], r32.J, r32.e, r64.J, r64.e, blocks)[0]
    c = 3 + int(np.argmax(np.abs(J[:, 3:75]).max(0)))
    bad = J.copy()
    bad[:, c] *= f32(1 + 1e-3)
    fails = compare_linearisation(bad, out["e"][0], r32.J, r32.e, r64.J, r64.e, blocks)[0]
    assert fails, "a 1e-3 change of column %d went unnoticed" % c
    # also a column that is not the largest one: the block-wise and row-wise scales still see it
    c2 = 3 + int(np.argsort(np.abs(J[:, 3:75]).max(0))[-10])
    bad = J.copy()
    bad[:, c2] *= f32(1 + 1e-3)
    assert compare_linearisation(bad, out["e"][0], r32.J, r32.e, r64.J, r64.e, blocks)[0]


def test_rest_shape_limit_sides(models):
    """The two task sets of rest_le597 / rest_gt597 lie on the two sides of the tcgen05 rest-shape limit: the tcgen05
    rest shape (variant 0) differs from the FFMA one in the last bits below it and is the FFMA one above it."""
    from smplpp_b200 import synth
    params, smpl, _, _ = models["smpl"]
    le, gt, n_le, n_gt = rest_limit_faces(params, CONFIGS["rest_le597"].seed)
    beta, theta = synth.make_forward_inputs(130, 3)
    for faces, nv, tc in ((le, n_le, True), (gt, n_gt, False)):
        ts = _task_set(smpl, faces)
        assert ts.vertex_count == nv and (nv <= REST_TC_MAX_VERTICES) == tc
        r0, _ = ts.restShape(beta, theta, 0)
        r1, _ = ts.restShape(beta, theta, 1)
        assert torch.equal(r0, r1) != tc
        assert (r0 - r1).abs().max().item() < 1e-6  # rounding of rest positions of up to ~1 m


@pytest.mark.parametrize("config", ["motion", "body", "vposer", "dense_skinning"])
def test_step_faces_equals_shared_record_fused_step(models, oracle_cache, config):
    """smplpp_ik_step_faces with every frame carrying the task set's own faces builds per-frame records equal to the
    shared ones and runs the same fused kernel: bitwise the fused step (402)."""
    cfg, ts, inp, _ = prepared(config, models, oracle_cache)
    a = run_step(cfg, ts, inp, "fused")
    b = run_step(cfg, ts, inp, "faces")
    for k in ("status", "e", "J", "A", "b", "delta", "theta", "beta", "vw"):
        assert np.array_equal(a[k], b[k]), k


def _raw_step(ts, opt, theta, beta, vw, tgt):
    """smplpp_ik_step's return code (IkTaskSet.step raises instead)."""
    from smplpp_b200 import api, capi
    bsz = theta.shape[0]
    dim = int(capi.lib().smplpp_ik_dim(C.byref(opt), C.c_int32(ts.n)))
    status = torch.empty((bsz,), dtype=torch.int32, device="cuda:0")
    e = torch.empty((bsz, 4 * ts.n), dtype=torch.float32, device="cuda:0")
    J = torch.empty((bsz, 4 * ts.n, dim), dtype=torch.float32, device="cuda:0")
    ws = torch.empty(capi.lib().smplpp_ik_workspace_bytes(ts._h, C.byref(opt), C.c_int64(bsz)), dtype=torch.uint8,
                     device="cuda:0")
    rc = capi.lib().smplpp_ik_step(ts.smpl.handle, None, ts._h, C.byref(opt), api._stream(torch.device("cuda:0")),
                                   C.c_int64(bsz), api._ptr(theta), api._ptr(beta), C.c_int64(10), api._ptr(vw),
                                   api._ptr(tgt), None, None, api._ptr(status), api._ptr(e), api._ptr(J), None, None, None,
                                   api._ptr(ws), C.c_size_t(ws.numel()))
    torch.cuda.synchronize()
    return rc, status, e, J


def test_largest_task_set_and_clean_refusal(models, oracle_cache):
    """The largest random task set the two-kernel step accepts (bisection on its return code, motion options) against the
    oracle on one frame; one face more is refused with SMPLPP_ERR_INVALID and the documented text, and the same SMPL
    handle runs a normal step afterwards."""
    from smplpp_b200 import api, capi
    params, smpl, _, om = models["smpl"]
    cfg = Cfg("random", dict(MOTION), frames=(0,))
    opt = api.ik_options(skip_if_too_few=0, **cfg.opts)
    order = np.random.default_rng(77).permutation(params.face_indices.shape[0]).astype(np.int64)
    cfg_m, ts_m, inp_m, _ = prepared("motion", models, oracle_cache)
    before = run_step(cfg_m, ts_m, inp_m, "default", frames=(0,))

    def attempt(n):
        ts = _task_set(smpl, order[:n])
        rng = np.random.default_rng(n)
        theta = synth_theta()
        vw = rng.dirichlet(np.ones(3), size=(1, n)).astype(f32)
        tgt = ts.forward_positions(np.zeros((1, 10), f32), theta.reshape(1, 25, 3), vw, 0.015).cpu().numpy()
        tgt += rng.normal(scale=0.01, size=tgt.shape).astype(f32)
        beta = np.zeros((1, 10), f32)
        rc, status, e, J = _raw_step(ts, opt, cu(theta), cu(beta), cu(vw), cu(tgt))
        return rc, ts, Inputs(order[:n], theta, beta, vw, tgt, None, None), status, e, J

    lo, hi = 41, 82
    while attempt(hi)[0] == 0:
        lo, hi = hi, 2 * hi
        assert hi < 4096
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if attempt(mid)[0] == 0:
            lo = mid
        else:
            hi = mid
    rc, ts, inp, status, e, J = attempt(hi)
    assert rc == -1  # SMPLPP_ERR_INVALID
    msg = capi.lib().smplpp_last_error().decode()
    assert msg in ("IkTask Error: task set too large for one CTA per frame",
                   "IkTask Error: IK problem too large for one CTA per frame"), msg
    rc, ts, inp, status, e, J = attempt(lo)
    assert rc == 0 and int(status.cpu()[0]) == 0
    print("largest task set of the two-kernel step: n = %d faces (%d task vertices); n = %d: %s" % (lo, ts.vertex_count, hi, msg))
    r32, r64 = oracle_frame(om, cfg, inp, 0, torch.float32), oracle_frame(om, cfg, inp, 0, F64)
    Jg, eg = J[0].cpu().numpy(), e[0].cpu().numpy()
    fails, g, r = compare_linearisation(Jg, eg, r32.J, r32.e, r64.J, r64.e, column_blocks(75, lo, Jg.shape[1]))
    TABLE.append(("largest_n%d" % lo, "default", g, r, float(np.abs(eg - r64.e).max())))
    assert not fails, fails
    after = run_step(cfg_m, ts_m, inp_m, "default", frames=(0,))
    for k in ("status", "e", "J", "A", "b", "delta", "theta", "vw"):
        assert np.array_equal(before[k], after[k]), k


def synth_theta():
    from smplpp_b200 import synth
    return synth.make_motion(1, 55).reshape(1, 75).astype(f32)
