"""TEST INFRASTRUCTURE — CPU restatement (the "oracle") of the reference algorithm for the hot path.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this
module, and only as the CHECKER.  The product (smplpp_b200/) never imports it.

The reference computes everything with libtorch CPU float32 tensor ops and obtains Jacobians from autograd;
this restatement uses the same ATen ops through the Python front end (torch CPU, float32, autograd) in the
same order, so it reproduces the reference's arithmetic — including its quirks — rather than a textbook
SMPL.  Each function cites the reference lines it follows.  It is pinned (tests/test_oracle.py) against
  (1) the known-answer vectors of src/toolbox/Tester.cpp (tests/golden/tester_kat.json),
  (2) the reference's own property tests (tests/src/TestGeometryUtils.cpp, tests/src/TestVPoser.cpp),
  (3) outputs of the UNMODIFIED reference sources compiled here (oracle/_ref/libsmplpp_ref.so via
      oracle/ref_lib.py; committed as tests/golden/ref_*.npz by tests/golden/make_ref_golden.py).
The QP of node/node.cpp:907-930 is solved by a third-party library (QpSolverCollection -> eigen-qld, both
unpinned and not vendored): "parity unpinned" at that boundary — the strictly convex box-QP is solved here by
an fp64 primal active-set method and checked through its KKT conditions.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np
import torch

JOINT_NUM = 24
SHAPE_DIM = 10
POSE_DIM = 207
LATENT_DIM = 32
FLT_EPS = float(np.finfo(np.float32).eps)


def _t(a, dtype=torch.float32):
    return a if isinstance(a, torch.Tensor) else torch.as_tensor(np.asarray(a), dtype=dtype)


# ------------------------------------------------------------------------------------------------------------
# BlendShape (src/BlendShape.cpp)
# ------------------------------------------------------------------------------------------------------------

def rodrigues(theta: torch.Tensor) -> torch.Tensor:
    """src/BlendShape.cpp:803-844.  theta (N,24,3) -> (N,24,3,3).  Note `norm(theta + 1e-8)` (:813) and
    `axes = theta / angles` (:814): the epsilon enters the angle only."""
    n = theta.shape[0]
    angles = torch.norm(theta + 1e-8, 2, [2], True)  # (N,24,1)
    axes = theta / angles
    zeros = torch.zeros(n, theta.shape[1])
    skew = torch.stack(
        [zeros, -axes[:, :, 2], axes[:, :, 1], axes[:, :, 2], zeros, -axes[:, :, 0], -axes[:, :, 1], axes[:, :, 0],
         zeros], 2).reshape(n, theta.shape[1], 3, 3)
    eye = torch.eye(3).expand(n, theta.shape[1], 3, 3)
    sine = torch.sin(angles.unsqueeze(3).expand(n, theta.shape[1], 3, 3))
    cosine = torch.cos(angles.unsqueeze(3).expand(n, theta.shape[1], 3, 3))
    return eye + skew * sine + torch.matmul(skew, skew) * (1 - cosine)


def pose_blend_coeffs(pose_rot: torch.Tensor) -> torch.Tensor:
    """linRotMin + unroll, src/BlendShape.cpp:865-928 (rest pose = identity, :740-744). (N,24,3,3) -> (N,207)."""
    n = pose_rot.shape[0]
    un = pose_rot.reshape(n, JOINT_NUM * 9)[:, 9:]
    rest = torch.eye(3).expand(n, JOINT_NUM, 3, 3).reshape(n, JOINT_NUM * 9)[:, 9:]
    return un - rest


def pose_blend(coeffs: torch.Tensor, pose_basis: torch.Tensor) -> torch.Tensor:
    """src/BlendShape.cpp:764: tensordot over the 207 axis. -> (N,V,3)"""
    return torch.tensordot(coeffs, pose_basis, ([1], [2]))


def shape_blend(beta: torch.Tensor, shape_basis: torch.Tensor) -> torch.Tensor:
    """src/BlendShape.cpp:670-683. -> (N,V,3)"""
    return torch.tensordot(beta, shape_basis, ([1], [2]))


# ------------------------------------------------------------------------------------------------------------
# JointRegression (src/JointRegression.cpp)
# ------------------------------------------------------------------------------------------------------------

def linear_combine(templ, shape_bs, pose_bs):
    """src/JointRegression.cpp:551-565"""
    return templ + shape_bs + pose_bs


def joint_regress(templ, shape_bs, joint_regressor):
    """src/JointRegression.cpp:583-598 — pose blend is NOT included (:588)."""
    blend = templ + shape_bs
    return torch.transpose(torch.tensordot(blend, joint_regressor, ([1], [1])), 1, 2)


# ------------------------------------------------------------------------------------------------------------
# WorldTransformation (src/WorldTransformation.cpp)
# ------------------------------------------------------------------------------------------------------------

def world_transform(pose_rot, joints, parents: Sequence[int]):
    """transform(): localTransform :508-536, globalTransform :583-610, relativeTransform :657-677.
    pose_rot (N,24,3,3), joints (N,24,3) -> relative transforms (N,24,4,4)."""
    n = pose_rot.shape[0]
    rot_homo = torch.cat([pose_rot, torch.zeros(n, JOINT_NUM, 1, 3)], 2)  # (N,24,4,3)
    trans = [joints[:, 0, :]]
    for i in range(1, JOINT_NUM):
        trans.append(joints[:, i, :] - joints[:, int(parents[i]), :])
    local_t = torch.stack(trans, 1).unsqueeze(3)  # (N,24,3,1)
    local_t = torch.cat([local_t, torch.ones(n, JOINT_NUM, 1, 1)], 2)
    local = torch.cat([rot_homo, local_t], 3)  # (N,24,4,4)
    glob = [local[:, 0]]
    for i in range(1, JOINT_NUM):
        glob.append(torch.matmul(glob[int(parents[i])], local[:, i]))
    glob = torch.stack(glob, 1)
    elim = torch.matmul(glob[:, :, 0:3, 0:3], joints.unsqueeze(3))  # (N,24,3,1)
    elim = torch.cat([elim, torch.zeros(n, JOINT_NUM, 1, 1)], 2)
    elim = torch.cat([torch.zeros(n, JOINT_NUM, 4, 3), elim], 3)
    return glob - elim, glob


# ------------------------------------------------------------------------------------------------------------
# LinearBlendSkinning (src/LinearBlendSkinning.cpp)
# ------------------------------------------------------------------------------------------------------------

def skinning(weights, rest_shape, transforms, root_pos=None):
    """src/LinearBlendSkinning.cpp:445-483 (+cart2homo :505-516, homo2cart :538-553).  The homogeneous
    divide by h[3] = sum_j W[v,j] is kept.  root_pos (N,1,3) is added (:475)."""
    n, v = rest_shape.shape[0], rest_shape.shape[1]
    homo = torch.cat([rest_shape, torch.ones(n, v, 1)], 2)
    coeff = torch.tensordot(weights, transforms, ([1], [1]))  # (V,N,4,4)
    coeff = torch.transpose(coeff, 0, 1)
    vh = torch.matmul(coeff, homo.unsqueeze(3)).squeeze(3)  # (N,V,4)
    cart = (vh / vh[:, :, 3].unsqueeze(2))[:, :, 0:3]
    if root_pos is not None:
        cart = cart + root_pos.expand(-1, v, -1)
    return cart


# ------------------------------------------------------------------------------------------------------------
# SMPL facade (src/SMPL.cpp)
# ------------------------------------------------------------------------------------------------------------

@dataclass
class SmplModel:
    """Tensors of SMPL::init (src/SMPL.cpp:560-613) + the adjacency table of :619-640."""
    face_indices: torch.Tensor  # (F,3) int64, 1-based as stored
    shape_basis: torch.Tensor
    pose_basis: torch.Tensor
    templ: torch.Tensor
    joint_regressor: torch.Tensor
    parents: List[int]
    weights: torch.Tensor
    adjacent: List[List[int]] = field(default_factory=list)

    @staticmethod
    def from_params(p) -> "SmplModel":
        tree = np.asarray(p.kinematic_tree)
        parents = [int(x) if x < JOINT_NUM else -1 for x in tree[0].tolist()]
        faces = torch.as_tensor(np.asarray(p.face_indices, dtype=np.int64))
        nv = p.vertices_template.shape[0]
        adj: List[List[int]] = [[] for _ in range(nv)]
        for f, tri in enumerate((np.asarray(p.face_indices, dtype=np.int64) - 1).tolist()):
            for vi in tri:
                if f not in adj[vi]:
                    adj[vi].append(f)
        return SmplModel(faces, _t(p.shape_blend_shapes), _t(p.pose_blend_shapes), _t(p.vertices_template),
                         _t(p.joint_regressor), parents, _t(p.weights), adj)

    def to(self, dtype: torch.dtype) -> "SmplModel":
        """A copy with the floating-point tensors in `dtype` (face indices, parents and adjacency shared)."""
        return SmplModel(self.face_indices, self.shape_basis.to(dtype), self.pose_basis.to(dtype), self.templ.to(dtype),
                         self.joint_regressor.to(dtype), self.parents, self.weights.to(dtype), self.adjacent)


@dataclass
class ForwardResult:
    vertices: torch.Tensor  # (N,V,3)
    joints: torch.Tensor  # (N,24,3)   SMPL::getRestJoint
    rest_shape: torch.Tensor  # (N,V,3)    SMPL::getRestShape
    transforms: torch.Tensor  # (N,24,4,4) relative
    pose_rot: torch.Tensor
    global_transforms: torch.Tensor


def smpl_launch(model: SmplModel, beta: torch.Tensor, theta: torch.Tensor) -> ForwardResult:
    """SMPL::launch, src/SMPL.cpp:671-737.  beta (N,10); theta (N,25,3): row 0 = root translation
    (:726-727), rows 1..24 axis-angle (:685-686)."""
    pose_rot = rodrigues(theta[:, 1:, :])
    pbs = pose_blend(pose_blend_coeffs(pose_rot), model.pose_basis)
    sbs = shape_blend(beta, model.shape_basis)
    rest = linear_combine(model.templ, sbs, pbs)
    joints = joint_regress(model.templ, sbs, model.joint_regressor)
    rel, glob = world_transform(pose_rot, joints, model.parents)
    verts = skinning(model.weights, rest, rel, theta[:, :1, :])
    return ForwardResult(verts, joints, rest, rel, pose_rot, glob)


def _normalize(x: torch.Tensor) -> torch.Tensor:
    """torch.nn.functional.normalize(dim=-1), eps 1e-12: x / max(||x||, eps)."""
    return torch.nn.functional.normalize(x, dim=-1)


def calc_normal(model: SmplModel, verts0: torch.Tensor, face_idx: int) -> torch.Tensor:
    """SMPL::calcNormal, src/SMPL.cpp:518-525 (batch element 0; 1-based face storage, :520)."""
    ids = model.face_indices[face_idx] - 1
    fv = verts0[ids]
    return _normalize(torch.linalg.cross(fv[1] - fv[0], fv[2] - fv[0]))


def calc_vertex_normal(model: SmplModel, verts0: torch.Tensor, idx: int) -> torch.Tensor:
    """SMPL::calcVertexNormal, src/SMPL.cpp:527-535: normalize(sum_f (1/deg) n_f)."""
    faces = model.adjacent[idx]
    wgt = np.float32(1.0) / np.float32(len(faces))
    acc = torch.zeros(3)
    for f in faces:
        acc = acc + float(wgt) * calc_normal(model, verts0, f)
    return _normalize(acc)


# ------------------------------------------------------------------------------------------------------------
# IkTask (src/IkTask.cpp, include/smplpp/toolbox/GeometryUtils.h)
# ------------------------------------------------------------------------------------------------------------

def triangle_vertex_weights(pos: torch.Tensor, tri: torch.Tensor) -> torch.Tensor:
    """calcTriangleVertexWeights, include/smplpp/toolbox/GeometryUtils.h:42-52."""
    w = torch.stack([
        torch.linalg.cross(tri[1] - pos, tri[2] - pos).norm(),
        torch.linalg.cross(tri[2] - pos, tri[0] - pos).norm(),
        torch.linalg.cross(tri[0] - pos, tri[1] - pos).norm(),
    ])
    return w / w.sum()


@dataclass
class IkTask:
    """include/smplpp/IkTask.h:59-84 (defaults) — plain data + the methods of src/IkTask.cpp."""
    face_idx: int
    target_pos: torch.Tensor = field(default_factory=lambda: torch.zeros(3))
    target_normal: torch.Tensor = field(default_factory=lambda: torch.tensor([0.0, 0.0, 1.0]))
    pos_task_weight: float = 1.0
    normal_task_weight: float = 1.0
    phi_limit: float = 0.04
    normal_offset: float = 0.0
    vertex_weights: torch.Tensor = field(default_factory=lambda: torch.full((3,), 1.0 / 3.0))
    tangents: torch.Tensor = field(default_factory=lambda: torch.zeros(3, 2))
    phi: torch.Tensor = field(default_factory=lambda: torch.zeros(2))

    def face_vertices(self, model, verts0):
        return verts0[model.face_indices[self.face_idx] - 1]

    def calc_tangents(self, model, verts0):
        """src/IkTask.cpp:33-47 (detached)."""
        fv = self.face_vertices(model, verts0).detach().clone()
        t1 = fv[1] - fv[0]
        normal = torch.linalg.cross(t1, fv[2] - fv[0])
        t2 = torch.linalg.cross(normal, t1)
        self.tangents = torch.stack([_normalize(t1), _normalize(t2)], 1).detach()

    def calc_vertex_weights(self, model, verts0, actual_pos):
        """src/IkTask.cpp:49-57: the only path through which phi receives a gradient."""
        fv = self.face_vertices(model, verts0).detach().clone()
        pos = actual_pos + torch.matmul(self.tangents, self.phi)
        self.vertex_weights = triangle_vertex_weights(pos, fv)

    def calc_actual_normal(self, model, verts0):
        """src/IkTask.cpp:74-86"""
        ids = (model.face_indices[self.face_idx] - 1).tolist()
        acc = torch.zeros(3)
        for i in range(3):
            acc = acc + self.vertex_weights[i] * calc_vertex_normal(model, verts0, ids[i])
        return _normalize(acc)

    def calc_actual_pos(self, model, verts0):
        """src/IkTask.cpp:59-72"""
        fv = self.face_vertices(model, verts0)
        pos = torch.matmul(torch.transpose(fv, 0, 1), self.vertex_weights)
        if self.normal_offset > 0.0:
            pos = pos + self.normal_offset * self.calc_actual_normal(model, verts0)
        return pos


# ------------------------------------------------------------------------------------------------------------
# VPoser decoder (src/VPoser.cpp)
# ------------------------------------------------------------------------------------------------------------

def rotmat_to_axis_angle(rot: torch.Tensor) -> torch.Tensor:
    """convertRotMatToAxisAngle, src/VPoser.cpp:25-120.  (N,3,3) -> (N,3).  Branches are evaluated on
    gathered subsets exactly like the reference so that autograd only sees the selected branch."""
    eps = FLT_EPS
    eps_sqrt = math.sqrt(eps)
    eps_sqrt2 = math.sqrt(eps_sqrt)
    n = rot.shape[0]
    trace = rot.diagonal(0, 1, 2).sum(-1)
    theta = torch.arccos((1.0 - eps) * 0.5 * (trace - 1.0))
    w = torch.stack([rot[:, 2, 1] - rot[:, 1, 2], rot[:, 0, 2] - rot[:, 2, 0], rot[:, 1, 0] - rot[:, 0, 1]], 1)
    near_pi = (1.0 + trace < eps_sqrt2)
    idx_a = torch.nonzero(near_pi).flatten()
    idx_b = torch.nonzero(~near_pi).flatten()
    out = torch.zeros(n, 3)
    if idx_a.numel() > 0:
        ra, tra, tha = rot[idx_a], trace[idx_a], theta[idx_a]
        s = (2.0 * ra.diagonal(0, 1, 2) + (1.0 - tra).view(-1, 1).expand(-1, 3)) / (3.0 - tra).view(-1, 1)
        tn = torch.sqrt(s + eps) * tha.view(-1, 1)
        with torch.no_grad():
            sign = torch.ones_like(tn)
            a1 = tha > math.pi - 1e-4
            tnd, wd = tn.detach(), w[idx_a].detach()
            for r in range(idx_a.numel()):
                if bool(a1[r]):  # :62-96
                    if tnd[r, 0] > 0.0:
                        if ra[r, 0, 1] + ra[r, 1, 0] < 0.0:
                            sign[r, 1] = -1.0
                        if ra[r, 0, 2] + ra[r, 2, 0] < 0.0:
                            sign[r, 2] = -1.0
                    elif tnd[r, 1] > 0.0:
                        if ra[r, 1, 2] + ra[r, 2, 1] < 0.0:
                            sign[r, 2] = -1.0
                else:  # :98-101 element-wise
                    for k in range(3):
                        if not bool(wd[r, k] >= 0.0):
                            sign[r, k] = -1.0
        out = out.index_put((idx_a,), tn * sign)
    if idx_b.numel() > 0:
        trb, thb, wb = trace[idx_b], theta[idx_b], w[idx_b]
        near0 = torch.abs(3.0 - trb) < eps_sqrt
        i0 = torch.nonzero(near0).flatten()
        i1 = torch.nonzero(~near0).flatten()
        res = torch.zeros(idx_b.numel(), 3)
        if i0.numel() > 0:  # :105-111
            t0 = thb[i0]
            res = res.index_put((i0,), 0.5 * wb[i0] * (1.0 + torch.pow(t0, 2) / 6.0
                                                        + torch.pow(t0, 4) * 7.0 / 360.0).view(-1, 1))
        if i1.numel() > 0:  # :112-116
            t1 = thb[i1]
            res = res.index_put((i1,), wb[i1] * torch.div(t1, 2.0 * torch.sin(t1)).view(-1, 1))
        out = out.index_put((idx_b,), res)
    return out


def cont_rot_repr_decode(x: torch.Tensor) -> torch.Tensor:
    """ContinousRotReprDecoderImpl::forward, src/VPoser.cpp:129-141. (N,126) -> (N*21,3,3), columns b1,b2,b3."""
    r = x.reshape(-1, 3, 2)
    c1, c2 = r[:, :, 0], r[:, :, 1]
    a1 = torch.nn.functional.normalize(c1, dim=1)
    a2 = torch.nn.functional.normalize(c2 - (a1 * c2).sum(1, True) * a1, dim=-1)
    a3 = torch.linalg.cross(a1, a2, dim=1)
    return torch.stack([a1, a2, a3], -1).view(-1, 3, 3)


@dataclass
class VPoserDecoder:
    """VPoserDecoderImpl, src/VPoser.cpp:143-167 (eval mode: Dropout = identity)."""
    w0: torch.Tensor
    b0: torch.Tensor
    w3: torch.Tensor
    b3: torch.Tensor
    w5: torch.Tensor
    b5: torch.Tensor

    @staticmethod
    def from_params(p: dict) -> "VPoserDecoder":
        return VPoserDecoder(*[_t(p[k]) for k in ("decoder_net.0.weight", "decoder_net.0.bias", "decoder_net.3.weight",
                                                  "decoder_net.3.bias", "decoder_net.5.weight", "decoder_net.5.bias")])

    def to(self, dtype: torch.dtype) -> "VPoserDecoder":
        """A copy with the weights in `dtype`."""
        return VPoserDecoder(*[w.to(dtype) for w in (self.w0, self.b0, self.w3, self.b3, self.w5, self.b5)])

    def mlp(self, z):
        lrelu = torch.nn.functional.leaky_relu
        h = lrelu(torch.nn.functional.linear(z, self.w0, self.b0), 0.01)
        h = lrelu(torch.nn.functional.linear(h, self.w3, self.b3), 0.01)
        return torch.nn.functional.linear(h, self.w5, self.b5)

    def forward(self, z: torch.Tensor) -> torch.Tensor:
        """(B,32) -> (B,21,3)"""
        b = z.shape[0]
        return rotmat_to_axis_angle(cont_rot_repr_decode(self.mlp(z))).view(b, -1, 3)


# ------------------------------------------------------------------------------------------------------------
# IK iteration (node/node.cpp:705-968)
# ------------------------------------------------------------------------------------------------------------

def cholesky_solve_neg(A: np.ndarray, b: np.ndarray) -> np.ndarray:
    """deltaConfig = -LLT(A).solve(b), node/node.cpp:933-938 (fp64)."""
    L = np.linalg.cholesky(A)
    y = np.linalg.solve(L, -b)
    return np.linalg.solve(L.T, y)


def solve_box_qp(A: np.ndarray, b: np.ndarray, lo: np.ndarray, hi: np.ndarray) -> np.ndarray:
    """min 1/2 x'Ax + b'x, lo <= x <= hi (node/node.cpp:909-930; QLD replaced, see module docstring).
    fp64 primal active-set; exact for strictly convex problems."""
    n = b.shape[0]
    x = np.clip(np.zeros(n), lo, hi)
    state = np.zeros(n, dtype=np.int64)  # 0 free, -1 lower, +1 upper, 2 pinned
    state[lo == hi] = 2
    at_minimiser = False  # last step was a full unblocked Newton step: go straight to the multiplier test
    for _ in range(20 * n + 50):
        g = A @ x + b
        free = np.nonzero(state == 0)[0]
        d = np.zeros(n)
        if free.size and not at_minimiser:
            d[free] = cholesky_solve_neg(A[np.ix_(free, free)], g[free])
        if at_minimiser or np.abs(d).max(initial=0.0) <= 1e-14 * max(1.0, np.abs(x).max(initial=0.0)):
            viol = np.where(state == -1, -g, np.where(state == 1, g, 0.0))
            k = int(np.argmax(viol))
            if viol[k] <= 1e-12:
                return x
            state[k] = 0
            at_minimiser = False
            continue
        alpha, block, side = 1.0, -1, 0
        for i in free:
            if d[i] > 0 and np.isfinite(hi[i]):
                a = (hi[i] - x[i]) / d[i]
                if a < alpha:
                    alpha, block, side = a, i, 1
            elif d[i] < 0 and np.isfinite(lo[i]):
                a = (lo[i] - x[i]) / d[i]
                if a < alpha:
                    alpha, block, side = a, i, -1
        x[free] += alpha * d[free]
        at_minimiser = block < 0
        if block >= 0:
            x[block] = hi[block] if side > 0 else lo[block]
            state[block] = side
    raise RuntimeError("box QP did not converge")


@dataclass
class IkResult:
    e: np.ndarray  # (4n,) fp64
    J: np.ndarray  # (4n, dim) fp64
    A: np.ndarray
    b: np.ndarray
    delta: np.ndarray
    theta_state: np.ndarray  # updated g_theta (in the dtype of the call)
    beta: np.ndarray  # updated g_beta (in the dtype of the call)
    vertex_weights: np.ndarray  # (n,3) after the re-weighting of node.cpp:803-804
    actual_pos: np.ndarray  # (n,3) marker positions (pre-update mesh, with the normal offset)
    skipped: bool
    theta_full: np.ndarray  # (25,3) theta fed to SMPL::launch


def assemble_theta(g_theta: torch.Tensor, vposer: Optional[VPoserDecoder]) -> torch.Tensor:
    """node/node.cpp:761-776.  VPoser state (44,) = [trans 3 | root aa 3 | latent 32 | hands 6]."""
    if vposer is None:
        return g_theta.view(JOINT_NUM + 1, 3)
    body = vposer.forward(g_theta[6:6 + LATENT_DIM].view(1, -1))[0]  # (21,3)
    return torch.cat([g_theta[0:3].view(1, 3), g_theta[3:6].view(1, 3), body,
                      g_theta[LATENT_DIM + 6:LATENT_DIM + 9].view(1, 3),
                      g_theta[LATENT_DIM + 9:LATENT_DIM + 12].view(1, 3)], 0)


def ik_iteration(model: SmplModel, tasks: List[IkTask], theta_state: np.ndarray, beta: np.ndarray,
                 vposer: Optional[VPoserDecoder] = None, optimize_beta: bool = False, enable_qp: bool = True,
                 skip_if_too_few: bool = False, dtype: torch.dtype = torch.float32) -> IkResult:
    """One pass of node/node.cpp:705-968 for ONE frame.  `tasks` carry targets/weights/limits and are
    updated in place (vertex_weights, tangents) as the node does.

    dtype=torch.float32 is the reference's arithmetic.  dtype=torch.float64 runs the same operations in double precision
    (a reference for the reference, where float32 autograd is ill-conditioned): the model and the VPoser decoder must then
    be float64 copies (SmplModel.to / VPoserDecoder.to), the tensors of `tasks` are cast to float64 in place, and the
    torch default dtype is float64 for the duration of the call (the restated reference builds constants with
    torch.zeros / torch.eye) and restored afterwards, also when the call raises."""
    if model.templ.dtype != dtype or (vposer is not None and vposer.w0.dtype != dtype):
        raise TypeError("ik_iteration(dtype=%s) needs the model and the decoder in that dtype (use .to(dtype))" % dtype)
    prev = torch.get_default_dtype()
    torch.set_default_dtype(dtype)
    try:
        if dtype != torch.float32:
            for t in tasks:
                for k in ("target_pos", "target_normal", "vertex_weights", "tangents", "phi"):
                    setattr(t, k, getattr(t, k).to(dtype))
        return _ik_iteration(model, tasks, theta_state, beta, vposer, optimize_beta, enable_qp, skip_if_too_few, dtype)
    finally:
        torch.set_default_dtype(prev)


def _ik_iteration(model, tasks, theta_state, beta, vposer, optimize_beta, enable_qp, skip_if_too_few, dtype):
    n = len(tasks)
    np_dtype = np.float32 if dtype == torch.float32 else np.float64
    g_theta = torch.tensor(np.asarray(theta_state, dtype=np_dtype).reshape(-1), requires_grad=True)
    g_beta = torch.tensor(np.asarray(beta, dtype=np_dtype).reshape(-1), requires_grad=bool(optimize_beta))
    theta_dim = g_theta.numel()
    assert theta_dim == (LATENT_DIM + 12 if vposer is not None else 3 * (JOINT_NUM + 1))
    phi_dim, beta_dim = 2 * n, (SHAPE_DIM if optimize_beta else 0)
    dim = theta_dim + phi_dim + beta_dim
    for t in tasks:  # :716-733
        t.phi = torch.zeros(2, requires_grad=t.phi_limit > 0.0)
    theta = assemble_theta(g_theta, vposer)
    fwd = smpl_launch(model, g_beta.view(1, -1), theta.view(1, JOINT_NUM + 1, 3))
    verts0 = fwd.vertices[0]
    valid = sum(1 for t in tasks if t.pos_task_weight > 0.0)
    skipped = bool(skip_if_too_few and valid < n // 2)  # :785

    e = np.zeros(4 * n)
    J = np.zeros((4 * n, dim))
    actual = np.zeros((n, 3), dtype=np.float32)

    def rows(scalar_fn, row, ti, task):
        wrt = [g_theta] + ([task.phi] if task.phi_limit > 0.0 else []) + ([g_beta] if optimize_beta else [])
        grads = torch.autograd.grad(scalar_fn, wrt, retain_graph=True, allow_unused=True)
        k = 0
        J[row, :theta_dim] = grads[k].detach().numpy().astype(np.float64) if grads[k] is not None else 0.0
        k += 1
        if task.phi_limit > 0.0:
            if grads[k] is not None:
                J[row, theta_dim + 2 * ti: theta_dim + 2 * ti + 2] = grads[k].detach().numpy().astype(np.float64)
            k += 1
        if optimize_beta and grads[k] is not None:
            J[row, theta_dim + phi_dim:] = grads[k].detach().numpy().astype(np.float64)

    for ti, task in enumerate(tasks):
        task.calc_tangents(model, verts0)  # :803
        task.calc_vertex_weights(model, verts0, task.calc_actual_pos(model, verts0).detach().clone())  # :804
        pos = task.calc_actual_pos(model, verts0)
        actual[ti] = pos.detach().numpy()
        pos_err = task.pos_task_weight * (pos - task.target_pos)  # :807
        e[4 * ti: 4 * ti + 3] = pos_err.detach().numpy().astype(np.float64)
        for i in range(3):  # :823-847
            rows(pos_err[i], 4 * ti + i, ti, task)
        if task.normal_task_weight > 0.0:  # :810-820, :848-873
            n_err = task.normal_task_weight * (torch.dot(task.calc_actual_normal(model, verts0),
                                                         task.target_normal) + 1.0)
            e[4 * ti + 3] = float(n_err.detach())
            rows(n_err, 4 * ti + 3, ti, task)

    A = J.T @ J  # :884-893
    b = J.T @ e
    e_sq = float(e @ e)
    reg = np.concatenate([np.full(theta_dim, 1e-3), np.full(phi_dim, 1e-1), np.full(beta_dim, 1e-3)])
    A[np.diag_indices(dim)] += reg + e_sq
    if vposer is not None:  # :895-904
        wv = np.full(theta_dim, 1e-5)
        wv[:6] = 0.0
        wv[-6:] = 1e3
        A[np.arange(theta_dim), np.arange(theta_dim)] += wv
        b[:theta_dim] += wv * g_theta.detach().numpy().astype(np.float64)
    if enable_qp:  # :907-930
        lo = np.full(dim, -np.inf)
        hi = np.full(dim, np.inf)
        for ti, task in enumerate(tasks):
            lo[theta_dim + 2 * ti: theta_dim + 2 * ti + 2] = -task.phi_limit
            hi[theta_dim + 2 * ti: theta_dim + 2 * ti + 2] = task.phi_limit
        if optimize_beta:
            lo[theta_dim + phi_dim:] = -0.5
            hi[theta_dim + phi_dim:] = 0.5
        delta = solve_box_qp(A, b, lo, hi)
    else:  # :933-938
        delta = cholesky_solve_neg(A, b)

    new_theta = g_theta.detach().numpy().copy()
    new_beta = g_beta.detach().numpy().copy()
    if not skipped:  # :946-968
        new_theta = new_theta + delta[:theta_dim].astype(np_dtype)
        if optimize_beta:
            new_beta = new_beta + delta[theta_dim + phi_dim:].astype(np_dtype)
    for t in tasks:
        t.phi = t.phi.detach()
        t.vertex_weights = t.vertex_weights.detach()
    vw = np.stack([t.vertex_weights.numpy() for t in tasks]) if n else np.zeros((0, 3), np.float32)
    return IkResult(e, J, A, b, delta, new_theta, new_beta, vw, actual, skipped, theta.detach().numpy())


# ------------------------------------------------------------------------------------------------------------
# numpy conveniences for the tests
# ------------------------------------------------------------------------------------------------------------

# ----------------------------------------------------------------------------------------------------------------
# projection onto the mesh (node/node.cpp:970-1001)
# ----------------------------------------------------------------------------------------------------------------
def closest_points_on_triangles(p: np.ndarray, a: np.ndarray, b: np.ndarray, c: np.ndarray) -> np.ndarray:
    """Closest point of every triangle (a_i, b_i, c_i) to the single point p, float64, vectorised over triangles.

    The reference calls igl::point_mesh_squared_distance (node/node.cpp:976-978); libigl v2.4.0
    (cmake/libigl.cmake:9) is a third-party dependency that is NOT under /root/reference and the reference has no
    test or golden vector for this call: "parity unpinned" at this boundary.  Its published algorithm is the exact
    point-triangle distance over the seven Voronoi regions of the triangle (vertex / edge / face), found through an
    AABB tree; the exact minimiser is unique, so the restatement is the region test of Ericson, "Real-Time Collision
    Detection", 5.1.5, evaluated on every triangle (the tree only prunes)."""
    ab, ac, ap = b - a, c - a, p - a
    d1, d2 = (ab * ap).sum(1), (ac * ap).sum(1)
    bp = p - b
    d3, d4 = (ab * bp).sum(1), (ac * bp).sum(1)
    cp = p - c
    d5, d6 = (ab * cp).sum(1), (ac * cp).sum(1)
    vc = d1 * d4 - d3 * d2
    vb = d5 * d2 - d1 * d6
    va = d3 * d6 - d5 * d4
    out = np.empty_like(a)
    done = np.zeros(len(a), dtype=bool)

    def put(mask, val):
        m = mask & ~done
        out[m] = val[m]
        done[m] = True

    with np.errstate(divide="ignore", invalid="ignore"):
        put((d1 <= 0) & (d2 <= 0), a)
        put((d3 >= 0) & (d4 <= d3), b)
        put((vc <= 0) & (d1 >= 0) & (d3 <= 0), a + ab * (d1 / (d1 - d3))[:, None])
        put((d6 >= 0) & (d5 <= d6), c)
        put((vb <= 0) & (d2 >= 0) & (d6 <= 0), a + ac * (d2 / (d2 - d6))[:, None])
        put((va <= 0) & ((d4 - d3) >= 0) & ((d5 - d6) >= 0), b + (c - b) * ((d4 - d3) / ((d4 - d3) + (d5 - d6)))[:, None])
        denom = 1.0 / (va + vb + vc)
        put(np.ones(len(a), dtype=bool), a + ab * (vb * denom)[:, None] + ac * (vc * denom)[:, None])
    return out


def project_points_on_mesh(verts: np.ndarray, faces0: np.ndarray, points: np.ndarray):
    """node/node.cpp:970-1001 for one frame: closest face (0-based, lowest index on ties), closest point, squared
    distance and the re-seated IkTask::vertexWeights_ = calcTriangleVertexWeights(closest, face)
    (GeometryUtils.h:42-52).  verts (V,3), faces0 (F,3) 0-based, points (n,3); float64 inside."""
    v = np.asarray(verts, dtype=np.float64)
    a, b, c = v[faces0[:, 0]], v[faces0[:, 1]], v[faces0[:, 2]]
    n = len(points)
    face = np.zeros(n, dtype=np.int64)
    closest = np.zeros((n, 3))
    sq = np.zeros(n)
    weights = np.zeros((n, 3))
    for i, p in enumerate(np.asarray(points, dtype=np.float64)):
        q = closest_points_on_triangles(p, a, b, c)
        d2 = ((q - p) ** 2).sum(1)
        k = int(np.argmin(d2))  # first minimum = lowest face index
        face[i], closest[i], sq[i] = k, q[k], d2[k]
        tri = np.stack([a[k], b[k], c[k]])
        w = np.array([np.linalg.norm(np.cross(tri[1] - q[k], tri[2] - q[k])),
                      np.linalg.norm(np.cross(tri[2] - q[k], tri[0] - q[k])),
                      np.linalg.norm(np.cross(tri[0] - q[k], tri[1] - q[k]))])
        weights[i] = w / w.sum()
    return face, closest, sq, weights


def forward_numpy(model: SmplModel, beta: np.ndarray, theta: np.ndarray, chunk: int = 64):
    """Batched forward without autograd; returns (vertices, joints, rest_shape, transforms) as float32 arrays."""
    outs = ([], [], [], [])
    with torch.no_grad():
        for s in range(0, beta.shape[0], chunk):
            r = smpl_launch(model, _t(beta[s:s + chunk]), _t(theta[s:s + chunk]))
            for o, t in zip(outs, (r.vertices, r.joints, r.rest_shape, r.transforms)):
                o.append(t.numpy())
    return tuple(np.concatenate(o, 0) for o in outs)


def sweep_grid_points(verts: np.ndarray):
    """toolbox/GridUtils.hpp:28-63 + node/node.cpp:1031-1049: grid_idx_min = floor(min corner / GRID_SCALE), grid_num from
    ceil(max corner / GRID_SCALE) (float positions divided by float(0.025)), and the grid points float(0.025) * index in the
    reference's loop order (x outermost, z innermost), as float64 (N, 3)."""
    v32 = np.asarray(verts, dtype=np.float32)
    gs32 = np.float32(0.025)
    lo = np.floor(v32.min(0) / gs32).astype(np.int32)
    hi = np.ceil(v32.max(0) / gs32).astype(np.int32)
    num = hi - lo + 1
    ix, iy, iz = np.meshgrid(np.arange(num[0]), np.arange(num[1]), np.arange(num[2]), indexing="ij")
    idx = np.stack([ix, iy, iz], -1).reshape(-1, 3) + lo[None]
    return lo, num, (gs32 * idx.astype(np.float32)).astype(np.float64)


def winding_number(verts: np.ndarray, faces0: np.ndarray, pts: np.ndarray):
    """Generalized winding number of a triangle mesh at pts (N, 3): sum of the signed solid angles of the faces / 4 pi
    (Van Oosterom & Strackee 1983; what igl::winding_number evaluates, node/node.cpp:1052 - libigl is un-vendored)."""
    v = np.asarray(verts, dtype=np.float32).astype(np.float64)
    A, B, C = v[faces0[:, 0]], v[faces0[:, 1]], v[faces0[:, 2]]
    pts = np.asarray(pts, dtype=np.float64)
    w = np.zeros(len(pts))
    for s in range(0, len(pts), 256):  # chunks keep the (points, faces, 3) temporaries small
        p = pts[s:s + 256, None, :]
        a, b, c = A[None] - p, B[None] - p, C[None] - p
        la, lb, lc = np.linalg.norm(a, axis=2), np.linalg.norm(b, axis=2), np.linalg.norm(c, axis=2)
        det = np.einsum("pfi,pfi->pf", a, np.cross(b, c))
        den = la * lb * lc + np.einsum("pfi,pfi->pf", a, b) * lc + np.einsum("pfi,pfi->pf", b, c) * la \
            + np.einsum("pfi,pfi->pf", c, a) * lb
        w[s:s + 256] = (2.0 * np.arctan2(det, den)).sum(1) / (4.0 * np.pi)
    return w


def sweep_grid(verts: np.ndarray, faces0: np.ndarray):
    """node/node.cpp:1023-1073 for one frame: the 2.5 cm grid around the mesh and the winding number of every grid point
    (float64 inside).  Returns (grid_idx_min (3,), grid_num (3,), winding (nx, ny, nz)); a cell is occupied where
    winding > 0.5 (node.cpp:1056).  NOTE: the reference stores libigl's result in an Eigen::VectorXi (node.cpp:1051) -
    whether libigl rounds or truncates into it cannot be checked here, so the oracle keeps the real number."""
    lo, num, pts = sweep_grid_points(verts)
    return lo, num, winding_number(verts, faces0, pts).reshape(num[0], num[1], num[2])
