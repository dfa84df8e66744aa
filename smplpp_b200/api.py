"""Host-side mirror of the reference's operator interface for the hot path, over the C-ABI library.

Same class and method names, argument meaning and error behaviour as the reference:
    smplpp::SMPL                 include/smplpp/SMPL.h:210-270        -> SMPL
    smplpp::BlendShape           include/smplpp/BlendShape.h:221-244  -> BlendShape
    smplpp::JointRegression      include/smplpp/JointRegression.h     -> JointRegression
    smplpp::WorldTransformation  include/smplpp/WorldTransformation.h -> WorldTransformation
    smplpp::LinearBlendSkinning  include/smplpp/LinearBlendSkinning.h -> LinearBlendSkinning
Tensors are torch CUDA float32 tensors (torch is used for device memory and streams only; every computation
is a call into smplpp_b200/libsmplpp_b200.so).  Shape violations raise SmplppError with the reference's
message text (e.g. "BlendShape Error: Failed to set beta!", src/BlendShape.cpp:340).
"""
from __future__ import annotations

import ctypes as C
import json
from typing import Optional

import numpy as np
import torch

from . import capi
from .capi import SmplppError, check, lib

JOINT_NUM = 24
SHAPE_BASIS_DIM = 10
POSE_BASIS_DIM = 207
FACE_INDEX_NUM = 13776
LATENT_DIM = 32


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _dev_f32(x, device) -> torch.Tensor:
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=torch.float32).contiguous()
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32), device=device)


def _np_f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _require_cuda(device: torch.device) -> None:
    if device.type != "cuda" or not torch.cuda.is_available():
        raise SmplppError("SMPL Error: Failed to fetch device index! (smplpp_b200 needs a CUDA device; "
                          "there is no CPU fallback)")


class _PinnedBlock:
    """Owns one smplpp_host_alloc allocation; freed when the last numpy view goes away."""

    def __init__(self, nbytes: int):
        self.ptr = C.c_void_p()
        check(lib().smplpp_host_alloc(C.byref(self.ptr), C.c_size_t(max(1, nbytes))))
        self.nbytes = nbytes

    def __del__(self):
        if getattr(self, "ptr", None) and capi._lib is not None:
            capi._lib.smplpp_host_free(self.ptr)
            self.ptr = None


def pinned_empty(shape, dtype=np.float32) -> np.ndarray:
    """numpy array in page-locked host memory (smplpp_host_alloc): the DMA source/target of the host-buffer calls."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape))
    block = _PinnedBlock(n * dtype.itemsize)
    buf = (C.c_char * max(1, block.nbytes)).from_address(block.ptr.value)
    buf._smplpp_owner = block  # keeps the allocation alive as long as the buffer (numpy's base) is
    return np.frombuffer(buf, dtype=dtype, count=n).reshape(shape)


class SMPL:
    """smplpp::SMPL (src/SMPL.cpp).  `launch` runs K1 (pose features + chain) and K2 (fused blend + skinning)."""

    def __init__(self, params=None, device="cuda:0"):
        self.m__device = torch.device(device)
        self.m__modelPath = None
        self._h = None
        self._params = params
        self._beta = self._theta = None
        self._vertices = self._joints = self._rest = self._transforms = None
        self._ws = None
        if params is not None:
            self.init()

    # -- setters / getters of SMPL.h:250-264 --
    def setDevice(self, device):
        device = torch.device(device)
        if device.index is None:
            raise SmplppError("SMPL Error: Failed to fetch device index!")  # SMPL.cpp:299
        self.m__device = device

    def getDevice(self):
        return self.m__device

    def setModelPath(self, path: str):
        import os
        if not os.path.exists(path):
            raise SmplppError("SMPL Error: Failed to initialize model path!")  # SMPL.cpp:337
        self.m__modelPath = path

    def init(self):
        """SMPL::init (src/SMPL.cpp:560-643): load the model arrays and pack them on the device."""
        _require_cuda(self.m__device)
        p = self._params
        if p is None:
            if self.m__modelPath is None:
                raise SmplppError("SMPL Error: Cannot initialize a SMPL model!")  # SMPL.cpp:616
            p = load_model_file(self.m__modelPath)
            self._params = p
        arrs = dict(
            face_indices=np.ascontiguousarray(p.face_indices, dtype=np.int32),
            shape=_np_f32(p.shape_blend_shapes), pose=_np_f32(p.pose_blend_shapes),
            templ=_np_f32(p.vertices_template), jreg=_np_f32(p.joint_regressor),
            tree=np.ascontiguousarray(p.kinematic_tree, dtype=np.int64), weights=_np_f32(p.weights))
        V = arrs["templ"].shape[0]
        if arrs["shape"].shape != (V, 3, SHAPE_BASIS_DIM):
            raise SmplppError("SMPL Error: Shape parameter dimensions are invalid: %d != %d"
                              % (arrs["shape"].shape[-1], SHAPE_BASIS_DIM))  # SMPL.cpp:581
        if arrs["pose"].shape != (V, 3, POSE_BASIS_DIM):
            raise SmplppError("SMPL Error: Pose parameter dimensions are invalid: %d != %d"
                              % (arrs["pose"].shape[-1], POSE_BASIS_DIM))  # SMPL.cpp:588
        desc = capi.ModelDesc(
            V, arrs["face_indices"].shape[0], arrs["face_indices"].ctypes.data_as(capi.c_i32p),
            arrs["shape"].ctypes.data_as(capi.c_f32p), arrs["pose"].ctypes.data_as(capi.c_f32p),
            arrs["templ"].ctypes.data_as(capi.c_f32p), arrs["jreg"].ctypes.data_as(capi.c_f32p),
            arrs["tree"].ctypes.data_as(capi.c_i64p), arrs["weights"].ctypes.data_as(capi.c_f32p))
        h = C.c_void_p()
        with torch.cuda.device(self.m__device):
            check(lib().smplpp_model_create(C.byref(desc), C.byref(h)))
        self._h = h
        self.vertex_num = V
        self._faces_host = arrs["face_indices"]
        self._face_dev = None
        self._adjacent = None

    @classmethod
    def from_json_native(cls, path: str, device="cuda:0") -> "SMPL":
        """setModelPath + init through the C-ABI loader smplpp_model_load_json (the C++ twin of load_model_file):
        what the header-only facade's SMPL::init() calls."""
        self = cls(None, device)
        _require_cuda(self.m__device)
        self.m__modelPath = path
        h = C.c_void_p()
        with torch.cuda.device(self.m__device):
            loader = lib().smplpp_model_load_npz if path.endswith(".npz") else lib().smplpp_model_load_json
            check(loader(path.encode(), C.byref(h)))
        self._h = h
        self.vertex_num = int(lib().smplpp_model_vertex_num(h))
        self._faces_host = np.ascontiguousarray(read_json_arrays(path, ["face_indices"])["face_indices"], dtype=np.int32)
        self._face_dev = None
        self._adjacent = None
        return self

    def __del__(self):
        try:
            if getattr(self, "_h", None) is not None and capi is not None and capi._lib is not None:
                capi._lib.smplpp_model_destroy(self._h)
                self._h = None
        except Exception:  # interpreter shutdown: module globals may already be gone
            pass

    @property
    def handle(self):
        if self._h is None:
            raise SmplppError("SMPL Error: Cannot launch a SMPL model!")
        return self._h

    def _workspace(self, batch: int) -> torch.Tensor:
        need = lib().smplpp_forward_workspace_bytes(self.handle, C.c_int64(batch))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.m__device)
        return self._ws

    def launch(self, beta, theta, want_transforms: bool = False):
        """SMPL::launch (src/SMPL.cpp:671-737).  beta (N,10) [or (10,)/(1,10) shared by all frames],
        theta (N,25,3): row 0 root translation, rows 1..24 axis-angle."""
        theta = _dev_f32(theta, self.m__device)
        beta = _dev_f32(beta, self.m__device)
        if theta.dim() != 3 or theta.shape[1:] != (JOINT_NUM + 1, 3):
            raise SmplppError("SMPL Error: Cannot launch a SMPL model!")  # SMPL.cpp:676
        n = theta.shape[0]
        if beta.dim() == 1:
            beta = beta.view(1, -1)
        if beta.shape[-1] != SHAPE_BASIS_DIM or beta.shape[0] not in (1, n):
            raise SmplppError("BlendShape Error: Failed to set beta!")  # BlendShape.cpp:340
        stride = 0 if (beta.shape[0] == 1 and n > 1) else SHAPE_BASIS_DIM
        self._beta, self._theta, self._beta_stride = beta, theta, stride
        V = self.vertex_num
        self._vertices = torch.empty((n, V, 3), dtype=torch.float32, device=self.m__device)
        self._joints = torch.empty((n, JOINT_NUM, 3), dtype=torch.float32, device=self.m__device)
        self._transforms = (torch.empty((n, JOINT_NUM, 4, 4), dtype=torch.float32, device=self.m__device)
                            if want_transforms else None)
        self._rest = None
        ws = self._workspace(n)
        with torch.cuda.device(self.m__device):
            check(lib().smplpp_forward(self.handle, _stream(self.m__device), C.c_int64(n), _ptr(beta),
                                       C.c_int64(stride), _ptr(theta), _ptr(self._vertices), _ptr(self._joints),
                                       _ptr(self._transforms), None, _ptr(ws), C.c_size_t(ws.numel())))

    def launch_host(self, beta: np.ndarray, theta: np.ndarray, want_joints: bool = True, out_vertices=None,
                    out_joints=None):
        """Host-buffer variant of launch + getVertex (+getRestJoint): numpy in, numpy out, copies included.
        `out_vertices` / `out_joints` may be caller-owned float32 arrays (page-locked ones from `pinned_empty`
        are DMA targets themselves; pageable ones are staged)."""
        beta, theta = _np_f32(beta), _np_f32(theta)
        if theta.ndim != 3 or theta.shape[1:] != (JOINT_NUM + 1, 3):
            raise SmplppError("SMPL Error: Cannot launch a SMPL model!")  # SMPL.cpp:676
        n = theta.shape[0]
        if beta.ndim == 1:
            beta = beta.reshape(1, -1)
        if beta.shape[-1] != SHAPE_BASIS_DIM or beta.shape[0] not in (1, n):
            raise SmplppError("BlendShape Error: Failed to set beta!")  # BlendShape.cpp:340
        stride = 0 if (beta.shape[0] == 1 and n > 1) else SHAPE_BASIS_DIM
        verts = out_vertices if out_vertices is not None else np.empty((n, self.vertex_num, 3), np.float32)
        joints = out_joints if out_joints is not None else (np.empty((n, JOINT_NUM, 3), np.float32) if want_joints else None)
        for a, shape in ((verts, (n, self.vertex_num, 3)), (joints, (n, JOINT_NUM, 3))):
            if a is not None and (a.dtype != np.float32 or a.shape != shape or not a.flags.c_contiguous):
                raise SmplppError("SMPL Error: Cannot launch a SMPL model! (output buffer shape/dtype)")
        with torch.cuda.device(self.m__device):
            check(lib().smplpp_forward_host(self.handle, C.c_int64(n), beta.ctypes.data_as(capi.c_f32p),
                                            C.c_int64(stride), theta.ctypes.data_as(capi.c_f32p),
                                            verts.ctypes.data_as(capi.c_f32p),
                                            joints.ctypes.data_as(capi.c_f32p) if joints is not None else None))
        return verts, joints

    def _launched(self, what):
        if self._vertices is None:
            raise SmplppError(what)

    def getVertex(self) -> torch.Tensor:
        self._launched("LinearBlendSknning Error: Failed to get vertices of new pose!")  # LinearBlendSkinning.cpp:409
        return self._vertices.clone()

    def projectPoints(self, points, vertices: Optional[torch.Tensor] = None, want_weights: bool = True):
        """Closest point on the posed mesh for (B, n, 3) points: the igl::point_mesh_squared_distance call and the
        faceIdx_ / calcVertexWeights re-seat of node/node.cpp:970-1001, batched over frames.  `vertices` defaults to
        the last launch.  Returns (face_idx (B,n) int32 0-based, closest (B,n,3), sq_dist (B,n), weights (B,n,3))."""
        dev = self.m__device
        if vertices is None:
            self._launched("LinearBlendSknning Error: Failed to get vertices of new pose!")
            vertices = self._vertices
        v = _dev_f32(vertices, dev)
        pts = _dev_f32(points, dev)
        if pts.dim() != 3 or pts.shape[0] != v.shape[0] or pts.shape[2] != 3:
            raise SmplppError("IkTask Error: Failed to project points onto the mesh!")
        b, n = pts.shape[0], pts.shape[1]
        face = torch.empty((b, n), dtype=torch.int32, device=dev)
        closest = torch.empty((b, n, 3), dtype=torch.float32, device=dev)
        sq = torch.empty((b, n), dtype=torch.float32, device=dev)
        w = torch.empty((b, n, 3), dtype=torch.float32, device=dev) if want_weights else None
        with torch.cuda.device(dev):
            check(lib().smplpp_closest_points(self.handle, _stream(dev), C.c_int64(b), C.c_int64(n), _ptr(v), _ptr(pts),
                                              C.c_void_p(face.data_ptr()), _ptr(closest), _ptr(sq), _ptr(w)))
        return face, closest, sq, w

    def sweepGrid(self, vertices: Optional[torch.Tensor] = None, index: int = 0):
        """Sweep-grid occupancy of one posed mesh (node/node.cpp:1023-1073): the 2.5 cm grid around the mesh of batch
        element `index` and the winding number of every grid point.  Returns (grid_idx_min (3,) int32, grid_num (3,)
        int32, winding (nx, ny, nz) float32, occupied (nx, ny, nz) bool); grid point (ix, iy, iz) sits at
        0.025 * (grid_idx_min + (ix, iy, iz))."""
        dev = self.m__device
        if vertices is None:
            self._launched("LinearBlendSknning Error: Failed to get vertices of new pose!")
            vertices = self._vertices
        v = _dev_f32(vertices, dev)
        v = (v[index] if v.dim() == 3 else v).contiguous()
        lo, num = (C.c_int32 * 3)(), (C.c_int32 * 3)()
        with torch.cuda.device(dev):
            check(lib().smplpp_sweep_grid_bounds(self.handle, _stream(dev), _ptr(v), lo, num))
            total = num[0] * num[1] * num[2]
            w = torch.empty(total, dtype=torch.float32, device=dev)
            occ = torch.empty(total, dtype=torch.uint8, device=dev)
            check(lib().smplpp_sweep_grid_winding(self.handle, _stream(dev), _ptr(v), lo, num, _ptr(w), C.c_void_p(occ.data_ptr())))
        shape = (num[0], num[1], num[2])
        return np.array(list(lo), np.int32), np.array(list(num), np.int32), w.view(shape), occ.view(shape).bool()

    def setVertPath(self, path: str):
        self.m__vertPath = path

    def out(self, index: int):
        """SMPL::out (src/SMPL.cpp:757-790): the mesh of batch element `index` as Wavefront OBJ at the vertex path."""
        self._launched("SMPL Error: Cannot export the deformed mesh!")
        if getattr(self, "m__vertPath", None) is None:
            raise SmplppError("SMPL Error: Cannot export the deformed mesh!")
        v = np.ascontiguousarray(self._vertices[index].cpu().numpy(), dtype=np.float32)
        fi = np.ascontiguousarray(self._faces_host, dtype=np.int32)
        check(lib().smplpp_write_obj(self.m__vertPath.encode(), C.c_int64(v.shape[0]), v.ctypes.data_as(capi.c_f32p),
                                     C.c_int64(fi.shape[0]), fi.ctypes.data_as(capi.c_i32p)))

    def getVertexRaw(self, idx):
        """Batch element 0 only, like the reference (LinearBlendSkinning.cpp:419-427)."""
        self._launched("LinearBlendSknning Error: Failed to get vertices of new pose!")
        return self._vertices[0, idx]

    def getRestJoint(self) -> torch.Tensor:
        self._launched("JointRegression Error: Failed to get joints!")
        return self._joints.clone()

    def getRestShape(self) -> torch.Tensor:
        """SMPL::getRestShape: T + S beta + P c (JointRegression.cpp:557); computed on demand (unfused pass)."""
        self._launched("JointRegression Error: Failed to get rest shape!")
        if self._rest is None:
            n = self._theta.shape[0]
            self._rest = torch.empty((n, self.vertex_num, 3), dtype=torch.float32, device=self.m__device)
            ws = self._workspace(n)
            with torch.cuda.device(self.m__device):
                check(lib().smplpp_forward(self.handle, _stream(self.m__device), C.c_int64(n), _ptr(self._beta),
                                           C.c_int64(self._beta_stride), _ptr(self._theta), None, None, None,
                                           _ptr(self._rest), _ptr(ws), C.c_size_t(ws.numel())))
        return self._rest.clone()

    def getTransformation(self) -> torch.Tensor:
        """WorldTransformation::getTransformation (N,24,4,4) of the last launch(want_transforms=True)."""
        if self._transforms is None:
            raise SmplppError("WorldTransformation Error: Failed to get transformations!")
        return self._transforms.clone()

    def getFaceIndex(self) -> torch.Tensor:
        if self._faces_host.shape != (FACE_INDEX_NUM, 3) and self.vertex_num == 6890:
            raise SmplppError("SMPL Error: Failed to get face indices!")  # SMPL.cpp:404
        return torch.as_tensor(self._faces_host.copy(), device=self.m__device)

    def getFaceIndexRaw(self, idx: int) -> torch.Tensor:
        return torch.as_tensor(self._faces_host[idx])

    def getAdjacentFaces(self, idx: int) -> dict:
        """SMPL::getAdjacentFaces (SMPL.cpp:619-640): {faceIdx: 1/deg}."""
        if self._adjacent is None:
            adj = [[] for _ in range(self.vertex_num)]
            for f, tri in enumerate((self._faces_host.astype(np.int64) - 1).tolist()):
                for v in tri:
                    if f not in adj[v]:
                        adj[v].append(f)
            self._adjacent = adj
        faces = self._adjacent[idx]
        return {f: np.float32(1.0) / np.float32(len(faces)) for f in faces}

    def normals(self, face_idx=None, vert_idx=None):
        """Batched SMPL::calcNormal / calcVertexNormal (SMPL.cpp:518-535) for all launched frames."""
        self._launched("LinearBlendSknning Error: Failed to get vertices of new pose!")
        n = self._vertices.shape[0]
        dev = self.m__device
        fi = torch.as_tensor(np.asarray([] if face_idx is None else face_idx, dtype=np.int64), device=dev)
        vi = torch.as_tensor(np.asarray([] if vert_idx is None else vert_idx, dtype=np.int64), device=dev)
        fn = torch.empty((n, fi.numel(), 3), dtype=torch.float32, device=dev)
        vn = torch.empty((n, vi.numel(), 3), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            check(lib().smplpp_normals(self.handle, _stream(dev), C.c_int64(n), _ptr(self._vertices),
                                       C.c_int64(fi.numel()), _ptr(fi), _ptr(fn), C.c_int64(vi.numel()), _ptr(vi),
                                       _ptr(vn)))
        return fn, vn

    def calcNormal(self, faceIdx: int) -> torch.Tensor:
        return self.normals(face_idx=[faceIdx])[0][0, 0]

    def calcVertexNormal(self, idx: int) -> torch.Tensor:
        return self.normals(vert_idx=[idx])[1][0, 0]


def load_model_file(path: str):
    """Model arrays from the reference's JSON (keys of src/SMPL.cpp:573-611) or the .npz twin written by
    scripts/preprocess.py:109-121."""
    from .synth import SmplParams
    if path.endswith(".npz"):
        z = np.load(path)
        get = lambda k: z[k]  # noqa: E731
    else:
        with open(path) as f:
            j = json.load(f)
        get = lambda k: np.asarray(j[k])  # noqa: E731
    return SmplParams(
        face_indices=np.asarray(get("face_indices"), dtype=np.int32),
        shape_blend_shapes=np.asarray(get("shape_blend_shapes"), dtype=np.float32),
        pose_blend_shapes=np.asarray(get("pose_blend_shapes"), dtype=np.float32),
        vertices_template=np.asarray(get("vertices_template"), dtype=np.float32),
        joint_regressor=np.asarray(get("joint_regressor"), dtype=np.float32),
        kinematic_tree=np.asarray(get("kinematic_tree"), dtype=np.int64),
        weights=np.asarray(get("weights"), dtype=np.float32))


def read_json_arrays(path: str, keys):
    """Numeric arrays of a parameter file (.json, or its .npz twin) through the C-ABI reader (smplpp_json_* /
    smplpp_npz_open): {key: float64 ndarray}."""
    h = C.c_void_p()
    opener = lib().smplpp_npz_open if path.endswith(".npz") else lib().smplpp_json_open
    check(opener(path.encode(), C.byref(h)))
    try:
        out = {}
        for k in keys:
            ndim, shape, data = C.c_int32(), (C.c_int64 * 8)(), C.POINTER(C.c_double)()
            check(lib().smplpp_json_array(h, k.encode(), C.byref(ndim), shape, C.byref(data)))
            shp = tuple(int(shape[i]) for i in range(ndim.value))
            n = int(np.prod(shp)) if shp else 1
            out[k] = (np.ctypeslib.as_array(data, shape=(n,)).copy() if n else np.zeros(0)).reshape(shp)
        return out
    finally:
        lib().smplpp_json_close(h)


class C3D:
    """A C3D motion-capture file as node/node.cpp:572-595, 667-691 reads it through ezc3d: labels, frame rate, frame
    count and, per frame and point, x / y / z / isEmpty (C-ABI reader smplpp_c3d_*, host only)."""

    def __init__(self, path: str):
        self._h = C.c_void_p()
        self._lib = lib()
        check(self._lib.smplpp_c3d_open(path.encode(), C.byref(self._h)))
        self.frames = int(self._lib.smplpp_c3d_frame_count(self._h))
        self.points = int(self._lib.smplpp_c3d_point_count(self._h))
        self.frame_rate = float(self._lib.smplpp_c3d_frame_rate(self._h))
        self.units = self._lib.smplpp_c3d_units(self._h).decode()
        self.labels = [self._lib.smplpp_c3d_label(self._h, C.c_int64(i)).decode() for i in range(self.points)]

    def find_label(self, name: str) -> int:
        """Index of the first label ending with `name` (node.cpp:580-594); `points` when there is none."""
        return int(self._lib.smplpp_c3d_find_label(self._h, name.encode()))

    def read(self, first: int = 0, count: Optional[int] = None):
        """(xyz (count, points, 3) float32, valid (count, points) bool); missing points are returned as zeros."""
        count = self.frames - first if count is None else count
        xyz = np.empty((count, self.points, 3), np.float32)
        valid = np.empty((count, self.points), np.uint8)
        check(self._lib.smplpp_c3d_read(self._h, C.c_int64(first), C.c_int64(count), xyz.ctypes.data_as(C.c_void_p),
                                        valid.ctypes.data_as(C.c_void_p)))
        return xyz, valid.astype(bool)

    def marker_targets(self, task_names, first: int = 0, count: Optional[int] = None):
        """Targets of the IK tasks for a block of frames: (target_pos (count, n, 3), pos_task_weight (count, n)) with
        weight 0 and a zero target for a missing marker (node.cpp:667-691)."""
        idx = [self.find_label(n) for n in task_names]
        missing = [n for n, i in zip(task_names, idx) if i >= self.points]
        if missing:
            raise SmplppError("node Error: mocap markers not found in the C3D file: %s" % ", ".join(missing))
        xyz, valid = self.read(first, count)
        return np.ascontiguousarray(xyz[:, idx]), np.ascontiguousarray(valid[:, idx].astype(np.float32))

    def close(self):
        if self._h:
            self._lib.smplpp_c3d_close(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def write_mocap_body(path: str, beta, names, face_idx, vertex_weights) -> None:
    """MocapBody.yaml of the body stage (node/node.cpp:1425-1441)."""
    beta = _np_f32(beta).reshape(-1)
    w = _np_f32(vertex_weights).reshape(-1, 3)
    fi = np.ascontiguousarray(face_idx, dtype=np.int64)
    arr = (C.c_char_p * len(names))(*[n.encode() for n in names])
    check(lib().smplpp_write_mocap_body_yaml(path.encode(), beta.ctypes.data_as(capi.c_f32p), C.c_int32(len(names)), arr,
                                             fi.ctypes.data_as(capi.c_i64p), w.ctypes.data_as(capi.c_f32p)))


def read_mocap_body(path: str):
    """(beta (10,), names, face_idx (n,), vertex_weights (n, 3)) as the motion stage loads them (node/node.cpp:509-535)."""
    h = C.c_void_p()
    check(lib().smplpp_mocap_body_open(path.encode(), C.byref(h)))
    try:
        n = int(lib().smplpp_mocap_body_task_count(h))
        beta, fi, w = np.empty(10, np.float32), np.empty(n, np.int64), np.empty((n, 3), np.float32)
        check(lib().smplpp_mocap_body_get(h, beta.ctypes.data_as(capi.c_f32p), fi.ctypes.data_as(capi.c_i64p),
                                          w.ctypes.data_as(capi.c_f32p)))
        names = [lib().smplpp_mocap_body_task_name(h, C.c_int32(i)).decode() for i in range(n)]
        return beta, names, fi, w
    finally:
        lib().smplpp_mocap_body_close(h)


def write_motion_text(path: str, theta) -> None:
    """One frame per line, 75 values (scripts/convertRosbagToText.py:13-19)."""
    th = _np_f32(theta).reshape(-1, 75)
    check(lib().smplpp_write_motion_text(path.encode(), C.c_int64(th.shape[0]), th.ctypes.data_as(capi.c_f32p)))


def read_motion_text(path: str) -> np.ndarray:
    n = C.c_int64()
    check(lib().smplpp_read_motion_text(path.encode(), C.c_int64(0), None, C.byref(n)))
    th = np.empty((n.value, 25, 3), np.float32)
    check(lib().smplpp_read_motion_text(path.encode(), n, th.ctypes.data_as(capi.c_f32p), C.byref(n)))
    return th


# ----------------------------------------------------------------------------------------------------------------
# the four pipeline modules (setter -> compute -> getter, like the reference)
# ----------------------------------------------------------------------------------------------------------------

class _Module:
    def __init__(self, device="cuda:0"):
        self.m__device = torch.device(device)

    def setDevice(self, device):
        self.m__device = torch.device(device)

    def _set(self, name, value, shape_tail, err):
        t = _dev_f32(value, self.m__device)
        if tuple(t.shape[-len(shape_tail):]) != tuple(shape_tail):
            raise SmplppError(err)
        setattr(self, name, t)


class BlendShape(_Module):
    """smplpp::BlendShape (src/BlendShape.cpp)."""

    def setBeta(self, beta):
        self._set("_beta", beta, (SHAPE_BASIS_DIM,), "BlendShape Error: Failed to set beta!")

    def setTheta(self, theta):
        self._set("_theta", theta, (JOINT_NUM, 3), "BlendShape Error: Failed to set theta!")

    def setShapeBlendBasis(self, basis):
        self._set("_shape_basis", basis, (3, SHAPE_BASIS_DIM), "BlendShape Error: Failed to set shape blend basis!")

    def setPoseBlendBasis(self, basis):
        self._set("_pose_basis", basis, (3, POSE_BASIS_DIM), "BlendShape Error: Failed to set pose blend basis!")

    def blend(self):
        _require_cuda(self.m__device)
        n, v = self._theta.shape[0], self._pose_basis.shape[0]
        dev = self.m__device
        self._shape_bs = torch.empty((n, v, 3), dtype=torch.float32, device=dev)
        self._pose_bs = torch.empty((n, v, 3), dtype=torch.float32, device=dev)
        self._pose_rot = torch.empty((n, JOINT_NUM, 3, 3), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            check(lib().smplpp_blend_shape(_stream(dev), C.c_int64(n), C.c_int64(v), _ptr(self._beta), _ptr(self._theta),
                                           _ptr(self._shape_basis), _ptr(self._pose_basis), _ptr(self._shape_bs),
                                           _ptr(self._pose_bs), _ptr(self._pose_rot)))

    def getShapeBlendShape(self):
        return self._shape_bs.clone()

    def getPoseBlendShape(self):
        return self._pose_bs.clone()

    def getPoseRotation(self):
        return self._pose_rot.clone()


class JointRegression(_Module):
    """smplpp::JointRegression (src/JointRegression.cpp)."""

    def setTemplateRestShape(self, t):
        self._set("_templ", t, (3,), "JointRegression Error: Failed to set template shape!")

    def setJointRegressor(self, r):
        t = _dev_f32(r, self.m__device)
        if t.shape[0] != JOINT_NUM:
            raise SmplppError("JointRegression Error: Failed to set joint regressor!")
        self._jreg = t

    def setShapeBlendShape(self, s):
        self._set("_shape_bs", s, (3,), "JointRegression Error: Failed to set shape blend shape!")

    def setPoseBlendShape(self, p):
        self._set("_pose_bs", p, (3,), "JointRegression Error: Failed to set pose blend shape!")

    def regress(self):
        _require_cuda(self.m__device)
        n, v = self._shape_bs.shape[0], self._templ.shape[0]
        dev = self.m__device
        self._rest = torch.empty((n, v, 3), dtype=torch.float32, device=dev)
        self._joints = torch.empty((n, JOINT_NUM, 3), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            check(lib().smplpp_joint_regression(_stream(dev), C.c_int64(n), C.c_int64(v), _ptr(self._templ),
                                                _ptr(self._jreg), _ptr(self._shape_bs), _ptr(self._pose_bs),
                                                _ptr(self._rest), _ptr(self._joints)))

    def getRestShape(self):
        return self._rest.clone()

    def getJoint(self):
        return self._joints.clone()


class WorldTransformation(_Module):
    """smplpp::WorldTransformation (src/WorldTransformation.cpp)."""

    def setKinematicTree(self, tree):
        t = torch.as_tensor(np.asarray(tree, dtype=np.int64) if not isinstance(tree, torch.Tensor) else tree)
        if tuple(t.shape) != (2, JOINT_NUM):
            raise SmplppError("WorldTransformation Error: Failed to set kinematic tree!")
        self._tree = t.to(device=self.m__device, dtype=torch.int64).contiguous()

    def setJoint(self, j):
        self._set("_joints", j, (JOINT_NUM, 3), "WorldTransformation Error: Failed to set joints!")

    def setPoseRotation(self, r):
        self._set("_rot", r, (JOINT_NUM, 3, 3), "WorldTransformation Error: Failed to set pose rotations!")

    def transform(self):
        _require_cuda(self.m__device)
        n = self._joints.shape[0]
        dev = self.m__device
        self._xf = torch.empty((n, JOINT_NUM, 4, 4), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            check(lib().smplpp_world_transformation(_stream(dev), C.c_int64(n), _ptr(self._tree), _ptr(self._joints),
                                                    _ptr(self._rot), _ptr(self._xf)))

    def getTransformation(self):
        return self._xf.clone()


class LinearBlendSkinning(_Module):
    """smplpp::LinearBlendSkinning (src/LinearBlendSkinning.cpp)."""

    _root = None

    def setWeight(self, w):
        self._set("_weights", w, (JOINT_NUM,), "LinearBlendSkinning Error: Failed to set weights!")

    def setRestShape(self, r):
        self._set("_rest", r, (3,), "LinearBlendSkinning Error: Failed to set rest shape!")

    def setTransformation(self, t):
        self._set("_xf", t, (JOINT_NUM, 4, 4), "LinearBlendSkinning Error: Failed to set transformations!")

    def setRootPos(self, p):
        self._root = _dev_f32(p, self.m__device).reshape(-1, 3).contiguous()

    def skinning(self):
        _require_cuda(self.m__device)
        n, v = self._rest.shape[0], self._weights.shape[0]
        dev = self.m__device
        self._verts = torch.empty((n, v, 3), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            check(lib().smplpp_linear_blend_skinning(_stream(dev), C.c_int64(n), C.c_int64(v), _ptr(self._weights),
                                                     _ptr(self._rest), _ptr(self._xf), _ptr(self._root),
                                                     _ptr(self._verts)))

    def getVertex(self):
        return self._verts.clone()


# ----------------------------------------------------------------------------------------------------------------
# VPoser decoder (include/smplpp/VPoser.h:33-90)
# ----------------------------------------------------------------------------------------------------------------

_VPOSER_KEYS = ("decoder_net.0.weight", "decoder_net.0.bias", "decoder_net.3.weight", "decoder_net.3.bias",
                "decoder_net.5.weight", "decoder_net.5.bias")
_VPOSER_SHAPES = ((512, LATENT_DIM), (512,), (512, 512), (512,), (126, 512), (126,))


class VPoserDecoder:
    """smplpp::VPoserDecoder (src/VPoser.cpp:143-238).  forward(latent (B,32)) -> (B,21,3) axis-angle."""

    hiddenDim_ = 512
    jointNum_ = 21

    def __init__(self, params: Optional[dict] = None, device="cuda:0"):
        self.m__device = torch.device(device)
        self._h = None
        if params is not None:
            self.loadParams(params)

    def to(self, device):
        self.m__device = torch.device(device)
        return self

    def eval(self):  # Dropout is the identity in eval mode; the kernels implement exactly that
        return self

    def loadParamsFromJson(self, jsonPath: str):
        """VPoserDecoderImpl::loadParamsFromJson (VPoser.cpp:169-238)."""
        import os
        if not os.path.exists(jsonPath):
            raise SmplppError("VPoser Error: Cannot find a JSON file!")  # VPoser.cpp:182
        with open(jsonPath) as f:
            j = json.load(f)
        self.loadParams({k: np.asarray(j[k], dtype=np.float32) for k in _VPOSER_KEYS})

    def loadParamsFromJsonNative(self, jsonPath: str):
        """The same through the C-ABI loader smplpp_vposer_load_json (what the C++ facade calls)."""
        _require_cuda(self.m__device)
        h = C.c_void_p()
        with torch.cuda.device(self.m__device):
            check(lib().smplpp_vposer_load_json(jsonPath.encode(), C.byref(h)))
        self._h = h

    def loadParams(self, params: dict):
        _require_cuda(self.m__device)
        arrs = []
        for key, shape in zip(_VPOSER_KEYS, _VPOSER_SHAPES):
            a = _np_f32(params[key])
            if a.shape != shape:
                raise SmplppError("VPoser Error: invalid dimension of %s from JSON file!" % key)  # VPoser.cpp:190
            arrs.append(a)
        desc = capi.VposerDesc(*[a.ctypes.data_as(capi.c_f32p) for a in arrs])
        h = C.c_void_p()
        with torch.cuda.device(self.m__device):
            check(lib().smplpp_vposer_create(C.byref(desc), C.byref(h)))
        self._h = h

    def __del__(self):
        try:
            if getattr(self, "_h", None) is not None and capi is not None and capi._lib is not None:
                capi._lib.smplpp_vposer_destroy(self._h)
                self._h = None
        except Exception:  # interpreter shutdown
            pass

    @property
    def handle(self):
        if self._h is None:
            raise SmplppError("VPoser Error: Cannot find a JSON file!")
        return self._h

    def forward(self, latent, jacobian: bool = False):
        z = _dev_f32(latent, self.m__device)
        if z.dim() != 2 or z.shape[1] != LATENT_DIM:
            raise SmplppError("VPoser Error: invalid latent tensor!")
        b = z.shape[0]
        aa = torch.empty((b, self.jointNum_, 3), dtype=torch.float32, device=self.m__device)
        jac = torch.empty((b, 63, LATENT_DIM), dtype=torch.float32, device=self.m__device) if jacobian else None
        with torch.cuda.device(self.m__device):
            check(lib().smplpp_vposer_decode(self.handle, _stream(self.m__device), C.c_int64(b), _ptr(z), _ptr(aa),
                                             _ptr(jac)))
        return (aa, jac) if jacobian else aa

    __call__ = forward


def convertRotMatToAxisAngle(rotMat) -> torch.Tensor:
    """smplpp::convertRotMatToAxisAngle (src/VPoser.cpp:25-120): (N,3,3) -> (N,3)."""
    dev = rotMat.device if isinstance(rotMat, torch.Tensor) and rotMat.is_cuda else torch.device("cuda:0")
    _require_cuda(dev)
    r = _dev_f32(rotMat, dev)
    n = r.shape[0]
    out = torch.empty((n, 3), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        check(lib().smplpp_rotmat_to_axis_angle(_stream(dev), C.c_int64(n), _ptr(r), _ptr(out)))
    return out


# ----------------------------------------------------------------------------------------------------------------
# IK (include/smplpp/IkTask.h:13-85 and the loop body of node/node.cpp:753-968, batched over frames)
# ----------------------------------------------------------------------------------------------------------------

def ik_options(**kw) -> capi.IkOptions:
    """smplpp_ik_options with the constants of node/node.cpp (see include/smplpp_b200.h); override by keyword."""
    o = capi.IkOptions()
    lib().smplpp_ik_options_default(C.byref(o))
    for k, v in kw.items():
        if not hasattr(o, k):
            raise SmplppError("IkTask Error: unknown IK option %s" % k)
        setattr(o, k, v)
    return o


def calcTriangleVertexWeights(pos, vertices) -> torch.Tensor:
    """smplpp::calcTriangleVertexWeights (GeometryUtils.h:42-52), batched: pos (N,3), vertices (N,3,3) -> (N,3)."""
    dev = torch.device("cuda:0")
    _require_cuda(dev)
    p = _dev_f32(pos, dev).reshape(-1, 3)
    t = _dev_f32(vertices, dev).reshape(-1, 3, 3)
    out = torch.empty_like(p)
    with torch.cuda.device(dev):
        check(lib().smplpp_triangle_vertex_weights(_stream(dev), C.c_int64(p.shape[0]), _ptr(p), _ptr(t), _ptr(out)))
    return out


class IkTaskSet:
    """n smplpp::IkTask objects (one attachment face each) handled as one batch over B frames.

    Per-task fields of IkTask.h:59-84 that the node varies per frame (targetPos_, posTaskWeight_,
    vertexWeights_) are (B,n,...) device tensors owned by the caller; the ones it sets once per mode
    (normalTaskWeight_, phiLimit_, normalOffset_) live in the options."""

    def __init__(self, smpl: SMPL, face_idx, vposer: Optional[VPoserDecoder] = None):
        self.smpl, self.vposer = smpl, vposer
        self.face_idx = np.ascontiguousarray(face_idx, dtype=np.int64)
        self.n = int(self.face_idx.shape[0])
        h = C.c_void_p()
        with torch.cuda.device(smpl.m__device):
            check(lib().smplpp_tasks_create(smpl.handle, C.c_int32(self.n), self.face_idx.ctypes.data_as(capi.c_i64p),
                                            C.byref(h)))
        self._h = h
        self._ws = None

    def __del__(self):
        try:
            if getattr(self, "_h", None) is not None and capi is not None and capi._lib is not None:
                capi._lib.smplpp_tasks_destroy(self._h)
                self._h = None
        except Exception:  # interpreter shutdown
            pass

    @property
    def vertex_count(self) -> int:
        return int(lib().smplpp_tasks_vertex_count(self._h))

    def default_vertex_weights(self, batch: int) -> torch.Tensor:
        """IkTask::vertexWeights_ default 1/3 (IkTask.h:78)."""
        return torch.full((batch, self.n, 3), 1.0 / 3.0, dtype=torch.float32, device=self.smpl.m__device)

    def positions(self, vertices: torch.Tensor, vertex_weights: torch.Tensor, normal_offset: float = 0.0,
                  want_normals: bool = False):
        """IkTask::calcActualPos (+calcActualNormal) for every frame of a (B,V,3) vertex buffer."""
        dev = self.smpl.m__device
        v = _dev_f32(vertices, dev)
        w = _dev_f32(vertex_weights, dev)
        b = v.shape[0]
        pos = torch.empty((b, self.n, 3), dtype=torch.float32, device=dev)
        nrm = torch.empty((b, self.n, 3), dtype=torch.float32, device=dev) if want_normals else None
        with torch.cuda.device(dev):
            check(lib().smplpp_task_positions(self.smpl.handle, self._h, _stream(dev), C.c_int64(b), _ptr(v), _ptr(w),
                                              C.c_float(normal_offset), _ptr(pos), _ptr(nrm)))
        return (pos, nrm) if want_normals else pos

    def _marker_args(self, beta, theta, vertex_weights):
        """shapes of the markers-only forward pass -> (B, beta stride, vertex weights stride)."""
        b = int(theta.shape[0])
        if tuple(theta.shape) != (b, JOINT_NUM + 1, 3):
            raise SmplppError("SMPL Error: Cannot launch a SMPL model!")
        nb = int(np.prod(beta.shape)) // SHAPE_BASIS_DIM if beta.shape[-1] == SHAPE_BASIS_DIM else -1
        if nb not in (1, b) or len(beta.shape) > 2:
            raise SmplppError("BlendShape Error: Failed to set beta!")
        nw = int(np.prod(vertex_weights.shape)) // (3 * self.n)
        if tuple(vertex_weights.shape[-2:]) != (self.n, 3) or nw not in (1, b) or len(vertex_weights.shape) > 3:
            raise SmplppError("IkTask Error: invalid task tensors!")
        return b, (0 if nb == 1 and b > 1 else SHAPE_BASIS_DIM), (0 if nw == 1 and b > 1 else 3 * self.n)

    def forward_positions(self, beta, theta, vertex_weights, normal_offset: float = 0.0, want_normals: bool = False):
        """Markers-only forward pass (smplpp_task_forward): IkTask::calcActualPos (+ calcActualNormal) of every task for
        every pose without building the mesh.  beta (B,10) or (10,) / (1,10) shared, theta (B,25,3), vertex_weights
        (B,n,3) or (n,3) / (1,n,3) shared.  Returns positions (B,n,3) [and normals (B,n,3)] as CUDA tensors."""
        dev = self.smpl.m__device
        be, th, w = _dev_f32(beta, dev), _dev_f32(theta, dev), _dev_f32(vertex_weights, dev)
        b, bstride, wstride = self._marker_args(be, th, w)
        pos = torch.empty((b, self.n, 3), dtype=torch.float32, device=dev)
        nrm = torch.empty((b, self.n, 3), dtype=torch.float32, device=dev) if want_normals else None
        ws = self._workspace(lib().smplpp_task_forward_workspace_bytes(self._h, b))
        with torch.cuda.device(dev):
            check(lib().smplpp_task_forward(self.smpl.handle, self._h, _stream(dev), b, _ptr(be), bstride, _ptr(th),
                                            _ptr(w), wstride, normal_offset, _ptr(pos), _ptr(nrm), _ptr(ws), ws.numel()))
        return (pos, nrm) if want_normals else pos

    def forward_positions_host(self, beta: np.ndarray, theta: np.ndarray, vertex_weights: np.ndarray,
                               normal_offset: float = 0.0, want_normals: bool = False, out_positions=None,
                               out_normals=None):
        """forward_positions with HOST arrays (smplpp_task_forward_host: chunked, uploads / compute / downloads overlapped).
        Page-locked arrays (pinned_empty) are DMA'd directly, pageable ones are staged.  Returns numpy positions (B,n,3)
        [and normals]; out_positions / out_normals receive the result when given (C-contiguous float32 (B,n,3))."""
        be, th, w = _np_f32(beta), _np_f32(theta), _np_f32(vertex_weights)
        b, bstride, wstride = self._marker_args(be, th, w)
        pos = np.empty((b, self.n, 3), np.float32) if out_positions is None else out_positions
        nrm = None
        if want_normals:
            nrm = np.empty((b, self.n, 3), np.float32) if out_normals is None else out_normals
        for a in (pos, nrm):
            if a is not None and not (isinstance(a, np.ndarray) and a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
                                      and a.shape == (b, self.n, 3)):
                raise SmplppError("IkTask Error: invalid task tensors!")

        def p(a):
            return None if a is None else a.ctypes.data_as(C.c_void_p)

        with torch.cuda.device(self.smpl.m__device):
            check(lib().smplpp_task_forward_host(self.smpl.handle, self._h, b, p(be), bstride, p(th), p(w), wstride,
                                                 normal_offset, p(pos), p(nrm)))
        return (pos, nrm) if want_normals else pos

    def assemble_theta(self, theta_state: torch.Tensor) -> torch.Tensor:
        """(B,75) -> (B,25,3) as is; (B,44) VPoser state [trans 3 | root 3 | latent 32 | hands 6] through the decoder
        (node/node.cpp:761-772)."""
        b = theta_state.shape[0]
        if theta_state.shape[1] == 75:
            return theta_state.reshape(b, 25, 3)
        if self.vposer is None:
            raise SmplppError("VPoser Error: Cannot find a JSON file!")
        body = self.vposer.forward(theta_state[:, 6:38].contiguous())
        return torch.cat([theta_state[:, 0:3].reshape(b, 1, 3), theta_state[:, 3:6].reshape(b, 1, 3), body,
                          theta_state[:, 38:41].reshape(b, 1, 3), theta_state[:, 41:44].reshape(b, 1, 3)], dim=1).contiguous()

    def reproject(self, opt: capi.IkOptions, theta_state: torch.Tensor, beta: torch.Tensor, vertex_weights: torch.Tensor,
                  face_idx: torch.Tensor, dphi: Optional[torch.Tensor] = None, want_sq_dist: bool = False):
        """The tail of an IK iteration in the reference (node/node.cpp:949-1001) for every frame, through
        smplpp_ik_reproject: on the mesh of `theta_state` / `beta` (the node uses the PRE-update state of the iteration)
        the point p = calcActualPos() + tangents * dphi of every task is projected onto the mesh and the attachment is
        re-seated IN PLACE: face_idx (B,n) int32 <- closest face, vertex_weights (B,n,3) <-
        calcTriangleVertexWeights(closest point, face).  Returns the squared distances (B,n) when asked for."""
        dev = self.smpl.m__device
        b = theta_state.shape[0]
        for name, t, dt in (("theta_state", theta_state, torch.float32), ("vertex_weights", vertex_weights, torch.float32),
                            ("face_idx", face_idx, torch.int32)):
            if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dt and t.is_contiguous()):
                raise SmplppError("IkTask Error: %s must be a contiguous CUDA tensor" % name)
        beta_t = _dev_f32(beta, dev)
        stride = 0 if beta_t.numel() == SHAPE_BASIS_DIM and b > 1 else SHAPE_BASIS_DIM
        sq = torch.empty((b, self.n), dtype=torch.float32, device=dev) if want_sq_dist else None
        need = lib().smplpp_ik_reproject_workspace_bytes(self.smpl.handle, self._h, C.c_int64(b))
        ws = self._workspace(need)
        vp = self.vposer.handle if (opt.enable_vposer and self.vposer is not None) else None
        with torch.cuda.device(dev):
            check(lib().smplpp_ik_reproject(self.smpl.handle, vp, self._h, C.byref(opt), _stream(dev), C.c_int64(b),
                                            _ptr(theta_state), _ptr(beta_t), C.c_int64(stride), _ptr(vertex_weights),
                                            _ptr(face_idx), _ptr(dphi), _ptr(sq), _ptr(ws), C.c_size_t(ws.numel())))
        return sq

    def iterate(self, opt: capi.IkOptions, theta_state: torch.Tensor, beta: torch.Tensor, vertex_weights: torch.Tensor,
                face_idx: torch.Tensor, target_pos: torch.Tensor, pos_task_weight: Optional[torch.Tensor] = None,
                outputs: bool = False):
        """One COMPLETE iteration of the reference's loop body (node/node.cpp:753-1001) for every frame: the step on
        the per-frame attachments, then the projection of the moved task points onto the pre-update mesh and the
        re-seated faces / weights.  theta_state, beta (per frame when optimize_beta), vertex_weights, face_idx in place."""
        dev = self.smpl.m__device
        b = theta_state.shape[0]
        theta_pre, beta_pre = theta_state.clone(), beta.clone()
        dphi = torch.zeros((b, self.n, 2), dtype=torch.float32, device=dev)
        r = self.step(opt, theta_state, beta, vertex_weights, target_pos, pos_task_weight=pos_task_weight, outputs=outputs,
                      face_idx=face_idx, dphi_out=dphi)
        self.reproject(opt, theta_pre, beta_pre, vertex_weights, face_idx, dphi=dphi)
        return r

    def _workspace(self, nbytes: int) -> torch.Tensor:
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = torch.empty(nbytes, dtype=torch.uint8, device=self.smpl.m__device)
        return self._ws

    def restShape(self, beta, theta, variant: int = 0):
        """Rest shape of the vertices the task set depends on (SMPL::getRestShape on those rows): returns (rest (B, nU, 3)
        CUDA tensor, vertex_ids (nU,) int32 numpy).  variant 0: tcgen05 where available, 1: FFMA kernel."""
        dev = self.smpl.m__device
        b = _dev_f32(beta, dev).reshape(-1, 10).contiguous()
        th = _dev_f32(theta, dev).reshape(-1, 75).contiguous()
        B = th.shape[0]
        nu = self.vertex_count
        rest = torch.empty((B, nu, 3), dtype=torch.float32, device=dev)
        ids = np.zeros(nu, dtype=np.int32)
        with torch.cuda.device(dev):
            check(lib().smplpp_tasks_rest_shape(self.smpl.handle, self._h, _stream(dev), C.c_int64(B), _ptr(b),
                                                C.c_int64(0 if b.shape[0] == 1 else 10), _ptr(th), _ptr(rest),
                                                ids.ctypes.data_as(capi.c_i32p), C.c_int32(variant)))
        return rest, ids

    def jacobian(self, opt: capi.IkOptions, theta_state: torch.Tensor, beta: torch.Tensor, vertex_weights: torch.Tensor,
                 target_pos: torch.Tensor, pos_task_weight: Optional[torch.Tensor] = None,
                 target_normal: Optional[torch.Tensor] = None, want_jacobian: bool = True):
        """The linearisation of the IK step alone (smplpp_ik_jacobian; the reference runs one Tensor::backward per residual
        row for this, node/node.cpp:823-873).  theta_state and beta are read only; vertex_weights receives the re-weighting
        of node.cpp:803-804.  Returns e (B,4n) and J (B,4n,dim) (None unless want_jacobian) in the layout of step()."""
        dev = self.smpl.m__device
        for name, t in (("theta_state", theta_state), ("beta", beta), ("vertex_weights", vertex_weights),
                        ("target_pos", target_pos)):
            if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
                raise SmplppError("IkTask Error: %s must be a contiguous float32 CUDA tensor" % name)
        b = theta_state.shape[0]
        theta_dim = int(lib().smplpp_ik_theta_dim(C.byref(opt)))
        if theta_state.shape != (b, theta_dim):
            raise SmplppError("IkTask Error: theta state must be (B, %d)" % theta_dim)
        if vertex_weights.shape != (b, self.n, 3) or target_pos.shape != (b, self.n, 3):
            raise SmplppError("IkTask Error: task tensors must be (B, %d, 3)" % self.n)
        stride = 0 if beta.numel() == SHAPE_BASIS_DIM and b > 1 else SHAPE_BASIS_DIM
        dim = int(lib().smplpp_ik_dim(C.byref(opt), C.c_int32(self.n)))
        e = torch.empty((b, 4 * self.n), dtype=torch.float32, device=dev)
        jac = torch.empty((b, 4 * self.n, dim), dtype=torch.float32, device=dev) if want_jacobian else None
        vp = self.vposer.handle if (opt.enable_vposer and self.vposer is not None) else None
        need = lib().smplpp_ik_workspace_bytes(self._h, C.byref(opt), C.c_int64(b))
        ws = self._workspace(need)
        with torch.cuda.device(dev):
            check(lib().smplpp_ik_jacobian(
                self.smpl.handle, vp, self._h, C.byref(opt), _stream(dev), C.c_int64(b), _ptr(theta_state), _ptr(beta),
                C.c_int64(stride), _ptr(vertex_weights), _ptr(target_pos), _ptr(target_normal), _ptr(pos_task_weight),
                _ptr(e), _ptr(jac), _ptr(ws), C.c_size_t(ws.numel())))
        return e, jac

    def step(self, opt: capi.IkOptions, theta_state: torch.Tensor, beta: torch.Tensor, vertex_weights: torch.Tensor,
             target_pos: torch.Tensor, pos_task_weight: Optional[torch.Tensor] = None,
             target_normal: Optional[torch.Tensor] = None, outputs: bool = False,
             face_idx: Optional[torch.Tensor] = None, dphi_out: Optional[torch.Tensor] = None):
        """One IK iteration for all frames (node/node.cpp:753-968 per frame).  theta_state (B,75|44), beta
        ((B,10) or (10,) shared) and vertex_weights (B,n,3) are updated IN PLACE.  Returns status (B,) int32 and,
        with outputs=True, a dict of e (B,4n), J (B,4n,dim), A (B,dim,dim), b, delta in the reference layout."""
        dev = self.smpl.m__device
        for name, t in (("theta_state", theta_state), ("beta", beta), ("vertex_weights", vertex_weights),
                        ("target_pos", target_pos)):
            if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
                raise SmplppError("IkTask Error: %s must be a contiguous float32 CUDA tensor" % name)
        b = theta_state.shape[0]
        theta_dim = int(lib().smplpp_ik_theta_dim(C.byref(opt)))
        if theta_state.shape != (b, theta_dim):
            raise SmplppError("IkTask Error: theta state must be (B, %d)" % theta_dim)
        if vertex_weights.shape != (b, self.n, 3) or target_pos.shape != (b, self.n, 3):
            raise SmplppError("IkTask Error: task tensors must be (B, %d, 3)" % self.n)
        stride = 0 if beta.numel() == SHAPE_BASIS_DIM and b > 1 else SHAPE_BASIS_DIM
        dim = int(lib().smplpp_ik_dim(C.byref(opt), C.c_int32(self.n)))
        status = torch.empty((b,), dtype=torch.int32, device=dev)
        out = None
        if outputs:
            out = dict(e=torch.empty((b, 4 * self.n), dtype=torch.float32, device=dev),
                       J=torch.empty((b, 4 * self.n, dim), dtype=torch.float32, device=dev),
                       A=torch.empty((b, dim, dim), dtype=torch.float64, device=dev),
                       b=torch.empty((b, dim), dtype=torch.float64, device=dev),
                       delta=torch.empty((b, dim), dtype=torch.float64, device=dev))
        vp = self.vposer.handle if (opt.enable_vposer and self.vposer is not None) else None
        if face_idx is not None:
            # per-frame attachments (IkTask::faceIdx_ after the projection step, node.cpp:993-1001)
            if not (face_idx.is_cuda and face_idx.dtype == torch.int32 and face_idx.is_contiguous()
                    and face_idx.shape == (b, self.n)):
                raise SmplppError("IkTask Error: face_idx must be a contiguous int32 CUDA tensor of shape (B, %d)" % self.n)
            need = lib().smplpp_ik_faces_workspace_bytes(self._h, C.byref(opt), C.c_int64(b))
            ws = self._workspace(need)
            with torch.cuda.device(dev):
                check(lib().smplpp_ik_step_faces(
                    self.smpl.handle, vp, self._h, C.byref(opt), _stream(dev), C.c_int64(b), _ptr(theta_state), _ptr(beta),
                    C.c_int64(stride), _ptr(vertex_weights), _ptr(face_idx), _ptr(target_pos), _ptr(target_normal),
                    _ptr(pos_task_weight), _ptr(status), _ptr(out["e"]) if out else None, _ptr(out["J"]) if out else None,
                    _ptr(out["A"]) if out else None, _ptr(out["b"]) if out else None, _ptr(out["delta"]) if out else None,
                    _ptr(dphi_out), _ptr(ws), C.c_size_t(ws.numel())))
            return (status, out) if outputs else status
        need = lib().smplpp_ik_workspace_bytes(self._h, C.byref(opt), C.c_int64(b))
        ws = self._workspace(need)
        with torch.cuda.device(dev):
            check(lib().smplpp_ik_step(
                self.smpl.handle, vp, self._h, C.byref(opt), _stream(dev), C.c_int64(b), _ptr(theta_state), _ptr(beta),
                C.c_int64(stride), _ptr(vertex_weights), _ptr(target_pos), _ptr(target_normal), _ptr(pos_task_weight),
                _ptr(status), _ptr(out["e"]) if out else None, _ptr(out["J"]) if out else None,
                _ptr(out["A"]) if out else None, _ptr(out["b"]) if out else None, _ptr(out["delta"]) if out else None,
                _ptr(ws), C.c_size_t(ws.numel())))
        return (status, out) if outputs else status

    def solve_host(self, opt: capi.IkOptions, iterations: int, theta_state: np.ndarray, beta: np.ndarray,
                   vertex_weights: np.ndarray, target_pos: np.ndarray, pos_task_weight: Optional[np.ndarray] = None,
                   want_residual: bool = True):
        """smplpp_ik_solve_host: `iterations` IK steps for all frames with HOST arrays (numpy, pageable or page-locked);
        theta_state (B,75|44), vertex_weights (B,n,3) (and beta with optimize_beta) are updated in place.
        Returns (status (B,) int32, residual (B,) float32 or None)."""
        b = theta_state.shape[0]
        theta_dim = int(lib().smplpp_ik_theta_dim(C.byref(opt)))
        for name, a, shape in (("theta_state", theta_state, (b, theta_dim)), ("vertex_weights", vertex_weights, (b, self.n, 3)),
                               ("target_pos", target_pos, (b, self.n, 3))):
            if not (isinstance(a, np.ndarray) and a.dtype == np.float32 and a.flags["C_CONTIGUOUS"] and a.shape == shape):
                raise SmplppError("IkTask Error: %s must be a C-contiguous float32 array of shape %s" % (name, (shape,)))
        if not (beta.dtype == np.float32 and beta.flags["C_CONTIGUOUS"]):
            raise SmplppError("BlendShape Error: Failed to set beta!")
        stride = 0 if beta.size == SHAPE_BASIS_DIM and b > 1 else SHAPE_BASIS_DIM
        status = np.empty((b,), np.int32)
        res = np.empty((b,), np.float32) if want_residual else None
        pw = None
        if pos_task_weight is not None:
            pw = np.ascontiguousarray(pos_task_weight, dtype=np.float32)
        vp = self.vposer.handle if (opt.enable_vposer and self.vposer is not None) else None

        def p(a):
            return None if a is None else a.ctypes.data_as(C.c_void_p)

        with torch.cuda.device(self.smpl.m__device):
            check(lib().smplpp_ik_solve_host(self.smpl.handle, vp, self._h, C.byref(opt), C.c_int64(b), C.c_int32(iterations),
                                             p(theta_state), p(beta), C.c_int64(stride), p(vertex_weights), p(target_pos),
                                             p(pw), p(status), p(res)))
        return status, res

    def shared_beta_step(self, opt: capi.IkOptions, theta_state: torch.Tensor, shared_beta: torch.Tensor,
                         vertex_weights: torch.Tensor, target_pos: torch.Tensor,
                         pos_task_weight: Optional[torch.Tensor] = None, process_group=None, return_reduced=False):
        """MoSh++ shape stage over the frames of ALL ranks: per-frame Schur complement onto the 10 shared betas,
        ONE all-reduce of 111 doubles (only collective of the path), identical 10-dim box QP on every rank,
        back-substitution.  theta_state (B,75|44) and shared_beta (10,) are updated in place."""
        from . import parallel
        dev = self.smpl.m__device
        b = theta_state.shape[0]
        status = torch.empty((b,), dtype=torch.int32, device=dev)
        reduced = torch.empty((111,), dtype=torch.float64, device=dev)
        need = lib().smplpp_ik_shared_beta_workspace_bytes(self._h, C.byref(opt), C.c_int64(b))
        ws = self._workspace(need)
        vp = self.vposer.handle if (opt.enable_vposer and self.vposer is not None) else None
        with torch.cuda.device(dev):
            check(lib().smplpp_ik_shared_beta_reduce(
                self.smpl.handle, vp, self._h, C.byref(opt), _stream(dev), C.c_int64(b), _ptr(theta_state),
                _ptr(shared_beta), _ptr(vertex_weights), _ptr(target_pos), _ptr(pos_task_weight), _ptr(status),
                _ptr(reduced), _ptr(ws), C.c_size_t(ws.numel())))
            parallel.all_reduce_shared_beta(reduced, process_group)  # NCCL over NVLink on the B200 box; 888 bytes
            check(lib().smplpp_ik_shared_beta_apply(self._h, C.byref(opt), _stream(dev), C.c_int64(b), _ptr(theta_state),
                                                    _ptr(shared_beta), _ptr(status), _ptr(reduced), _ptr(ws),
                                                    C.c_size_t(ws.numel())))
        return (status, reduced) if return_reduced else status


class IkTask:
    """smplpp::IkTask for ONE face on batch element 0 of the last SMPL::launch — the reference's object-level
    interface (IkTask.h:20-84), kept for callers that drive single tasks; batched work uses IkTaskSet."""

    def __init__(self, smpl: SMPL, faceIdx: int, targetPos=None, targetNormal=None):
        self.smpl_, self.faceIdx_ = smpl, int(faceIdx)
        dev = smpl.m__device
        self.posTaskWeight_, self.normalTaskWeight_, self.phiLimit_, self.normalOffset_ = 1.0, 1.0, 0.04, 0.0
        self.targetPos_ = torch.zeros(3, device=dev) if targetPos is None else _dev_f32(targetPos, dev)
        self.targetNormal_ = (torch.tensor([0.0, 0.0, 1.0], device=dev) if targetNormal is None
                              else _dev_f32(targetNormal, dev))
        self.vertexWeights_ = torch.full((3,), 1.0 / 3.0, device=dev)
        self.tangents_ = torch.zeros(3, 2, device=dev)
        self.phi_ = torch.zeros(2, device=dev)
        self._set = IkTaskSet(smpl, [self.faceIdx_])

    def _face_vertices(self):
        ids = torch.as_tensor(self.smpl_._faces_host[self.faceIdx_].astype(np.int64) - 1, device=self.smpl_.m__device)
        return self.smpl_.getVertexRaw(ids)

    def calcTangents(self):
        fv = self._face_vertices()
        t1 = fv[1] - fv[0]
        normal = torch.linalg.cross(t1, fv[2] - fv[0])
        t2 = torch.linalg.cross(normal, t1)
        self.tangents_ = torch.stack([torch.nn.functional.normalize(t1, dim=-1),
                                      torch.nn.functional.normalize(t2, dim=-1)], 1)

    def calcVertexWeights(self, actualPos):
        pos = _dev_f32(actualPos, self.smpl_.m__device) + self.tangents_ @ self.phi_
        self.vertexWeights_ = calcTriangleVertexWeights(pos.view(1, 3), self._face_vertices().view(1, 3, 3))[0]

    def calcActualPos(self) -> torch.Tensor:
        v = self.smpl_._vertices[:1]
        return self._set.positions(v, self.vertexWeights_.view(1, 1, 3), float(self.normalOffset_))[0, 0]

    def calcActualNormal(self) -> torch.Tensor:
        v = self.smpl_._vertices[:1]
        return self._set.positions(v, self.vertexWeights_.view(1, 1, 3), 0.0, want_normals=True)[1][0, 0]


def solve_mocap_motion(smpl: SMPL, vposer: Optional[VPoserDecoder], c3d_path: str, body_yaml_path: str, opt: capi.IkOptions,
                       initial_state, warmup_iterations: int = 31, iterations: int = 1, reproject: bool = False,
                       first_frame: int = 0, frame_count: int = 0, motion_text_path: Optional[str] = None) -> dict:
    """smplpp_solve_mocap_motion: the motion stage of the mocap mode (node/node.cpp:509-535, 571-595, 667-691, 785,
    1369-1407) as one call - C3D file + MocapBody.yaml in, theta (frames,75), status, residual and a summary out."""
    c3d = C3D(c3d_path)
    frames = c3d.frames - first_frame if frame_count <= 0 else min(frame_count, c3d.frames - first_frame)
    theta = np.empty((frames, 75), np.float32)
    status = np.empty((frames,), np.int32)
    res = np.empty((frames,), np.float32)
    summ = capi.MocapSummary()
    init = np.ascontiguousarray(initial_state, dtype=np.float32).reshape(-1)
    vp = vposer.handle if (opt.enable_vposer and vposer is not None) else None
    with torch.cuda.device(smpl.m__device):
        check(lib().smplpp_solve_mocap_motion(
            smpl.handle, vp, c3d_path.encode(), body_yaml_path.encode(), C.byref(opt), C.c_int32(warmup_iterations),
            C.c_int32(iterations), C.c_int32(int(reproject)), init.ctypes.data_as(C.c_void_p), C.c_int64(first_frame),
            C.c_int64(frame_count), theta.ctypes.data_as(C.c_void_p), status.ctypes.data_as(C.c_void_p),
            res.ctypes.data_as(C.c_void_p), motion_text_path.encode() if motion_text_path else None, C.byref(summ)))
    return dict(theta=theta.reshape(frames, 25, 3), status=status, residual=res,
                summary={k: getattr(summ, k) for k, _ in capi.MocapSummary._fields_})
