"""The fused tcgen05 forward kernel (variant 6, skin_tc3.cu) skins a 128-vertex tile over one 16-joint window when the
tile's joints fit one, and over both windows otherwise.  These models exercise each case against the FFMA kernel
(variant 1) on every frame and vertex, and against the oracle."""
import numpy as np
import pytest

from conftest import TOL_VERTEX_M

pytestmark = pytest.mark.gpu

f32 = np.float32


def _model(V, tile_joints, seed):
    """Synthetic model whose tile t draws the (up to 4) non-zero weights of each vertex from tile_joints[t]."""
    from smplpp_b200 import synth
    rng = np.random.default_rng(seed)
    tree = np.stack([synth.PARENTS.copy(), np.arange(24)])
    tree[0, 0] = 4294967295
    w = np.zeros((V, 24), f32)
    for v in range(V):
        joints = np.asarray(tile_joints[v // 128])
        k = min(4, len(joints))
        w[v, rng.choice(joints, size=k, replace=False)] = rng.uniform(0.05, 1.0, size=k)
    faces = np.stack([rng.permutation(V)[:3] for _ in range(2 * V)]).astype(np.int32) + 1
    return synth.SmplParams(
        face_indices=faces, shape_blend_shapes=rng.normal(size=(V, 3, 10)).astype(f32) * 0.01,
        pose_blend_shapes=rng.normal(size=(V, 3, 207)).astype(f32) * 0.002,
        vertices_template=rng.normal(size=(V, 3)).astype(f32) * 0.3,
        joint_regressor=rng.dirichlet(np.ones(V), size=24).astype(f32), kinematic_tree=tree, weights=w)


# Window 0 = joints 0-15 and window 1 = joints 8-23 are the choice for these tiles: tiles over 0-15 fit only window 0,
# tiles over 8-23 only window 1, tiles over all 24 joints (and the last, partial tile) need both.  V = 7 * 128 + 50.
_W0, _W1, _ALL = range(0, 16), range(8, 24), range(24)
_MIXED = dict(V=946, tile_joints=[_W0, _W1, _ALL, _W0, _W0, _W1, _ALL, _ALL], seed=21)


def _dense_model(V=300, seed=22):
    """Every vertex influenced by all 24 joints: every tile needs both windows."""
    p = _model(V, [_ALL] * ((V + 127) // 128), seed)
    p.weights[:] = np.random.default_rng(seed).uniform(0.1, 1.0, size=p.weights.shape).astype(f32)
    return p


def _check(params, batch, seed):
    from oracle import smpl_oracle as so
    from smplpp_b200 import api, capi, synth
    m = api.SMPL(params)
    beta, theta = synth.make_forward_inputs(batch, seed)
    out = {}
    for var in (1, 6):
        capi.check(capi.lib().smplpp_set_forward_variant(var))
        try:
            m.launch(beta, theta)
            out[var] = m.getVertex().cpu().numpy()
        finally:
            capi.check(capi.lib().smplpp_set_forward_variant(0))
    assert np.isfinite(out[6]).all()
    assert np.abs(out[6] - out[1]).max() < 1e-6
    v_o, _, _, _ = so.forward_numpy(so.SmplModel.from_params(params), beta, theta)
    assert np.abs(out[6] - v_o).max() <= TOL_VERTEX_M


@pytest.mark.parametrize("batch", [1, 95, 97, 193, 4096 + 37])
def test_mixed_window_modes(batch):
    """Window-0, window-1 and both-window tiles in one model; at B = 4133 the CTA ranges cross tiles of different
    modes, so the transform ring wraps with 12- and 24-entry items."""
    _check(_model(**_MIXED), batch, 40 + batch)


@pytest.mark.parametrize("batch", [1, 97, 4096 + 37])
def test_dense_weights_every_tile_both_windows(batch):
    """Dense skinning rows (24 non-zeros, sums != 1) on V >= 128, where the tcgen05 kernel runs."""
    _check(_dense_model(), batch, 60 + batch)


def test_synthetic_model_bench_size(smpl_gpu):
    """The benchmark's model and batch (every tile fits one window) against the FFMA kernel."""
    from smplpp_b200 import capi, synth
    beta, theta = synth.make_forward_inputs(4096, 88)
    out = {}
    for var in (1, 6):
        capi.check(capi.lib().smplpp_set_forward_variant(var))
        try:
            smpl_gpu.launch(beta, theta)
            out[var] = smpl_gpu.getVertex()
        finally:
            capi.check(capi.lib().smplpp_set_forward_variant(0))
    assert bool(out[6].isfinite().all())
    assert float((out[6] - out[1]).abs().max()) < 1e-6
