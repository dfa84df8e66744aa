"""CPU suite: the C-ABI library builds for sm_100a, loads, and exports every symbol of include/smplpp_b200.h
(no compute calls without a GPU), and the host-side mirror fails loudly without a device."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from smplpp_b200 import build, capi
    build.build()
    return capi.lib()


def test_header_symbols_are_exported(lib):
    from smplpp_b200 import capi
    header = open(os.path.join(ROOT, "include", "smplpp_b200.h")).read()
    declared = set(re.findall(r"\b(smplpp_[a-z0-9_]+)\s*\(", header))
    declared -= {"smplpp_model_desc", "smplpp_vposer_desc", "smplpp_ik_options"}
    assert declared, "no declarations found"
    assert declared == set(capi.EXPORTS)
    for name in sorted(declared):
        assert hasattr(lib, name), name


def test_struct_layouts_match_header():
    import ctypes as C
    from smplpp_b200 import capi
    assert C.sizeof(capi.IkOptions) == 6 * 4 + 9 * 4 + 3 * 4
    assert C.sizeof(capi.ModelDesc) == 9 * 8
    assert C.sizeof(capi.VposerDesc) == 6 * 8


def test_set_forward_variant_codes(lib):
    """smplpp_set_forward_variant accepts exactly the codes include/smplpp_b200.h documents; any other code is
    refused with the library's error text instead of being mapped to some other implementation."""
    documented = [0, 1, 3, 6, 200, 201, 202, 300, 301, 400, 401, 402, 410, 411, 420, 421, 422]
    try:
        for code in documented:
            assert lib.smplpp_set_forward_variant(code) == 0, code
        for code in (2, 4, 5, 7, 100, 101, 203):
            assert lib.smplpp_set_forward_variant(code) == -1, code
            assert "unknown forward variant" in lib.smplpp_last_error().decode(), code
    finally:
        for code in (0, 202, 300, 400, 410, 420):  # the defaults
            assert lib.smplpp_set_forward_variant(code) == 0


def test_no_cpu_fallback(lib, params):
    import torch
    from smplpp_b200 import api
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    assert lib.smplpp_device_count() == 0
    with pytest.raises(api.SmplppError, match="no CPU fallback"):
        api.SMPL(params, device="cuda:0")
    with pytest.raises(api.SmplppError):
        api.BlendShape().blend()


def test_ik_options_defaults(lib):
    """The constants of node/node.cpp that the step uses."""
    from smplpp_b200 import api
    o = api.ik_options()
    assert (o.enable_qp, o.update_state, o.skip_if_too_few) == (1, 1, 1)
    assert np.isclose(o.normal_offset, 0.015) and o.normal_task_weight == 0.0 and o.phi_limit == 0.0
    assert np.isclose(o.delta_theta_reg, 1e-3) and np.isclose(o.delta_phi_reg, 1e-1) and np.isclose(o.delta_beta_reg, 1e-3)
    assert np.isclose(o.delta_beta_limit, 0.5) and np.isclose(o.vposer_latent_reg, 1e-5) and np.isclose(o.vposer_hand_reg, 1e3)
    assert lib.smplpp_ik_theta_dim(__import__("ctypes").byref(o)) == 75
    assert lib.smplpp_ik_dim(__import__("ctypes").byref(o), 41) == 75 + 82
    assert lib.smplpp_ik_dim(__import__("ctypes").byref(api.ik_options(enable_vposer=1, optimize_beta=1)), 41) == 44 + 82 + 10


def test_synthetic_model_shapes(params, vposer_params, marker_tasks):
    """Official shapes: 6890 verts, 13776 faces (1-based), 24 joints, 10 betas, 207 pose dims, 32-d latent."""
    assert params.face_indices.shape == (13776, 3) and params.face_indices.min() == 1 and params.face_indices.max() == 6890
    assert params.shape_blend_shapes.shape == (6890, 3, 10) and params.pose_blend_shapes.shape == (6890, 3, 207)
    assert params.joint_regressor.shape == (24, 6890) and params.weights.shape == (6890, 24)
    assert params.kinematic_tree.shape == (2, 24) and params.kinematic_tree[0, 0] == 4294967295
    assert (np.count_nonzero(params.weights, axis=1) <= 4).all()
    assert np.allclose(params.weights.sum(1), 1.0, atol=1e-6)
    assert vposer_params["decoder_net.5.weight"].shape == (126, 512)
    names, face_idx, vw = marker_tasks
    assert len(names) == 41 and names == sorted(names) and len(set(face_idx.tolist())) == 41
    assert np.allclose(vw.sum(1), 1.0, atol=1e-6)


def test_cpp_facade_builds_and_fails_loudly_without_gpu(lib):
    """include/smplpp_b200/smplpp.hpp (the reference's class names over the C ABI) compiles with plain g++ and, on a
    machine without a device, stops with the library's no-CPU-fallback error instead of computing anything."""
    import subprocess
    import torch
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "tests", "cpp")])
    exe = os.path.join(ROOT, "tests", "cpp", "facade_smoke")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    if torch.cuda.is_available():
        assert r.returncode == 0 and "facade smoke: OK" in r.stdout, r.stdout + r.stderr
    else:
        assert r.returncode == 3 and "no CPU fallback" in r.stdout, r.stdout + r.stderr
