"""The float64 mode of the oracle's IK iteration (ik_iteration(dtype=torch.float64)) against the compiled reference's
golden IK rows (tests/golden/ref_ik.npz) in all five modes.  The float64 oracle is the reference of
tests/test_ik_linearisation_gpu.py on task sets where the float32 autograd of the reference is ill-conditioned; this
pins it to the compiled reference where both are well conditioned, and checks that the process-global torch default
dtype it switches is restored."""
import numpy as np
import pytest
import torch

from oracle import smpl_oracle as so

F64 = torch.float64
MODES = dict(motion=dict(nw=0.0, pl=0.0, no=0.015, ob=False, qp=True),
             body=dict(nw=0.0, pl=0.04, no=0.015, ob=True, qp=True),
             interactive=dict(nw=1.0, pl=0.0, no=0.0, ob=False, qp=True),
             llt=dict(nw=0.0, pl=0.0, no=0.0, ob=False, qp=False))


@pytest.fixture(scope="module")
def model64(oracle_model):
    return oracle_model.to(F64)


def _tasks(g, mode):
    n = len(g["face_idx"])
    if mode == "vposer":
        kw, tgt, pw = MODES["motion"], g["target_pos"], np.ones(n)
    else:
        kw, tgt, pw = MODES[mode], g[mode + "_target"], g.get(mode + "_pos_task_weight", np.ones(n))
    return [so.IkTask(int(g["face_idx"][i]), target_pos=torch.as_tensor(tgt[i]), pos_task_weight=float(pw[i]),
                      normal_task_weight=kw["nw"], phi_limit=kw["pl"], normal_offset=kw["no"],
                      vertex_weights=torch.as_tensor(g["vertex_weights_in"][i])) for i in range(n)]


@pytest.mark.parametrize("mode", ["motion", "body", "interactive", "llt", "vposer"])
def test_f64_oracle_vs_reference_golden(model64, oracle_vposer, golden_ik, mode):
    g = golden_ik
    tasks = _tasks(g, mode)
    if mode == "vposer":
        r = so.ik_iteration(model64, tasks, g["vposer_theta_in"], g["beta_in"], vposer=oracle_vposer.to(F64), dtype=F64)
        J, e, delta = g["vposer_J"], g["vposer_e"], g["vposer_delta"]
    else:
        kw = MODES[mode]
        r = so.ik_iteration(model64, tasks, g["theta_in"], g["beta_in"], optimize_beta=kw["ob"], enable_qp=kw["qp"],
                            dtype=F64)
        J, e, delta = g[mode + "_J"], g[mode + "_e"], g[mode + "_delta"]
        # calcTriangleVertexWeights of a float32 point: 1.4e-5 in the interactive mode
        assert np.abs(r.vertex_weights - g[mode + "_vertex_weights_out"]).max() < 1e-4
    assert torch.get_default_dtype() == torch.float32
    assert r.theta_state.dtype == np.float64 and all(t.vertex_weights.dtype == F64 for t in tasks)
    # the golden rows are the compiled reference's float32 arithmetic: what separates the two is float32 rounding
    # (measured 3e-7 .. 4.3e-5 of max |J|, the largest on the normal rows of the interactive mode)
    assert np.abs(r.J - J).max() / np.abs(J).max() <= 1e-4
    assert np.abs(r.e - e).max() < 2e-5
    assert np.abs(r.delta - delta).max() < 1e-5


def test_f64_oracle_restores_default_dtype(oracle_model, golden_ik):
    """The default dtype is process-global and the rest of the suite runs float32: it is restored after a normal call
    and after one that raises inside the iteration; a float32 model in a float64 call is refused before anything runs."""
    g = golden_ik
    model64 = oracle_model.to(F64)
    assert model64.templ.dtype == F64 and oracle_model.templ.dtype == torch.float32
    assert model64.face_indices is oracle_model.face_indices
    so.ik_iteration(model64, _tasks(g, "llt")[:4], g["theta_in"], g["beta_in"], enable_qp=False, dtype=F64)
    assert torch.get_default_dtype() == torch.float32
    with pytest.raises(AssertionError):  # a theta state of the wrong length fails inside the body of the call
        so.ik_iteration(model64, _tasks(g, "llt")[:4], np.zeros(44), g["beta_in"], dtype=F64)
    assert torch.get_default_dtype() == torch.float32
    with pytest.raises(TypeError):
        so.ik_iteration(oracle_model, _tasks(g, "llt")[:4], g["theta_in"], g["beta_in"], dtype=F64)
    assert torch.get_default_dtype() == torch.float32


def test_f32_oracle_unchanged_by_f64_calls(oracle_model, golden_ik):
    """The float32 iteration is bitwise the same before and after a float64 call (no state leaks between them)."""
    g = golden_ik

    def run():
        return so.ik_iteration(oracle_model, _tasks(g, "motion")[:6], g["theta_in"], g["beta_in"])
    a = run()
    so.ik_iteration(oracle_model.to(F64), _tasks(g, "motion")[:6], g["theta_in"], g["beta_in"], dtype=F64)
    b = run()
    assert a.theta_state.dtype == np.float32
    assert np.array_equal(a.J, b.J) and np.array_equal(a.e, b.e) and np.array_equal(a.delta, b.delta)
