"""Host-side data formats behind the C ABI (SURVEY.md 8f ranks 2-3): the JSON parameter reader against Python's json
on the files the synthetic model writer produces (same keys as scripts/preprocess.py / src/SMPL.cpp:572-612), and the
C3D reader against fixtures written by tests/c3d_writer.py.  No GPU: nothing here creates a model."""
import json

import numpy as np
import pytest

from c3d_writer import write_c3d


@pytest.fixture(scope="module")
def api():
    from smplpp_b200 import api as a
    return a


def test_json_reader_matches_python_json(tmp_path, api):
    from smplpp_b200 import synth
    path = str(tmp_path / "vposer.json")
    params = synth.make_vposer_params(1)
    synth.vposer_to_json(params, path)
    keys = ["decoder_net.%d.%s" % (l, k) for l in (0, 3, 5) for k in ("weight", "bias")]
    got = api.read_json_arrays(path, keys)
    with open(path) as f:
        ref = json.load(f)
    for k in keys:
        want = np.asarray(ref[k], dtype=np.float64)
        assert got[k].shape == want.shape
        assert np.array_equal(got[k], want)           # strtod and Python's float() agree bit for bit


def test_json_reader_model_keys_and_edge_cases(tmp_path, api):
    from smplpp_b200 import capi
    doc = {"face_indices": [[1, 2, 3], [2, 3, 4]], "kinematic_tree": [[4294967295, 0, 0], [0, 1, 2]],
           "name": 'smpl "quoted" model', "nested": {"a": [1, 2], "b": None}, "flag": True, "scalar": -1.5e-3,
           "deep": [[[1.0, 2.0], [3.0, 4.0]], [[5.0, 6.0], [7.0, 8.0]]], "ragged": [[1, 2], [3]], "empty": []}
    path = str(tmp_path / "m.json")
    with open(path, "w") as f:
        json.dump(doc, f, indent=1)
    got = api.read_json_arrays(path, ["face_indices", "kinematic_tree", "deep", "scalar", "empty"])
    assert got["face_indices"].shape == (2, 3) and got["face_indices"].astype(np.int32).tolist() == doc["face_indices"]
    assert got["kinematic_tree"].astype(np.int64)[0, 0] == 4294967295   # the root's parent survives (SMPL.cpp:605)
    assert got["deep"].shape == (2, 2, 2) and got["deep"].reshape(-1).tolist() == [1, 2, 3, 4, 5, 6, 7, 8]
    assert got["scalar"].shape == () and float(got["scalar"]) == -1.5e-3
    assert got["empty"].shape == (0,)
    for bad in ("ragged", "name", "missing"):
        with pytest.raises(capi.SmplppError, match="no rectangular numeric array"):
            api.read_json_arrays(path, [bad])
    with pytest.raises(capi.SmplppError, match="Cannot find a JSON file"):
        api.read_json_arrays(str(tmp_path / "absent.json"), ["x"])
    with open(str(tmp_path / "broken.json"), "w") as f:
        f.write('{"a": [1, 2, }')
    with pytest.raises(capi.SmplppError, match="Cannot parse the JSON file"):
        api.read_json_arrays(str(tmp_path / "broken.json"), ["a"])


def test_loaders_report_the_reference_messages_without_a_device(tmp_path):
    """smplpp_model_load_json / smplpp_vposer_load_json fail with the reference's texts BEFORE touching CUDA."""
    import ctypes as C
    from smplpp_b200 import capi
    lib = capi.lib()
    h = C.c_void_p()
    assert lib.smplpp_model_load_json(str(tmp_path / "none.json").encode(), C.byref(h)) != 0
    assert lib.smplpp_last_error().decode().startswith("SMPL Error: Cannot initialize a SMPL model!")    # SMPL.cpp:616
    assert lib.smplpp_vposer_load_json(str(tmp_path / "none.json").encode(), C.byref(h)) != 0
    assert lib.smplpp_last_error().decode().startswith("VPoser Error: Cannot find a JSON file!")         # VPoser.cpp:183
    V = 4
    doc = {"face_indices": [[1, 2, 3]], "shape_blend_shapes": np.zeros((V, 3, 9)).tolist(),
           "pose_blend_shapes": np.zeros((V, 3, 207)).tolist(), "vertices_template": np.zeros((V, 3)).tolist(),
           "joint_regressor": np.zeros((24, V)).tolist(), "kinematic_tree": np.zeros((2, 24)).tolist(),
           "weights": np.zeros((V, 24)).tolist()}
    p = str(tmp_path / "bad_shape.json")
    with open(p, "w") as f:
        json.dump(doc, f)
    assert lib.smplpp_model_load_json(p.encode(), C.byref(h)) != 0
    assert "Shape parameter dimensions are invalid: 9 != 10" in lib.smplpp_last_error().decode()        # SMPL.cpp:581
    doc["shape_blend_shapes"] = np.zeros((V, 3, 10)).tolist()
    doc["pose_blend_shapes"] = np.zeros((V, 3, 200)).tolist()
    with open(p, "w") as f:
        json.dump(doc, f)
    assert lib.smplpp_model_load_json(p.encode(), C.byref(h)) != 0
    assert "Pose parameter dimensions are invalid: 200 != 207" in lib.smplpp_last_error().decode()      # SMPL.cpp:588
    vp = {"decoder_net.0.weight": np.zeros((512, 31)).tolist()}
    p2 = str(tmp_path / "bad_vposer.json")
    with open(p2, "w") as f:
        json.dump(vp, f)
    assert lib.smplpp_vposer_load_json(p2.encode(), C.byref(h)) != 0
    assert "invalid dimension of decoder_net.0.weight from JSON file!" in lib.smplpp_last_error().decode()  # VPoser.cpp:191


@pytest.mark.parametrize("as_int16", [False, True])
def test_c3d_round_trip(tmp_path, api, as_int16):
    rng = np.random.default_rng(4)
    frames, points = 37, 49
    xyz = rng.uniform(-2, 2, (frames, points, 3)).astype(np.float32)
    valid = rng.random((frames, points)) > 0.1
    labels = ["Skeleton20220624:M%02d" % i for i in range(41)] + ["Unlabeled_11%02d" % i for i in range(8)]
    path = str(tmp_path / "t.c3d")
    write_c3d(path, xyz, valid, labels, rate=120.0, as_int16=as_int16, scale=0.0005, analog_per_frame=3 if as_int16 else 0)
    c = api.C3D(path)
    assert (c.frames, c.points, c.frame_rate, c.units) == (frames, points, 120.0, "m")
    assert c.labels == labels
    got, ok = c.read()
    assert np.array_equal(ok, valid)
    tol = 0.0005 / 2 + 1e-7 if as_int16 else 0.0
    assert np.abs(got[valid] - xyz[valid]).max() <= tol
    assert np.all(got[~valid] == 0.0)                       # node.cpp:682-683: missing marker -> zero target
    part, okp = c.read(5, 7)
    assert np.array_equal(part, got[5:12]) and np.array_equal(okp, ok[5:12])
    # suffix match of node.cpp:580-594, first hit wins, "not found" = point count
    assert c.find_label("M07") == 7 and c.find_label("Skeleton20220624:M07") == 7
    assert c.find_label("nope") == points
    tgt, w = c.marker_targets(["M00", "M40"], 0, 4)
    assert tgt.shape == (4, 2, 3) and np.array_equal(w, valid[:4][:, [0, 40]].astype(np.float32))
    from smplpp_b200 import capi
    with pytest.raises(capi.SmplppError, match="frame range outside the C3D file"):
        c.read(30, 10)
    with pytest.raises(capi.SmplppError, match="Cannot open the C3D file"):
        api.C3D(str(tmp_path / "absent.c3d"))
    with open(str(tmp_path / "junk.c3d"), "wb") as f:
        f.write(bytes(600))
    with pytest.raises(capi.SmplppError, match="not a C3D file"):
        api.C3D(str(tmp_path / "junk.c3d"))


def test_mocap_body_yaml_and_motion_text_round_trip(tmp_path, api):
    """Result files of the mocap modes: MocapBody.yaml (node.cpp:1425-1441 writes it, :509-535 loads it back) and the
    75-values-per-line motion dump (scripts/convertRosbagToText.py).  Exact float32 round trip; the YAML is also valid
    for a generic YAML parser."""
    import yaml
    from smplpp_b200 import capi
    rng = np.random.default_rng(2)
    beta = rng.normal(size=10).astype(np.float32)
    names = ["HeadTop", "WaistLFront", "RToeOut"]
    face_idx = np.array([7324, 2162, 13775], dtype=np.int64)
    w = rng.dirichlet(np.ones(3), size=3).astype(np.float32)
    path = str(tmp_path / "MocapBody.yaml")
    api.write_mocap_body(path, beta, names, face_idx, w)
    b2, n2, f2, w2 = api.read_mocap_body(path)
    assert np.array_equal(b2, beta) and n2 == names and np.array_equal(f2, face_idx) and np.array_equal(w2, w)
    with open(path) as f:
        doc = yaml.safe_load(f)
    assert np.array_equal(np.float32(doc["beta"]), beta) and doc["ikTaskList"][1]["faceIdx"] == 2162
    assert doc["ikTaskList"][2]["name"] == "RToeOut" and np.array_equal(np.float32(doc["ikTaskList"][0]["vertexWeights"]), w[0])
    with open(str(tmp_path / "short.yaml"), "w") as f:
        f.write("beta: [1, 2, 3]\nikTaskList:\n")
    with pytest.raises(capi.SmplppError, match="Size of beta must be 10 but 3"):   # node.cpp:511-515
        api.read_mocap_body(str(tmp_path / "short.yaml"))
    theta = rng.normal(size=(17, 25, 3)).astype(np.float32)
    tpath = str(tmp_path / "motion.txt")
    api.write_motion_text(tpath, theta)
    assert np.array_equal(api.read_motion_text(tpath), theta)
    with open(tpath) as f:
        first = f.readline().split()
    assert len(first) == 75 and np.float32(first[0]) == theta[0, 0, 0]
    with open(str(tmp_path / "bad.txt"), "w") as f:
        f.write("1 2 3\n")
    with pytest.raises(capi.SmplppError, match="does not hold 75 values"):
        api.read_motion_text(str(tmp_path / "bad.txt"))


def test_json_reader_random_documents(tmp_path, api):
    """Property test (hypothesis): rectangular float / int arrays of random rank, shape and formatting come back with
    the same shape and bit-identical values as Python's json module reads them."""
    from hypothesis import given, settings, strategies as st

    shapes = st.lists(st.integers(1, 4), min_size=1, max_size=4)
    counter = [0]

    @settings(max_examples=40, deadline=None)
    @given(shape=shapes, seed=st.integers(0, 2 ** 31 - 1), indent=st.sampled_from([None, 0, 2]), ints=st.booleans())
    def check(shape, seed, indent, ints):
        rng = np.random.default_rng(seed)
        arr = rng.integers(-2 ** 40, 2 ** 40, size=shape) if ints else rng.normal(size=shape) * 10.0 ** rng.integers(-30, 30)
        counter[0] += 1
        path = str(tmp_path / ("h%d.json" % counter[0]))
        with open(path, "w") as f:
            json.dump({"skip": {"x": [1, [2]]}, "a": arr.tolist(), "tail": "s"}, f, indent=indent)
        got = api.read_json_arrays(path, ["a"])["a"]
        with open(path) as f:
            want = np.asarray(json.load(f)["a"], dtype=np.float64)
        assert got.shape == want.shape and np.array_equal(got, want)

    check()


def test_obj_export_text(tmp_path):
    """SMPL::out (src/SMPL.cpp:757-790): "v x y z" with ostream's default float format (= %g) and 1-based "f a b c"."""
    import ctypes as C
    from smplpp_b200 import capi
    rng = np.random.default_rng(6)
    v = (rng.normal(size=(7, 3)) * np.array([1.0, 1e-5, 1e5])).astype(np.float32)
    f = np.array([[1, 2, 3], [5, 6, 7]], dtype=np.int32)
    path = str(tmp_path / "mesh.obj")
    capi.check(capi.lib().smplpp_write_obj(path.encode(), C.c_int64(7), v.ctypes.data_as(capi.c_f32p), C.c_int64(2),
                                           f.ctypes.data_as(capi.c_i32p)))
    lines = open(path).read().splitlines()
    assert len(lines) == 9
    for i in range(7):
        assert lines[i] == "v %g %g %g" % tuple(float(x) for x in v[i])
    assert lines[7] == "f 1 2 3" and lines[8] == "f 5 6 7"
    assert capi.lib().smplpp_write_obj(path.encode(), C.c_int64(0), None, C.c_int64(0), None) != 0
    assert "Cannot export the deformed mesh!" in capi.lib().smplpp_last_error().decode()


def test_npz_reader_matches_numpy(tmp_path, api):
    """The .npz twin (np.savez, scripts/preprocess.py:98-117): every array and dtype numpy stores for a model comes back
    with the same shape and values; compressed archives and Fortran order are refused with a clear message."""
    from smplpp_b200 import capi
    rng = np.random.default_rng(12)
    arrays = {
        "vertices_template": rng.normal(size=(11, 3)).astype(np.float32),
        "face_indices": rng.integers(1, 12, size=(7, 3)).astype(np.int32),
        "kinematic_tree": np.array([[4294967295, 0, 1], [0, 1, 2]], dtype=np.int64),
        "weights": rng.random((11, 24)),                                   # float64
        "pose_blend_shapes": rng.normal(size=(11, 3, 207)).astype(np.float32),
        "u4": np.arange(5, dtype=np.uint32), "scalar": np.float32(2.5),
    }
    path = str(tmp_path / "model.npz")
    np.savez(path, **arrays)
    got = api.read_json_arrays(path, list(arrays))
    for k, v in arrays.items():
        assert got[k].shape == np.shape(v), k
        assert np.array_equal(got[k], np.asarray(v, dtype=np.float64)), k
    cpath = str(tmp_path / "compressed.npz")
    np.savez_compressed(cpath, a=np.zeros((4, 4), np.float32))
    with pytest.raises(capi.SmplppError, match="compressed .npz members are not supported"):
        api.read_json_arrays(cpath, ["a"])
    fpath = str(tmp_path / "fortran.npz")
    np.savez(fpath, a=np.asfortranarray(rng.normal(size=(3, 4))))
    with pytest.raises(capi.SmplppError, match="Fortran-ordered"):
        api.read_json_arrays(fpath, ["a"])
    with pytest.raises(capi.SmplppError, match="Cannot find the .npz file"):
        api.read_json_arrays(str(tmp_path / "absent.npz"), ["a"])
    with open(str(tmp_path / "junk.npz"), "wb") as f:
        f.write(bytes(100))
    with pytest.raises(capi.SmplppError, match="not a zip archive"):
        api.read_json_arrays(str(tmp_path / "junk.npz"), ["a"])
