"""bindings/kiss_icp_pybind: the reference's `kiss_icp.pybind.kiss_icp_pybind` module (kiss_icp_pybind.cpp:44-144)
re-bound over the C-ABI. CPU tests: the surface (names, keyword arguments, exceptions) and — where the reference
checkout is available — that the reference's own Python layer imports and binds on top of it. The GPU test compares
every bound call with the ctypes mirror."""
import inspect
import os
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


@pytest.fixture(scope="module")
def mod():
    pytest.importorskip("pybind11")
    from bindings import build
    return build.load()


def _sig(doc):
    return doc.split("\n")[0]


def test_names_and_keyword_arguments_are_the_reference_s(mod):
    names = {n for n in dir(mod) if n.startswith("_") and not n.startswith("__")}
    assert names == {"_Vector3dVector", "_VoxelHashMap", "_Preprocessor", "_Registration", "_AdaptiveThreshold",
                     "_voxel_down_sample", "_correct_kitti_scan", "_kitti_seq_error", "_absolute_trajectory_error"}
    kw = [  # kiss_icp_pybind.cpp:56-57,77-78,91-92,104-105,111-112,120,123,138,141-143
        (mod._VoxelHashMap.__init__, ["voxel_size", "max_distance", "max_points_per_voxel"]),
        (mod._Preprocessor.__init__, ["max_range", "min_range", "deskew", "max_num_threads"]),
        (mod._Preprocessor._preprocess, ["points", "timestamps", "relative_motion"]),
        (mod._Registration.__init__, ["max_num_iterations", "convergence_criterion", "max_num_threads"]),
        (mod._Registration._align_points_to_map, ["points", "voxel_map", "initial_guess", "max_correspondance_distance", "kernel"]),
        (mod._AdaptiveThreshold.__init__, ["initial_threshold", "min_motion_th", "max_range"]),
        (mod._AdaptiveThreshold._update_model_deviation, ["model_deviation"]),
        (mod._voxel_down_sample, ["frame", "voxel_size"]),
        (mod._correct_kitti_scan, ["frame"]),
        (mod._kitti_seq_error, ["gt_poses", "results_poses"]),
        (mod._absolute_trajectory_error, ["gt_poses", "results_poses"]),
    ]
    for fn, names in kw:
        sig = _sig(fn.__doc__)
        pos = [sig.index(n + ":") for n in names]
        assert pos == sorted(pos), sig
    for meth in ("_clear", "_empty", "_update", "_add_points", "_remove_far_away_points", "_point_cloud"):
        assert hasattr(mod._VoxelHashMap, meth)


def test_vector3dvector_is_a_zero_copy_pass_through(mod):
    a = np.arange(12, dtype=np.float64).reshape(4, 3)
    v = mod._Vector3dVector(a)
    assert len(v) == 4 and np.shares_memory(np.asarray(v), a)
    assert np.array_equal(np.asarray(mod._Vector3dVector(a.astype(np.float32))), a)  # forcecast like the reference
    with pytest.raises(RuntimeError):  # pybind11::cast_error, stl_vector_eigen.h:71-73
        mod._Vector3dVector(np.zeros((4, 2)))


def test_host_only_parts_and_errors_without_a_gpu(mod):
    import kiss_icp_b200  # noqa: F401  (the metrics live in the Python package)
    th = mod._AdaptiveThreshold(initial_threshold=2.0, min_motion_th=0.1, max_range=100.0)
    assert th._compute_threshold() == 2.0
    T = np.eye(4)
    T[0, 3] = 1.0
    th._update_model_deviation(model_deviation=T)
    assert np.isclose(th._compute_threshold(), np.sqrt((4.0 + 1.0) / 2.0))
    with pytest.raises(ValueError):  # Sophus would abort on a non-SE(3) matrix
        th._update_model_deviation(np.zeros((4, 4)))
    g = np.tile(np.eye(4), (300, 1, 1))
    g[:, 0, 3] = np.arange(300)
    assert max(mod._kitti_seq_error(g, g)) < 1e-6
    assert mod._absolute_trajectory_error(g, g)[1] < 1e-6
    from kiss_icp_b200 import _native as N
    if N.lib().kb_device_count() < 1:
        with pytest.raises(RuntimeError, match="no CUDA device"):
            mod._VoxelHashMap(1.0, 100.0, 20)
        with pytest.raises(RuntimeError, match="no CUDA device"):
            mod._voxel_down_sample(np.zeros((3, 3)), 0.5)


# the python/ directory of an upstream kiss-icp checkout; its sources are not part of this repository
REF = os.environ.get("KISS_ICP_UPSTREAM_PYTHON", "")
HAVE_REF = bool(REF) and os.path.isdir(os.path.join(REF, "kiss_icp"))


def test_reference_python_layer_imports_on_top_of_it(mod):
    """python/kiss_icp/*.py, unmodified, with `kiss_icp.pybind.kiss_icp_pybind` supplied by this module: the calls the
    upstream layer made into it (import, default config, threshold estimate and update, KITTI metrics, KissICP's
    constructor), recorded by tests/golden/make_pybind_calls.py, are replayed; each must be accepted and give the
    recorded result, and without a device the pipeline's constructor must fail as it did then"""
    import json
    from kiss_icp_b200 import _native as N
    golden = os.path.join(ROOT, "tests", "golden", "pybind_calls_v1")
    log = json.load(open(golden + ".json"))
    arrays = np.load(golden + ".npz")
    objs = {}

    def dec(v):
        if isinstance(v, dict):
            return objs[v["obj"]] if "obj" in v else arrays[v["array"]]
        return [dec(x) for x in v] if isinstance(v, list) else v

    assert log["meta"]["first_threshold"] == log["meta"]["initial_threshold"]
    no_device = N.lib().kb_device_count() < 1
    for c in log["calls"]:
        fn = getattr(mod, c["func"]) if "func" in c else getattr(objs[c["obj"]], c["method"])
        args, kwargs = [dec(a) for a in c["args"]], {k: dec(v) for k, v in c["kwargs"].items()}
        if "raised" in c:
            assert c["raised"]["type"] == "RuntimeError" and "no CUDA device" in c["raised"]["message"]
            if no_device:
                with pytest.raises(RuntimeError, match="no CUDA device"):
                    fn(*args, **kwargs)
            continue
        r = fn(*args, **kwargs)
        want = c["result"]
        if isinstance(want, dict) and "obj" in want:
            objs[want["obj"]] = r
        elif want is None:
            assert r is None
        else:
            assert np.allclose(np.asarray(r, dtype=np.float64), np.asarray(dec(want), dtype=np.float64), rtol=1e-12, atol=1e-9), (c, r)


@pytest.mark.gpu
def test_every_bound_call_equals_the_ctypes_mirror(mod):
    import kiss_icp_b200 as K
    from kiss_icp_b200 import synthetic
    L = synthetic.small_shape(seed=4, beams=32, cols=512, stamps="column")
    p0, t0 = L.scan(0)
    p1, t1 = L.scan(1)
    assert np.array_equal(mod._voxel_down_sample(mod._Vector3dVector(p0), 0.5), K.voxel_down_sample(p0, 0.5))
    assert np.array_equal(mod._correct_kitti_scan(p0), K.correct_kitti_scan(p0))
    T = np.eye(4)
    T[0, 3] = 0.4
    pre_a = mod._Preprocessor(100.0, 0.0, True, 0)._preprocess(p1, t1, T)
    pre_b = K.Preprocessor(100.0, 0.0, True, 0).preprocess(p1, t1, T)
    assert np.array_equal(pre_a, pre_b)
    with pytest.raises(IndexError):  # std::out_of_range through pybind11
        mod._Preprocessor(100.0, 0.0, True, 0)._preprocess(p1, t1[:5], T)
    ma, mb = mod._VoxelHashMap(1.0, 100.0, 20), K.VoxelHashMap(1.0, 100.0, 20)
    assert ma._empty()
    ds = K.voxel_down_sample(p0, 0.5)
    ma._update(ds, np.eye(4))
    mb.update(ds, np.eye(4))
    ma._add_points(ds[:100] + 0.05)
    mb.add_points(ds[:100] + 0.05)
    ma._remove_far_away_points(np.array([30.0, 0.0, 0.0]))
    mb.remove_far_away_points(np.array([30.0, 0.0, 0.0]))
    assert not ma._empty() and np.array_equal(ma._point_cloud(), mb.point_cloud())
    src = K.voxel_down_sample(K.voxel_down_sample(p1, 0.5), 1.5)
    Ta = mod._Registration(500, 1e-4, 0)._align_points_to_map(src, ma, T, 3.0, 1.0)
    Tb = K.Registration(500, 1e-4, 0).align_points_to_map(src, mb, T, 3.0, 1.0)
    assert np.array_equal(Ta, Tb)
    ma._update(ds, np.array([1.0, 0.0, 0.0]))  # the (points, origin) overload, positional
    mb.update(ds, np.array([1.0, 0.0, 0.0]))
    assert np.array_equal(ma._point_cloud(), mb.point_cloud())
    ma._update(points=ds[:50] + 0.3, origin=np.zeros(3))  # ... and by keyword, like the reference's two py::arg lists
    ma._update(points=ds[:50] + 0.6, pose=np.eye(4))
    mb.update(ds[:50] + 0.3, np.zeros(3))
    mb.update(ds[:50] + 0.6, np.eye(4))
    assert np.array_equal(ma._point_cloud(), mb.point_cloud())
    with pytest.raises(TypeError):  # neither overload takes a (2, 2) second argument
        ma._update(ds, np.zeros((2, 2)))
    ma._clear()
    assert ma._empty()


class _ReferenceKissICP:
    """python/kiss_icp/kiss_icp.py:33-80 (class KissICP) restated on the bound module; where KISS_ICP_UPSTREAM_PYTHON
    points at an upstream checkout the test below uses the reference's own class instead"""

    def __init__(self, mod, max_range=100.0, voxel_size=1.0):
        self.m = mod
        self.voxel_size = voxel_size
        self.last_pose, self.last_delta = np.eye(4), np.eye(4)
        self.threshold = mod._AdaptiveThreshold(2.0, 0.1, max_range)
        self.pre = mod._Preprocessor(max_range, 0.0, True, 0)
        self.reg = mod._Registration(500, 1e-4, 0)
        self.map = mod._VoxelHashMap(voxel_size, max_range, 20)

    def register_frame(self, frame, timestamps):
        m = self.m
        frame = np.asarray(self.pre._preprocess(m._Vector3dVector(frame), timestamps, self.last_delta))
        ds = np.asarray(m._voxel_down_sample(m._Vector3dVector(frame), self.voxel_size * 0.5))
        source = np.asarray(m._voxel_down_sample(m._Vector3dVector(ds), self.voxel_size * 1.5))
        sigma = self.threshold._compute_threshold()
        guess = self.last_pose @ self.last_delta
        new_pose = self.reg._align_points_to_map(points=m._Vector3dVector(source), voxel_map=self.map, initial_guess=guess,
                                                 max_correspondance_distance=3 * sigma, kernel=sigma)
        self.threshold._update_model_deviation(np.linalg.inv(guess) @ new_pose)
        self.map._update(m._Vector3dVector(ds), new_pose)
        self.last_delta = np.linalg.inv(self.last_pose) @ new_pose
        self.last_pose = new_pose
        return frame, source


@pytest.mark.gpu
def test_reference_python_register_frame_loop_on_the_gpu(mod, O):
    """the reference's Python RegisterFrame loop (python/kiss_icp/kiss_icp.py:43-75) over this backend's pybind module
    against the oracle: 10 scans, pose per scan within 1e-9. Uses the reference's own unmodified class where the
    checkout exists, its restatement above otherwise."""
    import time
    from kiss_icp_b200 import synthetic
    L = synthetic.small_shape(seed=11, beams=32, cols=512, stamps="column")
    icp = None
    saved = {k: v for k, v in sys.modules.items() if k == "kiss_icp" or k.startswith("kiss_icp.")}
    use_ref = HAVE_REF
    try:
        if use_ref:
            sys.path.insert(0, REF)
            import kiss_icp
            pkg = types.ModuleType("kiss_icp.pybind")
            pkg.__path__ = []
            pkg.kiss_icp_pybind = mod
            sys.modules["kiss_icp.pybind"] = pkg
            sys.modules["kiss_icp.pybind.kiss_icp_pybind"] = mod
            kiss_icp.pybind = pkg
            from kiss_icp.config import load_config
            from kiss_icp.kiss_icp import KissICP
            icp = KissICP(load_config(None))
        else:
            icp = _ReferenceKissICP(mod)
        o = O.KissICP()
        t0 = time.perf_counter()
        for k in range(10):
            p, t = L.scan(k)
            icp.register_frame(p, t)
            o.register_frame(p, t, want_clouds=False)
            assert np.abs(np.asarray(icp.last_pose) - o.pose).max() < 1e-9, k
        print("reference Python loop on the pybind module: %.0f scans/s (incl. the oracle's time)" % (10 / (time.perf_counter() - t0)))
    finally:
        if use_ref:
            sys.path.remove(REF)
            for k in [k for k in sys.modules if k == "kiss_icp" or k.startswith("kiss_icp.")]:
                del sys.modules[k]
            sys.modules.update(saved)
