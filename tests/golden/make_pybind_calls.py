"""Generates tests/golden/pybind_calls_v1.json + .npz — the calls the upstream kiss-icp Python layer makes into
`kiss_icp.pybind.kiss_icp_pybind` when that module is bindings/kiss_icp_pybind (this project's re-binding).

The upstream package (python/kiss_icp/*.py, unmodified) is imported on top of the built module wrapped in a recorder,
then it reads its default config, estimates a threshold, updates it, computes the KITTI metrics of a trajectory and
constructs its KissICP pipeline. Every call it makes into the module is logged with its arguments, its result or the
exception it raised; tests/test_pybind_module.py replays the log, so the check needs no upstream checkout.
Run on a machine without a CUDA device (the pipeline's constructor must raise there, as it did when recorded):
    python tests/golden/make_pybind_calls.py <upstream kiss-icp checkout>/python
"""
import json
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
OUT = os.path.join(ROOT, "tests", "golden", "pybind_calls_v1")
sys.path.insert(0, ROOT)


class Recorder:
    def __init__(self, mod):
        self.mod, self.calls, self.arrays, self.n_obj = mod, [], {}, 0

    def enc(self, v):
        if isinstance(v, Obj):
            return {"obj": v._id}
        if isinstance(v, np.ndarray):
            key = f"a{len(self.arrays)}"
            self.arrays[key] = v
            return {"array": key}
        if isinstance(v, (tuple, list)):
            return [self.enc(x) for x in v]
        if isinstance(v, (bool, int, float, str, type(None))):
            return v
        raise TypeError(f"cannot record {type(v)}")

    def call(self, target, fn, args, kwargs):
        entry = {**target, "args": [self.enc(a) for a in args], "kwargs": {k: self.enc(v) for k, v in kwargs.items()}}
        self.calls.append(entry)
        real = lambda v: v._real if isinstance(v, Obj) else v
        try:
            r = fn(*[real(a) for a in args], **{k: real(v) for k, v in kwargs.items()})
        except Exception as e:
            entry["raised"] = {"type": type(e).__name__, "message": str(e)}
            raise
        if isinstance(r, (np.ndarray, tuple, list, bool, int, float, str, type(None))):
            entry["result"] = self.enc(r)
            return r
        self.n_obj += 1
        entry["result"] = {"obj": self.n_obj}
        return Obj(self, self.n_obj, r)


class Obj:
    def __init__(self, rec, id_, real):
        self._rec, self._id, self._real = rec, id_, real

    def __getattr__(self, name):
        fn = getattr(self._real, name)
        return lambda *a, **k: self._rec.call({"obj": self._id, "method": name}, fn, a, k)

    def __array__(self, dtype=None, copy=None):
        return np.asarray(self._real, dtype=dtype)

    def __len__(self):
        return len(self._real)


def main(upstream_python):
    from bindings import build
    from kiss_icp_b200 import _native as N
    if N.lib().kb_device_count() > 0:
        raise SystemExit("record on a machine without a CUDA device")
    mod = build.load()
    rec = Recorder(mod)
    proxy = types.ModuleType("kiss_icp.pybind.kiss_icp_pybind")
    for name in dir(mod):
        if name.startswith("_") and not name.startswith("__"):
            setattr(proxy, name, (lambda n: lambda *a, **k: rec.call({"func": n}, getattr(mod, n), a, k))(name))
    sys.path.insert(0, upstream_python)
    import kiss_icp
    pkg = types.ModuleType("kiss_icp.pybind")
    pkg.__path__ = []
    pkg.kiss_icp_pybind = proxy
    sys.modules["kiss_icp.pybind"] = pkg
    sys.modules["kiss_icp.pybind.kiss_icp_pybind"] = proxy
    kiss_icp.pybind = pkg
    import kiss_icp.mapping, kiss_icp.metrics, kiss_icp.preprocess, kiss_icp.registration, kiss_icp.voxelization  # noqa: E401,F401
    from kiss_icp.config import load_config
    from kiss_icp.kiss_icp import KissICP
    from kiss_icp.threshold import get_threshold_estimator
    cfg = load_config(None)
    est = get_threshold_estimator(cfg)
    first_threshold = est.get_threshold()
    T = np.eye(4)
    T[0, 3] = 1.0
    est.update_model_deviation(T)
    est.get_threshold()
    g = np.tile(np.eye(4), (300, 1, 1))
    g[:, 0, 3] = np.arange(300)
    kiss_icp.metrics.sequence_error(g, g)
    kiss_icp.metrics.absolute_trajectory_error(g, g)
    try:
        KissICP(cfg)
        raise SystemExit("KissICP(config) did not raise without a CUDA device")
    except RuntimeError:
        pass
    meta = {"initial_threshold": cfg.adaptive_threshold.initial_threshold, "first_threshold": first_threshold}
    with open(OUT + ".json", "w") as f:
        json.dump({"meta": meta, "calls": rec.calls}, f, indent=1)
    np.savez_compressed(OUT + ".npz", **rec.arrays)
    print(f"{len(rec.calls)} calls, {len(rec.arrays)} arrays -> {OUT}.json/.npz")


if __name__ == "__main__":
    main(sys.argv[1])
