"""Parity of the CUDA path (through the C-ABI) against the oracle, on the same seeded inputs,
against the committed golden vectors, and at BASELINE sizes through size-independent
properties. Bar: bit-exact for integer / index / ordering work and for FP64 stages that involve
no transcendental and no reordered sum; 1e-4 m / 1e-4 rad (BASELINE.json north_star) for poses,
with the much tighter values actually expected written beside each check."""
import numpy as np
import pytest

from conftest import canon_map, pose_error

pytestmark = pytest.mark.gpu
rng = np.random.default_rng(3)
DBL_MAX = np.finfo(float).max


# --------------------------------------------------------------------------- VoxelDownsample
@pytest.mark.parametrize("n,vs,scale", [(0, 1.0, 1), (1, 1.0, 1), (2, 0.5, 1), (3, 1.0, 0.01), (1000, 0.5, 10),
                                        (65536, 0.5, 60), (20000, 1.5, 80), (5000, 0.3, 3), (131072, 0.15, 40)])
def test_voxel_down_sample_bit_exact_and_ordered(K, O, n, vs, scale):
    pts = rng.normal(size=(n, 3)) * scale
    if n > 10:
        pts[:5] = np.round(pts[:5])
        pts[5:8] = pts[2:5]
    a, b = K.voxel_down_sample(pts, vs), O.voxel_down_sample(pts, vs)
    assert a.shape == b.shape and np.array_equal(a, b)


def test_voxel_down_sample_golden(K, golden):
    assert np.array_equal(K.voxel_down_sample(golden["ds_in"], 0.5), golden["ds_out_05"])
    assert np.array_equal(K.voxel_down_sample(golden["ds_out_05"], 1.5), golden["ds_out_15"])
    assert np.array_equal(K.voxel_down_sample(golden["ds_in"], 0.3), golden["ds_out_03"])


def test_voxel_down_sample_long_probe_runs(K, O):
    # many voxels on a line -> the reference hash clusters; exercises long robin-hood runs + wrap
    x = np.arange(4000) * 0.999 + 0.3
    pts = np.stack([x, np.zeros_like(x), np.zeros_like(x)], 1)
    pts = np.concatenate([pts, pts[::-1] + [0.0, 1.0, 0.0], pts[::7]])
    assert np.array_equal(K.voxel_down_sample(pts, 1.0), O.voxel_down_sample(pts, 1.0))
    # idempotence at full size: a downsampled cloud has one point per voxel already
    big = rng.normal(size=(131072, 3)) * 50
    once = K.voxel_down_sample(big, 1.0)
    twice = K.voxel_down_sample(once, 1.0)
    assert len(once) == len(twice) and np.array_equal(np.sort(once, 0), np.sort(twice, 0))


# --------------------------------------------------------------------------- Preprocessor
def test_preprocess_no_deskew_bit_exact(K, O):
    pts = rng.normal(size=(70000, 3)) * 40
    pts[:3] = [[0, 0, 0], [100.0, 0, 0], [0, 60, 80]]  # range 0, == max, == max
    for mx, mn, deskew, ts in [(100.0, 0.0, True, np.empty(0)), (30.0, 5.0, False, np.linspace(0, 1, 70000)),
                               (100.0, 0.0, False, np.empty(0))]:
        a = K.Preprocessor(mx, mn, deskew, 0).preprocess(pts, ts, np.eye(4))
        b = O.preprocess(pts, ts, np.eye(4), mx, mn, deskew)
        assert np.array_equal(a, b)


def test_preprocess_deskew_close(K, O):
    pts = rng.normal(size=(50000, 3)) * 30
    ts = rng.random(50000) + 5.0
    T = O.se3_exp([1.2, 0.05, -0.02, 0.004, -0.003, 0.04])
    a = K.Preprocessor(100.0, 0.5, True, 0).preprocess(pts, ts, T)
    b = O.preprocess(pts, ts, T, 100.0, 0.5, True)
    assert a.shape == b.shape
    assert np.abs(a - b).max() < 1e-11  # device sin/cos differ from glibc in the last ulps


def test_preprocess_errors(K):
    P = K.Preprocessor(100.0, 0.0, True, 0)
    with pytest.raises(IndexError):  # std::out_of_range from timestamps.at(idx), Preprocessing.cpp:76-77
        P.preprocess(np.ones((10, 3)), np.array([0.0, 1.0]), np.eye(4))
    with pytest.raises(ValueError):  # Sophus would abort on a non-SE(3) matrix
        P.preprocess(np.ones((10, 3)), np.empty(0), np.diag([2.0, 1, 1, 1]))
    with pytest.raises(RuntimeError):
        P.preprocess(np.ones((10, 2)), np.empty(0), np.eye(4))
    assert P.preprocess(np.empty((0, 3)), np.empty(0), np.eye(4)).shape == (0, 3)


# --------------------------------------------------------------------------- VoxelHashMap
def build_pair(K, O, lidar, n_scans, vs=1.0, cap=20, max_d=100.0):
    g, o = K.VoxelHashMap(vs, max_d, cap), O.VoxelHashMap(vs, max_d, cap)
    T0 = lidar.pose(0)
    for k in range(n_scans):
        p, _ = lidar.scan(k)
        ds = O.voxel_down_sample(p, vs * 0.5)
        Tk = np.linalg.inv(T0) @ lidar.pose(k)
        g.update(ds, Tk)
        o.update(ds, Tk)
    return g, o


def assert_maps_equal(g, o):
    gv, gc, gp = g.dump()
    ov, oc, op = canon_map(*o.dump())
    assert np.array_equal(gv, ov) and np.array_equal(gc, oc) and np.array_equal(gp, op)
    assert g.num_points() == o.num_points() and g.num_voxels() == o.num_voxels()


@pytest.fixture(scope="module")
def lidar():
    from kiss_icp_b200 import synthetic
    return synthetic.small_shape(seed=1, beams=32, cols=512)


def test_map_update_add_remove_bit_exact(K, O, lidar):
    g, o = build_pair(K, O, lidar, 5)
    assert_maps_equal(g, o)
    for origin in ([30.0, 0, 0], [-50.0, 20.0, 0.0]):
        g.remove_far_away_points(origin)
        o.remove_far_away_points(origin)
        assert_maps_equal(g, o)
    raw, _ = lidar.scan(6)  # raw scan: hundreds of candidates per voxel, order-dependent accept rule
    g.add_points(raw)
    o.add_points(raw)
    assert_maps_equal(g, o)
    g.update(raw[::3], np.array([1.0, 2.0, 0.5]))  # Update(points, origin) overload
    o.update(raw[::3], np.array([1.0, 2.0, 0.5]))
    assert_maps_equal(g, o)
    assert sorted(map(tuple, g.point_cloud())) == sorted(map(tuple, o.point_cloud()))
    g.clear()
    assert g.empty() and g.num_points() == 0 and g.point_cloud().shape == (0, 3)


@pytest.mark.parametrize("vs,cap", [(0.3, 20), (1.0, 1), (2.0, 37), (0.5, 3)])
def test_map_other_voxel_sizes_and_capacities(K, O, vs, cap):
    pts = rng.normal(size=(30000, 3)) * 6
    g, o = K.VoxelHashMap(vs, 15.0, cap), O.VoxelHashMap(vs, 15.0, cap)
    for chunk in np.array_split(pts, 3):
        g.add_points(chunk)
        o.add_points(chunk)
    assert_maps_equal(g, o)
    g.remove_far_away_points([1.0, 1.0, 1.0])
    o.remove_far_away_points([1.0, 1.0, 1.0])
    assert_maps_equal(g, o)


def test_map_growth_and_tombstone_rehash(K, O):
    # many insert/evict rounds force table growth and the tombstone-dropping rebuild
    g, o = K.VoxelHashMap(1.0, 12.0, 8), O.VoxelHashMap(1.0, 12.0, 8)
    for r in range(25):
        c = np.array([r * 3.0, 0.0, 0.0])
        pts = rng.normal(size=(6000, 3)) * 5 + c
        g.update(pts, c)
        o.update(pts, c)
    assert_maps_equal(g, o)
    big = rng.normal(size=(600000, 3)) * 40  # > one internal chunk, forces growth
    g.add_points(big)
    o.add_points(big)
    assert_maps_equal(g, o)


def test_closest_neighbors_bit_exact(K, O, lidar):
    for cap in (20, 32, 33, 37, 64):  # max_points_per_voxel <= 32: flat gather, > 32: voxel-by-voxel walk
        g, o = build_pair(K, O, lidar, 5, cap=cap)
        p3, _ = lidar.scan(3)
        q = O.se3_act(np.linalg.inv(lidar.pose(0)) @ lidar.pose(3), p3) + rng.normal(size=p3.shape) * 0.2
        q = np.concatenate([q, [[1e4, 1e4, 1e4]]])
        ap, ad = g.closest_neighbors(q)
        bp, bd = o.closest_neighbors(q)
        assert np.array_equal(ap, bp) and np.array_equal(ad, bd), cap
        assert ad[-1] == DBL_MAX and np.array_equal(ap[-1], [0, 0, 0]), cap  # VoxelHashMap.cpp:51-52


def test_closest_neighbors_golden_and_ties(K, golden):
    g = K.VoxelHashMap(1.0, 100.0, 20)
    g.add_points(golden["ds_in"])
    p, d = g.closest_neighbors(golden["nn_q"])
    assert np.array_equal(p, golden["nn_p"]) and np.array_equal(d, golden["nn_d"])
    # exact ties: two points equidistant from the query in different voxels -> the voxel that comes
    # first in the reference's voxel_shifts order wins (VoxelHashMap.cpp:35-41,63)
    t = K.VoxelHashMap(1.0, 100.0, 20)
    t.add_points(np.array([[1.25, 0.5, 0.5], [-0.25, 0.5, 0.5], [0.5, 1.25, 0.5]]))
    p, d = t.closest_neighbors(np.array([[0.5, 0.5, 0.5]]))
    assert d[0] == 0.75 and np.array_equal(p[0], [1.25, 0.5, 0.5])  # shift (1,0,0) precedes (-1,0,0), (0,1,0)
    # near tie: |a - q|^2 = 0.25 + 2^-54 > |b - q|^2 = 0.25, but both roots round to 0.5 and the reference keeps the
    # first of equal roots, a (voxel (0,0,0) comes first); a minimum on squared distances would answer b. The oracle's
    # answer is checked in test_oracle_core.py::test_closest_neighbor_near_tie_is_decided_on_rounded_roots.
    a, b = [0.5, 0.5 + 2.0**-27, 0.0], [1.0, 0.5, 0.5]
    n = K.VoxelHashMap(1.0, 100.0, 20)
    n.add_points(np.array([b, a]))
    p, d = n.closest_neighbors(np.array([[0.5, 0.5, 0.5]]))
    assert d[0] == 0.5 and np.array_equal(p[0], a)


def test_closest_neighbors_full_size_properties(K):
    # 1M-point map, 262144 queries (config-5 scale): every stored point is its own nearest
    # neighbour at distance 0, and results are independent of query batching
    pts = rng.uniform(-60, 60, size=(1_000_000, 3))
    pts[:, 2] *= 0.05
    g = K.VoxelHashMap(1.0, 1e9, 20)
    g.add_points(pts)
    stored = g.point_cloud()
    sel = stored[rng.integers(0, len(stored), 262144)]
    p, d = g.closest_neighbors(sel)
    assert np.array_equal(p, sel) and not d.any()
    q = sel + rng.normal(size=sel.shape) * 0.3
    p1, d1 = g.closest_neighbors(q)
    perm = rng.permutation(len(q))
    p2, d2 = g.closest_neighbors(q[perm])
    assert np.array_equal(p1[perm], p2) and np.array_equal(d1[perm], d2)
    hit = d1 < DBL_MAX
    assert hit.mean() > 0.9 and np.allclose(np.linalg.norm(p1[hit] - q[hit], axis=1), d1[hit], rtol=1e-15)


# --------------------------------------------------------------------------- Registration
def test_build_system_close(K, O, lidar, golden):
    g, o = build_pair(K, O, lidar, 5)
    src = O.voxel_down_sample(O.voxel_down_sample(lidar.scan(4)[0], 0.5), 1.5)
    srcm = O.se3_act(np.linalg.inv(lidar.pose(0)) @ lidar.pose(4), src)
    reg = K.Registration(500, 1e-4, 0)
    A, b, n1 = reg.build_system(srcm, g, 3.0, 1.0)
    A2, b2, n2 = O.build_system(o, srcm, 3.0, 1.0, nthreads=1)
    assert n1 == n2 and n1 > 100
    assert np.abs(A - A2).max() <= 1e-12 * np.abs(A2).max() and np.abs(b - b2).max() <= 1e-11 * np.abs(A2).max()
    gm = K.VoxelHashMap(1.0, 100.0, 20)
    gm.add_points(golden["ds_in"])
    A, b, n = reg.build_system(golden["nn_q"][:-1], gm, 1.5, 0.5)
    assert n == int(golden["sys_nc"]) and np.allclose(A, golden["sys_JTJ"], rtol=1e-12) and np.allclose(b, golden["sys_JTr"], rtol=1e-11, atol=1e-12)


def test_align_points_to_map_matches_oracle(K, O, lidar):
    for cap in (20, 37):  # 37 > 32 points per voxel: whole-grid loop, voxel-by-voxel walk
        g, o = build_pair(K, O, lidar, 5, cap=cap)
        src = O.voxel_down_sample(O.voxel_down_sample(lidar.scan(5)[0], 0.5), 1.5)
        T5 = np.linalg.inv(lidar.pose(0)) @ lidar.pose(5)
        reg = K.Registration(500, 1e-4, 0)
        for tangent in ([0.3, -0.2, 0.05, 0.01, -0.01, 0.02], [0.0] * 6, [-0.5, 0.4, 0.0, 0.0, 0.0, -0.03]):
            guess = T5 @ O.se3_exp(tangent)
            Pg = reg.align_points_to_map(src, g, guess, 3.0, 1.0)
            Po, it = O.align_points_to_map(o, src, guess, 3.0, 1.0)
            dt, dr = pose_error(Pg, Po)
            assert dt < 1e-4 and dr < 1e-4, (cap, dt, dr)      # BASELINE bar
            assert dt < 1e-9 and dr < 1e-9, (cap, dt, dr)      # expected: summation-order noise only
            assert reg.last_iterations == it, (cap, reg.last_iterations, it)
        # max_num_iterations is honoured
        reg1 = K.Registration(1, 1e-4, 0)
        P1 = reg1.align_points_to_map(src, g, T5 @ O.se3_exp([0.3, 0, 0, 0, 0, 0]), 3.0, 1.0)
        Po1, it1 = O.align_points_to_map(o, src, T5 @ O.se3_exp([0.3, 0, 0, 0, 0, 0]), 3.0, 1.0, max_iter=1)
        assert reg1.last_iterations == 1 == it1 and np.allclose(P1, Po1, atol=1e-12), cap


def test_align_degenerate_cases(K, O):
    reg = K.Registration(500, 1e-4, 0)
    guess = O.se3_exp([1, 2, 3, 0.1, 0.2, 0.3])
    src = rng.normal(size=(50, 3))
    empty = K.VoxelHashMap(1.0, 100.0, 20)
    assert np.allclose(reg.align_points_to_map(src, empty, guess, 3.0, 1.0), guess, atol=1e-15)  # Registration.cpp:143
    assert reg.last_iterations == 0
    far = K.VoxelHashMap(1.0, 1e9, 20)
    far.add_points(rng.normal(size=(100, 3)) + 1000.0)
    assert np.allclose(reg.align_points_to_map(src, far, guess, 3.0, 1.0), guess, atol=1e-15)  # JTJ = 0 -> dx = 0
    assert reg.last_iterations == 1
    assert np.allclose(reg.align_points_to_map(np.empty((0, 3)), far, guess, 3.0, 1.0), guess, atol=1e-15)
    with pytest.raises(ValueError):
        reg.align_points_to_map(src, far, np.diag([1.0, 1.0, -1.0, 1.0]), 3.0, 1.0)


def test_config1_known_answer(K, golden):
    g = K.VoxelHashMap(1.0, 100.0, 20)
    g.add_points(golden["c1_map_pts"])
    reg = K.Registration(500, 1e-4, 0)
    pose = reg.align_points_to_map(golden["c1_src"], g, golden["c1_guess"], 3.0, 1.0)
    dt, dr = pose_error(pose, golden["c1_pose"])
    assert dt < 1e-9 and dr < 1e-9 and reg.last_iterations == int(golden["c1_iters"])


# --------------------------------------------------------------------------- KissICP pipeline
@pytest.mark.parametrize("tag", ["a", "b"])
def test_pipeline_golden_streams(K, golden, tag):
    icp = K.KissICP(K.load_config())
    for k in range(10):
        pts = golden[f"{tag}_scan{k}"].astype(np.float64)
        ts = golden[f"{tag}_ts{k}"] if tag == "b" else np.empty(0)
        pre, src = icp.register_frame(pts, ts)
        dt, dr = pose_error(icp.last_pose, golden[f"{tag}_poses"][k])
        assert dt < 1e-4 and dr < 1e-4  # BASELINE bar
        assert dt < 1e-9 and dr < 1e-9  # expected
        assert len(pre) == golden[f"{tag}_npre"][k] and len(src) == golden[f"{tag}_nsrc"][k]
        assert icp.last_iterations == golden[f"{tag}_iters"][k]
        if k == 3:
            assert np.allclose(pre, golden[f"{tag}_pre3"], atol=1e-11)
            if tag == "a":
                assert np.array_equal(pre, golden["a_pre3"]) and np.array_equal(src, golden["a_src3"])
    gv, gc, gp = icp.local_map.dump()
    assert np.array_equal(gv, golden[f"{tag}_map_vox"]) and np.array_equal(gc, golden[f"{tag}_map_cnt"])
    assert np.allclose(gp, golden[f"{tag}_map_pts"], atol=1e-9)


@pytest.mark.parametrize("stamps,voxel,cap", [
    pytest.param("none", 1.0, 20, id="none-1.0"),
    pytest.param("column", 1.0, 20, id="column-1.0"),
    pytest.param("column", 0.3, 20, id="column-0.3"),
    pytest.param("none", 1.0, 40, id="none-1.0-cap40"),  # > 32 points per voxel: no ICP team, voxel-by-voxel walk
])
def test_pipeline_free_running_stream_vs_oracle(K, O, stamps, voxel, cap):
    from kiss_icp_b200 import synthetic
    L = synthetic.small_shape(seed=5, beams=32, cols=512, stamps=stamps)
    cfg = K.load_config(voxel_size=voxel, mapping__max_points_per_voxel=cap)
    g = K.KissICP(cfg)
    o = O.KissICP(voxel_size=voxel, max_points_per_voxel=cap)
    for k in range(25):
        p, t = L.scan(k)
        g.register_frame(p, t, return_clouds=False)
        o.register_frame(p, t, want_clouds=False)
        dt, dr = pose_error(g.last_pose, o.pose)
        assert dt < 1e-4 and dr < 1e-4, (k, dt, dr)
        assert dt < 1e-6 and dr < 1e-6, (k, dt, dr)  # expected: ~1e-15, up to ~1e-8 when a boundary point flips
        assert np.allclose(g.last_delta, o.delta, atol=1e-6)
    assert g.local_map.num_points() == o.local_map.num_points()
    assert np.isclose(g.adaptive_threshold.get_threshold(), o.sigma, rtol=1e-9)


def test_pipeline_modular_mode_equals_fused(K):
    """the reference's Python module-by-module sequence (kiss_icp.py:43-75) on the per-module
    device API gives the same trajectory as the fused kernel"""
    from kiss_icp_b200 import synthetic
    L = synthetic.small_shape(seed=9, beams=32, cols=512, stamps="column")
    a, b = K.KissICP(K.load_config(), fused=True), K.KissICP(K.load_config(), fused=False)
    for k in range(10):
        p, t = L.scan(k)
        fa, sa = a.register_frame(p, t)
        fb, sb = b.register_frame(p, t)
        assert np.allclose(fa, fb, atol=1e-12) and sa.shape == sb.shape
        dt, dr = pose_error(a.last_pose, b.last_pose)
        assert dt < 1e-9 and dr < 1e-9
    src, ds = a.voxelize(fa)
    src2, ds2 = b.voxelize(fa)
    assert np.array_equal(src, src2) and np.array_equal(ds, ds2)


def test_pipeline_kitti_shape_full_size(K, O):
    """BASELINE config-2 shape (64 x 1024) for a few scans, full size"""
    import torch
    from kiss_icp_b200 import synthetic
    L = synthetic.kitti_shape(seed=0, device="cuda" if torch.cuda.is_available() else "cpu")
    g, o = K.KissICP(K.load_config()), O.KissICP()
    for k in range(8):
        p, t = L.scan(k)
        assert len(p) > 60000
        g.register_frame(p, t, return_clouds=False)
        o.register_frame(p, t, want_clouds=False)
        dt, dr = pose_error(g.last_pose, o.pose)
        assert dt < 1e-8 and dr < 1e-8
    assert g.local_map.num_points() == o.local_map.num_points()


def test_pipeline_kitti_shape_500_scans_queued(K, O):
    """500 full-size KITTI-shape scans, free running through the QUEUED path (front-end prefetch, ICP team) against the
    oracle: pose per scan within 1e-6 m / 1e-6 rad (bar: 1e-4), identical iteration counts"""
    import torch
    from kiss_icp_b200 import synthetic
    L = synthetic.kitti_shape(seed=4, device="cuda")
    g, o = K.KissICP(K.load_config()), O.KissICP()
    worst, mism = 0.0, 0
    for lo in range(0, 500, 100):
        scans = [L.scan_torch(k)[0].contiguous() for k in range(lo, lo + 100)]
        torch.cuda.synchronize()
        g.start_history(100)
        poses = g._register_frames_raw([s.data_ptr() for s in scans], [s.shape[0] for s in scans], [None] * 100, [0] * 100, 2)
        its = [h.iterations for h in g.history()]
        for i, s in enumerate(scans):
            o.register_frame(s.cpu().numpy(), np.empty(0), want_clouds=False)
            dt, dr = pose_error(poses[i], o.pose)
            worst = max(worst, dt, dr)
            mism += int(its[i] != o.last_iterations)
            assert dt < 1e-4 and dr < 1e-4, (lo + i, dt, dr)
    assert worst < 1e-6 and mism == 0, (worst, mism)
    assert g.local_map.num_points() == o.local_map.num_points()


def test_pipeline_errors_and_state_accessors(K, O):
    icp = K.KissICP(K.load_config())
    with pytest.raises(IndexError):
        icp.register_frame(np.ones((10, 3)), np.array([0.0, 1.0]))
    T = O.se3_exp([1, 2, 3, 0.0, 0.0, 0.5])
    icp.last_pose = T
    assert np.allclose(icp.last_pose, T)
    with pytest.raises(ValueError):
        icp.last_delta = np.diag([1.0, 2.0, 1.0, 1.0])
    icp.register_frame(np.empty((0, 3)), np.empty(0))  # empty frame: pose = last_pose * last_delta
    assert np.allclose(icp.last_pose, T, atol=1e-12)


def test_pipeline_ouster128_shape_full_size(K, O):
    """BASELINE config-3 shape: 128 x 1024 rays, voxel 0.3 m, per-column stamps (deskew on), a few scans"""
    import torch
    from kiss_icp_b200 import synthetic
    L = synthetic.ouster128_shape(seed=2, device="cuda" if torch.cuda.is_available() else "cpu")
    g, o = K.KissICP(K.load_config(voxel_size=0.3)), O.KissICP(voxel_size=0.3)
    for k in range(5):
        p, t = L.scan(k)
        assert len(p) > 60000 and len(t) == len(p)
        g.register_frame(p, t, return_clouds=False)
        o.register_frame(p, t, want_clouds=False)
        dt, dr = pose_error(g.last_pose, o.pose)
        assert dt < 1e-4 and dr < 1e-4  # BASELINE bar
        assert dt < 1e-6 and dr < 1e-6  # expected ~1e-14 (device sin/cos in the deskew differ in the last ulps)
    assert abs(g.local_map.num_points() - o.local_map.num_points()) <= 2


def test_map_compact_keeps_content(K, O):
    pts = rng.normal(size=(40000, 3)) * 8
    g, o = K.VoxelHashMap(1.0, 20.0, 20), O.VoxelHashMap(1.0, 20.0, 20)
    g.add_points(pts)
    o.add_points(pts)
    g.remove_far_away_points([3.0, 0.0, 0.0])
    o.remove_far_away_points([3.0, 0.0, 0.0])
    g.compact()
    assert_maps_equal(g, o)
    q = pts[::7] + 0.1
    ap, ad = g.closest_neighbors(q)
    bp, bd = o.closest_neighbors(q)
    assert np.array_equal(ap, bp) and np.array_equal(ad, bd)


def test_pipeline_long_stream_with_table_rebuilds(K, O, monkeypatch):
    """300 free-running scans: eviction tombstones accumulate and the voxel table is rebuilt several times
    (growth into fresh allocations first, then same-size rebuilds that ping-pong with the spare table)"""
    from kiss_icp_b200 import synthetic
    monkeypatch.setenv("KB_MAP_RESERVE_SLOTS", "0")  # start from the minimal table instead of the sensor-sized one
    L = synthetic.small_shape(seed=21, beams=32, cols=512)
    g, o = K.KissICP(K.load_config(max_range=40.0)), O.KissICP(max_range=40.0, voxel_size=0.4)
    worst = 0.0
    for k in range(300):
        p, t = L.scan(k)
        g.register_frame(p, t, return_clouds=False)
        o.register_frame(p, t, want_clouds=False)
        dt, dr = pose_error(g.last_pose, o.pose)
        worst = max(worst, dt, dr)
        assert dt < 1e-4 and dr < 1e-4, (k, dt, dr)
    assert worst < 1e-6
    assert g.local_map.num_points() == o.local_map.num_points() and g.local_map.num_voxels() == o.local_map.num_voxels()
    gv, gc, gp = g.local_map.dump()
    ov, oc, op = canon_map(*o.local_map.dump())
    assert np.array_equal(gv, ov) and np.array_equal(gc, oc) and np.allclose(gp, op, atol=1e-9)


def test_pipeline_capacity_veto_and_retry(K, O, monkeypatch):
    """frames whose downsampled size exceeds the optimistic table sizing (every point its own voxel): the kernel
    vetoes the frame before touching any state, the host grows the table and replays it"""
    monkeypatch.setenv("KB_MAP_RESERVE_SLOTS", "0")  # start from the minimal table instead of the sensor-sized one
    g, o = K.KissICP(K.load_config(max_range=300.0, voxel_size=1.0)), O.KissICP(max_range=300.0, voxel_size=1.0)
    for k in range(4):
        pts = rng.uniform(-150, 150, size=(30000, 3)) * [1.0, 1.0, 0.2]
        g.register_frame(pts, np.empty(0), return_clouds=False)
        o.register_frame(pts, np.empty(0), want_clouds=False)
        dt, dr = pose_error(g.last_pose, o.pose)
        assert dt < 1e-6 and dr < 1e-6
        assert g.local_map.num_points() == o.local_map.num_points()
    assert g.grow_retries() >= 1


def test_pipeline_float32_ingestion_equals_float64(K):
    """kb_pipeline_register_frame_f32: float32 frames widened on the device give the same trajectory as the
    float64 call on the host-widened array"""
    from kiss_icp_b200 import synthetic
    for stamps in ("none", "column"):
        L = synthetic.small_shape(seed=13, beams=32, cols=512, stamps=stamps)
        a, b = K.KissICP(K.load_config()), K.KissICP(K.load_config())
        for k in range(8):
            p, t = L.scan(k)
            p32 = p.astype(np.float32)
            assert np.array_equal(p32.astype(np.float64), p)  # synthetic scans are fp32-representable like KITTI
            pa, sa = a.register_frame(p32, t)
            pb, sb = b.register_frame(p, t)
            assert np.array_equal(a.last_pose, b.last_pose)
            assert np.array_equal(pa, pb) and np.array_equal(sa, sb)


def test_pipeline_work_counters_and_profiling(K):
    """bookkeeping the bench relies on: per-frame ICP work counters, launch count, optional phase timestamps"""
    from kiss_icp_b200 import synthetic
    L = synthetic.small_shape(seed=17, beams=32, cols=512)
    icp = K.KissICP(K.load_config())
    icp.start_history(6)
    for k in range(6):
        if k == 3:
            icp.set_profiling(True)
        p, t = L.scan(k)
        icp.register_frame(p, t, return_clouds=False)
    h = icp.history()
    assert len(h) == 6 and h[0].iterations == 0 and h[0].icp_queries == 0
    for st in h[1:]:
        assert st.iterations >= 1 and st.icp_queries == st.iterations * st.n_source
        assert st.icp_candidates > st.icp_queries  # several candidate points per query on a populated map
        assert 0 < st.n_source <= st.n_downsampled <= st.n_preprocessed <= st.n_points_in
        assert st.map_points > 0 and st.map_voxels > 0
    assert all(sum(st.phase_us) == 0 for st in h[:3])          # timestamps are off by default
    assert all(10 < sum(st.phase_us) < 1e5 for st in h[3:])    # and plausible when switched on
    assert np.allclose(np.array(h[-1].pose).reshape(4, 4), icp.last_pose)


def test_register_frames_queue_equals_blocking_calls(K):
    """kb_pipeline_register_frames (queued, copy/compute overlapped) == the same frames through blocking
    RegisterFrame calls: poses bit-identical, same map, same history; f64 and f32 layouts, with and without stamps"""
    from kiss_icp_b200 import synthetic
    for stamps, f32 in (("column", False), ("none", False), ("column", True)):
        L = synthetic.small_shape(seed=5, beams=32, cols=512, stamps=stamps)
        scans = [L.scan(k) for k in range(25)]
        frames = [p.astype(np.float32) if f32 else p for p, _ in scans]
        ts = [t for _, t in scans]
        a, b = K.KissICP(K.load_config()), K.KissICP(K.load_config())
        a.start_history(25)
        b.start_history(25)
        want = np.empty((25, 4, 4))
        for k in range(25):
            a.register_frame(frames[k], ts[k], return_clouds=False)
            want[k] = a.last_pose
        got = np.concatenate([b.register_frames(frames[:7], ts[:7]), b.register_frames(frames[7:8], ts[7:8]),
                              b.register_frames(frames[8:], ts[8:])])
        assert np.array_equal(got, want)
        assert np.array_equal(b.last_pose, a.last_pose) and np.array_equal(b.last_delta, a.last_delta)
        for x, y in zip(a.local_map.dump(), b.local_map.dump()):
            assert np.array_equal(x, y)
        ha, hb = a.history(), b.history()
        assert [(h.iterations, h.n_source, h.map_points, h.icp_candidates) for h in ha] == \
               [(h.iterations, h.n_source, h.map_points, h.icp_candidates) for h in hb]
        # blocking calls continue seamlessly after a queued batch
        p, t = L.scan(25)
        a.register_frame(p.astype(np.float32) if f32 else p, t, return_clouds=False)
        b.register_frame(p.astype(np.float32) if f32 else p, t, return_clouds=False)
        assert np.array_equal(b.last_pose, a.last_pose)
    assert len(b.register_frames([], [])) == 0


def test_register_frames_veto_inside_the_queue(K, O, monkeypatch):
    """a frame in the middle of a queued sequence needs a bigger voxel table than planned: it vetoes itself, the
    frames queued behind it are skipped on the device, the host grows the table and replays from that frame"""
    monkeypatch.setenv("KB_MAP_RESERVE_SLOTS", "0")  # start from the minimal table instead of the sensor-sized one
    g, o = K.KissICP(K.load_config(max_range=300.0, voxel_size=1.0)), O.KissICP(max_range=300.0, voxel_size=1.0)
    frames = []
    for k in range(9):
        n = 30000 if k in (0, 4, 5) else 3000   # sparse clouds: every point its own voxel
        frames.append(rng.uniform(-150, 150, size=(n, 3)) * [1.0, 1.0, 0.2])
    poses = g.register_frames(frames)
    assert g.grow_retries() >= 2   # frame 0 (empty table) and the mid-queue one
    for k, f in enumerate(frames):
        o.register_frame(f, np.empty(0), want_clouds=False)
        dt, dr = pose_error(poses[k], o.pose)
        assert dt < 1e-6 and dr < 1e-6, (k, dt, dr)
    assert g.local_map.num_points() == o.local_map.num_points() and g.local_map.num_voxels() == o.local_map.num_voxels()


def test_register_frames_error_stops_the_sequence_where_the_loop_would(K):
    """frame 3 has too few timestamps (std::out_of_range in the reference): frames 0-2 are registered, then the
    error is raised, exactly like the dataset loop"""
    from kiss_icp_b200 import synthetic
    L = synthetic.small_shape(seed=6, beams=32, cols=512, stamps="column")
    scans = [L.scan(k) for k in range(5)]
    a, b = K.KissICP(K.load_config()), K.KissICP(K.load_config())
    for p, t in scans[:3]:
        a.register_frame(p, t, return_clouds=False)
    frames = [p for p, _ in scans]
    ts = [t for _, t in scans]
    ts[3] = ts[3][:10]
    with pytest.raises(IndexError):
        b.register_frames(frames, ts)
    assert np.array_equal(a.last_pose, b.last_pose)
    assert a.local_map.num_points() == b.local_map.num_points()


def test_correct_kitti_scan_matches_oracle(K, O):
    """kb_correct_kitti_scan[_dev] vs the oracle and the frozen vectors (float work: a few ulps allowed, the
    operation order is Eigen's so the expected difference is zero), then chained on the device into RegisterFrame"""
    import ctypes as C
    import os
    import torch
    from kiss_icp_b200 import _native as N, synthetic
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_kitti_v1.npz"))
    got = K.correct_kitti_scan(g["pts"])
    assert np.abs(got - g["corrected"]).max() <= 4e-14 * np.abs(g["pts"]).max()
    for n in (0, 1, 100_003):
        pts = rng.normal(size=(n, 3)) * [40.0, 40.0, 3.0]
        a, b = K.correct_kitti_scan(pts), O.correct_kitti_scan(pts)
        assert a.shape == b.shape and (n == 0 or np.abs(a - b).max() <= 4e-14 * 200.0)
    # device form: correct two scans on the device and register them without a host round trip
    L = synthetic.small_shape(seed=9, beams=32, cols=512)
    a, b = K.KissICP(K.load_config()), K.KissICP(K.load_config())
    for k in range(3):
        p, t = L.scan(k)
        a.register_frame(K.correct_kitti_scan(p), np.empty(0), return_clouds=False)
        d_in = torch.from_numpy(p).cuda()
        d_out = torch.empty_like(d_in)
        torch.cuda.synchronize()
        N.check(N.lib().kb_correct_kitti_scan_dev(C.c_void_p(d_in.data_ptr()), len(p), C.c_void_p(d_out.data_ptr())))
        torch.cuda.synchronize()  # the correction ran on the library's default stream of this thread
        assert np.array_equal(d_out.cpu().numpy(), K.correct_kitti_scan(p))
        N.check(N.lib().kb_pipeline_register_frame_dev(b._h, C.c_void_p(d_out.data_ptr()), len(p), None, 0))
        assert np.array_equal(a.last_pose, b.last_pose)


def test_one_host_thread_two_devices(K, O):
    """handles created by ONE host thread on device 0 and then on device 1 (kb_set_device): the opt-in to > 48 KB of dynamic
    shared memory is a per-device attribute of the kernels (it used to be cached per thread)"""
    from kiss_icp_b200 import _native as N, synthetic
    if N.lib().kb_device_count() < 2:
        pytest.skip("needs two GPUs")
    L = synthetic.small_shape(seed=2, beams=32, cols=512)
    try:
        for dev in (0, 1, 0):
            N.check(N.lib().kb_set_device(dev))
            g, o = K.KissICP(K.load_config()), O.KissICP()
            for k in range(4):
                p, t = L.scan(k)
                g.register_frame(p, t, return_clouds=False)
                o.register_frame(p, t, want_clouds=False)
                dt, dr = pose_error(g.last_pose, o.pose)
                assert dt < 1e-9 and dr < 1e-9, (dev, k)
    finally:
        N.check(N.lib().kb_set_device(0))
