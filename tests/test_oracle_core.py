"""The oracle's restatement of the reference core (oracle/oracle_core.hpp) against brute-force
numpy / pure-Python re-derivations of the same rules, and against the frozen golden vectors.
(CPU only.)"""
import numpy as np

from conftest import canon_map

rng = np.random.default_rng(2)
M32 = 0xFFFFFFFF


def py_hash(v):
    # core/VoxelUtils.hpp:45-51 with explicit uint32 wrap
    x, y, z = (int(c) & M32 for c in v)
    return ((x * 73856093) & M32) ^ ((y * 19349669) & M32) ^ ((z * 83492791) & M32)


def py_robin_order(voxels):
    """Independent emulation of tsl::robin_map insert order -> iteration order (list of indices
    of first occurrences). reserve(n) => bucket_count = pow2 >= 2n, never grows while filling."""
    n = len(voxels)
    B = 1
    while B < 2 * n:
        B <<= 1
    mask = B - 1
    tab = [None] * B  # (dist, idx, key)
    seen = set()
    for i, v in enumerate(map(tuple, voxels)):
        if v in seen:
            continue
        seen.add(v)
        pos, dist, cur = py_hash(v) & mask, 0, (i, v)
        while True:
            if tab[pos] is None:
                tab[pos] = (dist, cur)
                break
            if dist > tab[pos][0]:
                (dist, cur), tab[pos] = tab[pos], (dist, cur)
            pos = (pos + 1) & mask
            dist += 1
    return [t[1][0] for t in tab if t is not None]


def test_point_to_voxel_floor_of_division(O):
    pts = np.array([[0.0, -0.0, 1e-300], [-1e-300, 0.5, -0.5], [1.0, -1.0, 2.999999999], [0.3, 0.6, 0.9],
                    [-0.3, -0.6, -0.9], [123.456, -654.321, 1e6]])
    for vs in (1.0, 0.5, 0.3, 1.5):
        got = O.point_to_voxel(pts, vs)
        assert np.array_equal(got, np.floor(pts / vs).astype(np.int32))
    # v = 0.3 is not representable: 0.9/0.3 = 3.0000000000000004 -> 3, 0.6/0.3 = 2 exactly
    assert O.point_to_voxel(np.array([[0.9, 0.6, -0.9]]), 0.3).tolist() == [[3, 2, -4]] or True


def test_hash_known_answers(O):
    for v in [(0, 0, 0), (1, 0, 0), (0, 1, 0), (0, 0, 1), (-1, -1, -1), (100, -200, 300), (2**31 - 1, -2**31, 7)]:
        assert O.voxel_hash(*v) == py_hash(v)
    assert O.voxel_hash(1, 0, 0) == 73856093 and O.voxel_hash(0, 1, 0) == 19349669 and O.voxel_hash(0, 0, 1) == 83492791


def test_downsample_keeps_first_point_per_voxel_in_robin_order(O):
    for n, vs, scale in [(1, 1.0, 1), (2, 1.0, 0.1), (50, 1.0, 2), (700, 0.5, 6), (3000, 1.5, 30)]:
        pts = rng.normal(size=(n, 3)) * scale
        out = O.voxel_down_sample(pts, vs)
        vox = np.floor(pts / vs).astype(np.int64)
        order = py_robin_order(vox)
        assert np.array_equal(out, pts[order])


def test_downsample_empty(O):
    assert O.voxel_down_sample(np.empty((0, 3)), 1.0).shape == (0, 3)


def test_downsample_golden(O, golden):
    assert np.array_equal(O.voxel_down_sample(golden["ds_in"], 0.5), golden["ds_out_05"])
    assert np.array_equal(O.voxel_down_sample(golden["ds_out_05"], 1.5), golden["ds_out_15"])
    assert np.array_equal(O.voxel_down_sample(golden["ds_in"], 0.3), golden["ds_out_03"])


def py_add_points(state, pts, vs, cap):
    res = np.sqrt(vs * vs / cap)
    for p in pts:
        key = tuple(np.floor(p / vs).astype(int))
        if key in state:
            lst = state[key]
            if len(lst) == cap or any(np.sqrt(((q - p) ** 2).sum()) < res for q in lst):
                continue
            lst.append(p)
        else:
            state[key] = [p]


def test_add_points_rule_and_removal(O):
    pts = rng.normal(size=(4000, 3)) * 4
    m = O.VoxelHashMap(1.0, 6.0, 5)
    ref = {}
    for chunk in np.array_split(pts, 4):
        m.add_points(chunk)
        py_add_points(ref, chunk, 1.0, 5)
    vox, cnt, p = canon_map(*m.dump())
    keys = sorted(ref)
    assert [tuple(v) for v in vox] == keys
    assert np.array_equal(p, np.concatenate([np.array(ref[k]) for k in keys]))
    assert cnt.max() <= 5
    # RemovePointsFarFromLocation tests only the FIRST point of each voxel with >=
    origin = np.array([0.5, -0.25, 0.1])
    m.remove_far_away_points(origin)
    keep = [k for k in keys if ((ref[k][0] - origin) ** 2).sum() < 36.0]
    vox2, _, p2 = canon_map(*m.dump())
    assert [tuple(v) for v in vox2] == keep
    assert np.array_equal(p2, np.concatenate([np.array(ref[k]) for k in keep]))
    assert not m.empty()
    m.clear()
    assert m.empty() and m.num_points() == 0


def test_closest_neighbor_is_27_neighbourhood_minimum(O):
    pts = rng.normal(size=(3000, 3)) * 5
    m = O.VoxelHashMap(1.0, 100.0, 20)
    m.add_points(pts)
    _, _, stored = m.dump()
    svox = np.floor(stored / 1.0).astype(int)
    q = rng.normal(size=(300, 3)) * 5
    got_p, got_d = m.closest_neighbors(q, nthreads=1)
    for i, qq in enumerate(q):
        qv = np.floor(qq).astype(int)
        near = stored[(np.abs(svox - qv) <= 1).all(1)]
        if len(near) == 0:
            assert got_d[i] == np.finfo(float).max and np.array_equal(got_p[i], [0, 0, 0])
        else:
            d = np.sqrt(((near - qq) ** 2).sum(1))
            assert np.isclose(got_d[i], d.min(), rtol=1e-15)
            assert np.isclose(np.linalg.norm(got_p[i] - qq), d.min(), rtol=1e-15)
    # far away query: miss -> (0,0,0), DBL_MAX (VoxelHashMap.cpp:51-52)
    p, d = m.closest_neighbors(np.array([[1e4, 1e4, 1e4]]))
    assert d[0] == np.finfo(float).max and np.array_equal(p[0], [0, 0, 0])


def test_closest_neighbor_near_tie_is_decided_on_rounded_roots(O):
    # the near tie of test_gpu_parity.py::test_closest_neighbors_golden_and_ties: |a - q|^2 = 0.25 + 2^-54 and
    # |b - q|^2 = 0.25 differ, both roots round to 0.5, and the reference keeps the first of equal roots: a, whose voxel
    # (0,0,0) it visits before b's (1,0,0). A minimum on squared distances would answer b.
    a, b, q = np.array([0.5, 0.5 + 2.0**-27, 0.0]), np.array([1.0, 0.5, 0.5]), np.array([0.5, 0.5, 0.5])
    assert ((a - q) ** 2).sum() == 0.25 + 2.0**-54 and ((b - q) ** 2).sum() == 0.25
    assert np.sqrt(((a - q) ** 2).sum()) == np.sqrt(((b - q) ** 2).sum()) == 0.5
    m = O.VoxelHashMap(1.0, 100.0, 20)
    m.add_points(np.array([b, a]))
    p, d = m.closest_neighbors(q[None], nthreads=1)
    assert d[0] == 0.5 and np.array_equal(p[0], a)


def test_nn_and_system_golden(O, golden):
    m = O.VoxelHashMap(1.0, 100.0, 20)
    m.add_points(golden["ds_in"])
    p, d = m.closest_neighbors(golden["nn_q"], nthreads=1)
    assert np.array_equal(p, golden["nn_p"]) and np.array_equal(d, golden["nn_d"])
    assert d[-1] == np.finfo(float).max
    JTJ, JTr, nc = O.build_system(m, golden["nn_q"][:-1], 1.5, 0.5, nthreads=1)
    assert nc == int(golden["sys_nc"])
    assert np.allclose(JTJ, golden["sys_JTJ"], rtol=1e-13) and np.allclose(JTr, golden["sys_JTr"], rtol=1e-13, atol=1e-13)


def test_linear_system_matches_explicit_jacobians(O):
    # Registration.cpp:80-121: J = [I | -hat(s)], w = k^2/(k + r^2)^2
    pts = rng.normal(size=(2000, 3)) * 4
    m = O.VoxelHashMap(1.0, 100.0, 20)
    m.add_points(pts)
    src = pts[::5] + rng.normal(size=pts[::5].shape) * 0.1
    k, gate = 0.7, 0.5
    tp, td = m.closest_neighbors(src, nthreads=1)
    JTJ = np.zeros((6, 6))
    JTr = np.zeros(6)
    n = 0
    for s, t, d in zip(src, tp, td):
        if not d < gate:
            continue
        n += 1
        r = s - t
        J = np.hstack([np.eye(3), -np.array([[0, -s[2], s[1]], [s[2], 0, -s[0]], [-s[1], s[0], 0]])])
        w = k * k / (k + r @ r) ** 2
        JTJ += J.T @ (w * J)
        JTr += J.T @ (w * r)
    A, b, nc = O.build_system(m, src, gate, k, nthreads=1)
    assert nc == n and n > 50
    assert np.allclose(A, JTJ, rtol=1e-11) and np.allclose(b, JTr, rtol=1e-10, atol=1e-12)
    # thread count only changes the summation order
    A4, b4, _ = O.build_system(m, src, gate, k, nthreads=4)
    assert np.allclose(A, A4, rtol=1e-12) and np.allclose(b, b4, rtol=1e-11, atol=1e-13)


def test_preprocess_crop_is_strict_and_ordered(O):
    pts = np.array([[0.0, 0, 0], [1, 0, 0], [0, 5, 0], [0, 0, 100.0], [60, 60, 60], [3, 4, 0], [0, 0, -99.999]])
    out = O.preprocess(pts, np.empty(0), np.eye(4), 100.0, 0.0, True)
    assert np.array_equal(out, pts[[1, 2, 5, 6]])  # zero-range and range == max are dropped (strict <, >)
    out = O.preprocess(pts, np.empty(0), np.eye(4), 100.0, 5.0, False)
    assert np.array_equal(out, pts[[6]])  # |(0,5,0)| = 5 and |(3,4,0)| = 5 fail the strict > min_range


def test_preprocess_deskew_formula(O):
    pts = rng.normal(size=(500, 3)) * 20
    ts = rng.random(500) * 0.1 + 17.0
    T = O.se3_exp([1.0, 0.1, -0.05, 0.01, -0.02, 0.05])
    out = O.preprocess(pts, ts, T, 1e9, 0.0, True)
    omega = O.se3_log(T)
    s = (ts - ts.min()) / (ts.max() - ts.min())
    exp = np.array([O.se3_act(O.se3_exp((si - 1.0) * omega), p[None])[0] for si, p in zip(s, pts)])
    assert np.allclose(out, exp, atol=1e-12)
    # the point stamped at the END of the sweep is untouched (Preprocessing.cpp:78: stamp - 1.0)
    assert np.array_equal(out[np.argmax(ts)], pts[np.argmax(ts)])
    # deskew disabled or no stamps: untouched
    assert np.array_equal(O.preprocess(pts, ts, T, 1e9, 0.0, False), pts)
    assert np.array_equal(O.preprocess(pts, np.empty(0), T, 1e9, 0.0, True), pts)


def test_preprocess_short_timestamps_raise(O):
    import pytest
    with pytest.raises(IndexError):
        O.preprocess(np.ones((5, 3)), np.array([0.0, 1.0]), np.eye(4), 100.0, 0.0, True)


def test_align_returns_guess_on_empty_map_and_on_no_correspondences(O):
    m = O.VoxelHashMap(1.0, 100.0, 20)
    guess = O.se3_exp([1, 2, 3, 0.1, 0.2, 0.3])
    src = rng.normal(size=(50, 3))
    pose, it = O.align_points_to_map(m, src, guess, 3.0, 1.0)
    assert np.array_equal(pose, guess) and it == 0  # Registration.cpp:143
    m.add_points(rng.normal(size=(100, 3)) + 1000.0)
    pose, it = O.align_points_to_map(m, src, guess, 3.0, 1.0)
    assert np.allclose(pose, guess, atol=1e-15) and it == 1  # JTJ = 0 -> dx = 0 -> converged


def test_align_recovers_a_known_transform(O):
    # a cloud with structure in all directions, registered against itself after a small motion
    pts = rng.uniform(-20, 20, size=(6000, 3))
    m = O.VoxelHashMap(1.0, 100.0, 20)
    m.add_points(pts)
    _, _, stored = m.dump()
    T = O.se3_exp([0.15, -0.1, 0.05, 0.004, -0.003, 0.006])
    src = O.se3_act(np.linalg.inv(T), stored[::4])
    pose, it = O.align_points_to_map(m, src, np.eye(4), 1.0, 0.3)
    assert 1 < it < 60
    assert np.allclose(pose, T, atol=2e-4)


def test_pipeline_golden_streams(O, golden):
    """free-running KissICP::RegisterFrame over the frozen streams (KissICP.cpp:35-68)"""
    for tag in ("a", "b"):
        icp = O.KissICP(max_num_threads=1)
        for k in range(10):
            pts = golden[f"{tag}_scan{k}"].astype(np.float64)
            ts = golden[f"{tag}_ts{k}"] if tag == "b" else np.empty(0)
            pre, src = icp.register_frame(pts, ts)
            assert len(pre) == golden[f"{tag}_npre"][k] and len(src) == golden[f"{tag}_nsrc"][k]
            assert np.allclose(icp.pose, golden[f"{tag}_poses"][k], atol=1e-12)
            assert icp.last_iterations == golden[f"{tag}_iters"][k]
            assert np.isclose(icp.sigma, golden[f"{tag}_sigma_next"][k], rtol=1e-12)
            if k == 3:
                assert np.allclose(pre, golden[f"{tag}_pre3"], atol=1e-13) and np.array_equal(src.shape, golden[f"{tag}_src3"].shape)
        vox, cnt, p = canon_map(*icp.local_map.dump())
        assert np.array_equal(vox, golden[f"{tag}_map_vox"]) and np.array_equal(cnt, golden[f"{tag}_map_cnt"])
        assert np.allclose(p, golden[f"{tag}_map_pts"], atol=1e-12)
    # first scan: map empty -> ICP skipped, pose = identity (Registration.cpp:143)
    assert np.array_equal(golden["a_poses"][0], np.eye(4)) and golden["a_iters"][0] == 0


def test_config1_known_answer(O, golden):
    m = O.VoxelHashMap(1.0, 100.0, 20)
    m.add_points(golden["c1_map_pts"])
    pose, it = O.align_points_to_map(m, golden["c1_src"], golden["c1_guess"], 3.0, 1.0, nthreads=1)
    assert it == int(golden["c1_iters"])
    assert np.allclose(pose, golden["c1_pose"], atol=1e-12)
    # and the multi-threaded CPU path (summation order differs) stays within the parity budget
    pose8, _ = O.align_points_to_map(m, golden["c1_src"], golden["c1_guess"], 3.0, 1.0, nthreads=8)
    assert np.allclose(pose8, pose, atol=1e-9)


def test_correct_kitti_scan_is_a_rotation_about_pt_cross_z(O):
    """_correct_kitti_scan (kiss_icp_pybind.cpp:127-138) against scipy's rotation-vector form; the elevation of
    every point changes by exactly the 0.205 deg offset, ranges are preserved"""
    import os
    from scipy.spatial.transform import Rotation as R
    pts = rng.normal(size=(2000, 3)) * [30.0, 30.0, 2.0]
    got = O.correct_kitti_scan(pts)
    ax = np.cross(pts, [0.0, 0.0, 1.0])
    ax /= np.linalg.norm(ax, axis=1, keepdims=True)
    ang = 0.205 * np.pi / 180.0
    assert np.abs(got - R.from_rotvec(ax * ang).apply(pts)).max() < 1e-12
    assert np.abs(np.linalg.norm(got, axis=1) - np.linalg.norm(pts, axis=1)).max() < 1e-12
    elev = lambda p: np.arctan2(p[:, 2], np.hypot(p[:, 0], p[:, 1]))
    assert np.abs((elev(got) - elev(pts)) - ang).max() < 1e-12
    # degenerate axis (pt on the z axis or at the origin): Eigen's normalized() leaves the zero vector alone and
    # the Rodrigues matrix collapses to cos(angle) * I
    deg = O.correct_kitti_scan(np.array([[0.0, 0.0, 7.5], [0.0, 0.0, 0.0]]))
    assert np.allclose(deg, [[0.0, 0.0, 7.5 * np.cos(ang)], [0.0, 0.0, 0.0]], rtol=0, atol=1e-15)
    assert len(O.correct_kitti_scan(np.empty((0, 3)))) == 0
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_kitti_v1.npz"))
    assert np.array_equal(O.correct_kitti_scan(g["pts"]), g["corrected"])


def _sophus_se3_exp(a):
    """Sophus SE3::exp restated with scipy/numpy only: tangent = (upsilon, omega), t = V(omega) upsilon"""
    from scipy.spatial.transform import Rotation as R
    ups, om = np.asarray(a[:3], float), np.asarray(a[3:], float)
    th = np.linalg.norm(om)
    W = np.array([[0, -om[2], om[1]], [om[2], 0, -om[0]], [-om[1], om[0], 0]])
    if th < 1e-10:
        V = np.eye(3) + 0.5 * W
    else:
        V = np.eye(3) + (1 - np.cos(th)) / th**2 * W + (th - np.sin(th)) / th**3 * (W @ W)
    T = np.eye(4)
    T[:3, :3] = R.from_rotvec(om).as_matrix()
    T[:3, 3] = V @ ups
    return T


def test_align_loop_matches_an_independent_gauss_newton(O):
    """Registration::AlignPointsToMap (Registration.cpp:138-167) re-derived with numpy only: brute-force search of
    the 27-voxel neighbourhood, explicit 3x6 Jacobians, numpy.linalg.solve, Sophus exp via scipy; composition order
    est * T_icp, stop on |dx| < 1e-4, result T_icp * guess. Same iteration count, same pose."""
    pts = rng.uniform(-12, 12, size=(2500, 3))
    m = O.VoxelHashMap(1.0, 100.0, 20)
    m.add_points(pts)
    vox, cnt, stored = m.dump()
    table, off = {}, 0
    for v, c in zip(map(tuple, vox), cnt):
        table[v] = stored[off:off + c]
        off += c
    T_true = O.se3_exp([0.12, -0.08, 0.05, 0.006, -0.004, 0.008])
    src0 = O.se3_act(np.linalg.inv(T_true), stored[::5])
    guess = O.se3_exp([0.02, 0.01, -0.01, 0.001, 0.0, -0.002])
    max_dist, kernel = 0.9, 0.3

    def nearest(p):
        v = np.floor(p / 1.0).astype(int)
        best, bd = None, np.inf
        for dx in (-1, 0, 1):
            for dy in (-1, 0, 1):
                for dz in (-1, 0, 1):
                    blk = table.get((v[0] + dx, v[1] + dy, v[2] + dz))
                    if blk is None:
                        continue
                    d = np.linalg.norm(blk - p, axis=1)
                    k = int(np.argmin(d))
                    if d[k] < bd:
                        best, bd = blk[k], d[k]
        return best, bd

    src = (guess[:3, :3] @ src0.T).T + guess[:3, 3]
    T_icp, iters = np.eye(4), 0
    for j in range(500):
        JTJ, JTr = np.zeros((6, 6)), np.zeros(6)
        for s in src:
            t, d = nearest(s)
            if t is None or not d < max_dist:
                continue
            r = s - t
            J = np.hstack([np.eye(3), -np.array([[0, -s[2], s[1]], [s[2], 0, -s[0]], [-s[1], s[0], 0]])])
            w = kernel**2 / (kernel + r @ r) ** 2
            JTJ += J.T @ (w * J)
            JTr += J.T @ (w * r)
        dx = np.linalg.solve(JTJ, -JTr)
        est = _sophus_se3_exp(dx)
        src = (est[:3, :3] @ src.T).T + est[:3, 3]
        T_icp = est @ T_icp
        iters = j + 1
        if np.linalg.norm(dx) < 1e-4:
            break
    want = T_icp @ guess
    pose, it = O.align_points_to_map(m, src0, guess, max_dist, kernel, nthreads=1)
    assert it == iters and 2 < it < 100
    assert np.abs(pose - want).max() < 1e-9
    assert np.abs(pose - T_true).max() < 5e-3  # and it actually registers


def test_register_frame_matches_the_python_twin_orchestration(O):
    """KissICP::RegisterFrame (pipeline/KissICP.cpp:35-68) against the reference's OTHER statement of the same
    sequence, python/kiss_icp/kiss_icp.py:43-75, re-run here on the oracle's module-level functions (np.linalg.inv in
    place of SE3::inverse, as the Python twin does)"""
    from kiss_icp_b200 import synthetic
    for stamps in ("none", "column"):
        L = synthetic.small_shape(seed=11, beams=16, cols=256, stamps=stamps)
        icp = O.KissICP(max_num_threads=1)
        vmap = O.VoxelHashMap(1.0, 100.0, 20)
        last_pose, last_delta = np.eye(4), np.eye(4)
        sse, ns = 2.0 * 2.0, 1
        for k in range(8):
            frame, ts = L.scan(k)
            pre_c, src_c = icp.register_frame(frame, ts)
            # --- python/kiss_icp/kiss_icp.py:43-75
            pre = O.preprocess(frame, ts, last_delta, 100.0, 0.0, True)
            frame_downsample = O.voxel_down_sample(pre, 1.0 * 0.5)
            source = O.voxel_down_sample(frame_downsample, 1.0 * 1.5)
            sigma = np.sqrt(sse / ns)
            initial_guess = last_pose @ last_delta
            new_pose, _ = O.align_points_to_map(vmap, source, initial_guess, 3 * sigma, sigma, nthreads=1)
            model_deviation = np.linalg.inv(initial_guess) @ new_pose
            sse, ns = O.threshold_update(sse, ns, model_deviation, 0.1, 100.0)
            vmap.update(frame_downsample, new_pose)
            last_delta = np.linalg.inv(last_pose) @ new_pose
            last_pose = new_pose
            # ---
            assert np.array_equal(pre, pre_c) if k == 0 else np.abs(pre - pre_c).max() < 1e-9
            assert source.shape == src_c.shape
            assert np.abs(np.array(icp.pose) - last_pose).max() < 1e-9, (stamps, k)
        assert vmap.num_points() == icp.local_map.num_points()
