"""CPU tests of the oracle (no GPU): the C restatement against (1) the committed golden vectors produced
by the REFERENCE'S OWN kernel source (tests/golden, written by tests/golden/make_golden.py), (2) an independent
NumPy restatement of the index arithmetic."""
import os

import numpy as np
import pytest

from elevation_mapping_cupy_b200 import workloads as wl
from elevation_mapping_cupy_b200.parameter import Parameter, core_parameter
from helpers import digest, load_golden

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("seed", [0, 1])
def test_point_index_matches_reference_golden(oracle_mod, seed):
    """bit-identical (idx, valid, inside) vs the reference kernel's write-back (CK.py:260-262)"""
    g = np.load(os.path.join(GOLD, f"index_default202_seed{seed}.npz"))
    p = Parameter(); p.update()
    pts, R, t = wl.reference_test_cloud(seed, n=20000)
    if seed % 2:
        pts = (pts * np.float32(9.0) - np.float32(4.5)).astype(np.float32)
    idx, valid, inside, _ = oracle_mod.point_index(p, pts, R, t)
    assert np.array_equal(idx, g["idx"])
    assert np.array_equal(valid, g["valid"])
    assert np.array_equal(inside, g["inside"])
    # independent NumPy restatement of the same arithmetic
    ni, nv, nin = oracle_mod.point_index_numpy(p, pts, R, t)
    assert np.array_equal(ni, idx) and np.array_equal(nv, valid) and np.array_equal(nin, inside)


def test_index_numpy_vs_c_on_large_map(oracle_mod):
    p = core_parameter(2048)
    rng = np.random.default_rng(5)
    pts = rng.uniform(-45, 45, (50000, 3)).astype(np.float32)
    R = np.eye(3, dtype=np.float32); t = np.array([0.3, -0.2, 1.0], np.float32)
    a = oracle_mod.point_index(p, pts, R, t)
    b = oracle_mod.point_index_numpy(p, pts, R, t)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])


def test_frames_match_reference_golden(oracle_mod):
    """4 LiDAR frames on a 130^2 map: the oracle's state equals (a) its own committed output exactly and
    (b) the reference kernel source's output to 1e-6 on every cell whose outcome is order-independent."""
    g = np.load(os.path.join(GOLD, "frames_core130.npz"))
    p = core_parameter(130)
    om = oracle_mod.OracleElevationMap(p)
    for f in range(4):
        pts, R, t = wl.lidar_cloud(0, f, n_rings=24, n_az=500, max_range=4.0)
        om.move_to(t, R)
        om.input_pointcloud(pts, ["x", "y", "z"], R, t, 0.02, 0.02)
        for li in (0, 1, 2, 4, 5, 6):
            assert np.array_equal(om.elevation_map[li], g[f"oracle_state_{f}"][li]), (f, li)
        assert np.abs(om.elevation_map[3] - g[f"oracle_state_{f}"][3]).max() < 1e-6
        assert np.array_equal(om.normal_map, g[f"oracle_normal_{f}"])
        racy = g[f"racy_{f}"]
        assert racy.mean() < 0.05
        for li in (0, 1, 2, 4, 5, 6):
            d = np.abs(om.elevation_map[li] - g[f"ref_state_{f}"][li])
            assert d[~racy].max() <= 1e-6, (f, li, d[~racy].max())
        assert np.array_equal(om.last_point_record[0], g[f"ref_point_idx_{f}"])
        om.update_variance(); om.update_time()


def test_oracle_threads_are_deterministic(oracle_mod):
    p = core_parameter(130)
    a = oracle_mod.OracleElevationMap(p, nthreads=1); b = oracle_mod.OracleElevationMap(p, nthreads=4)
    for f in range(2):
        pts, R, t = wl.lidar_cloud(0, f, n_rings=24, n_az=500, max_range=4.0)
        for m in (a, b):
            m.input_pointcloud(pts, ["x", "y", "z"], R, t, 0.02, 0.02); m.update_time()
    assert np.array_equal(a.elevation_map, b.elevation_map)
    assert np.array_equal(a.normal_map, b.normal_map)


def test_multi_sensor_equals_concatenation_when_poses_equal(oracle_mod):
    p = core_parameter(130)
    a = oracle_mod.OracleElevationMap(p); b = oracle_mod.OracleElevationMap(p)
    pts, R, t = wl.lidar_cloud(0, 0, n_rings=24, n_az=500, max_range=4.0)
    a.input_pointcloud(pts, ["x", "y", "z"], R, t, 0.0, 0.0)
    b.input_sensors([pts[:5000], pts[5000:]], [R, R], [t, t], 0.0, 0.0)
    assert np.array_equal(a.elevation_map, b.elevation_map)


def test_traversability_matches_torch_cpu(oracle_mod):
    """traversability_filter.py:15-42 on the host with torch vs the oracle's direct convolution"""
    torch = pytest.importorskip("torch")
    p = core_parameter(130)
    rm_w = oracle_mod.load_weights(p)
    x = np.random.default_rng(0).standard_normal((130, 130)).astype(np.float32)
    ours = oracle_mod.traversability(130, x, rm_w)
    import torch.nn.functional as F
    w1, w2, w3, wo = [torch.from_numpy(w) for w in rm_w]
    e = torch.from_numpy(x).view(1, 1, 130, 130)
    o1 = F.conv2d(e, w1.view(4, 1, 3, 3), dilation=1)[:, :, 2:-2, 2:-2]
    o2 = F.conv2d(e, w2.view(4, 1, 3, 3), dilation=2)[:, :, 1:-1, 1:-1]
    o3 = F.conv2d(e, w3.view(4, 1, 3, 3), dilation=3)
    ref = torch.exp(-F.conv2d(torch.cat((o1, o2, o3), 1).abs(), wo.view(1, 12, 1, 1)))[0, 0].numpy()
    assert np.abs(ours - ref).max() < 2e-6


def test_smooth_matches_scipy(oracle_mod):
    from scipy import ndimage
    x = np.random.default_rng(1).standard_normal((202, 202)).astype(np.float32)
    ours = oracle_mod.smooth(202, x)
    ref = ndimage.uniform_filter(ndimage.uniform_filter(x, size=3), size=3)     # smooth_filter.py:57-58
    assert np.abs(ours - ref).max() < 1e-6


def test_dilation_and_normal_against_reference_source(oracle_mod):
    """pin against the reference's dilation / normal / min_filter kernels (their output stored in reference_cpu.npz)"""
    g = load_golden("reference_cpu")
    p = core_parameter(130)
    rng = np.random.default_rng(3)
    W = 130
    h = rng.standard_normal((W, W)).astype(np.float32)
    mask = (rng.random((W, W)) < 0.15).astype(np.float32)
    mask[:, :4] = (rng.random((W, 4)) < 0.6); mask[:, -4:] = (rng.random((W, 4)) < 0.6)   # exercise the row wrap-around
    ours, _ = oracle_mod.dilation(W, p.dilation_size, h, mask)
    assert digest(ours) == g["dilation_sha"]
    # the host build of the reference source has no FMA contraction (g++ -ffp-contract=off) while the oracle
    # follows nvcc's contraction of CK.py:497 (fma(nx,nx, ny*ny) + 1): last-ulp differences only
    on = oracle_mod.normal(W, p.resolution, ours, mask)
    assert digest(on != 0) == g["normal_nonzero_sha"]
    assert np.abs(on.reshape(3, -1)[:, g["normal_cells"]] - g["normal_vals"]).max() <= 2.4e-7
    # min_filter: the reference updates in place (Gauss-Seidel); with one iteration on a mask whose invalid
    # cells have no invalid neighbours inside the window the two orders coincide
    m2 = np.ones((W, W), np.float32); m2[5:-5:4, 5:-5:4] = 0
    ours_mf, _ = oracle_mod.min_filter(W, 1, 1, h, m2)
    assert digest(np.nan_to_num(ours_mf).astype(np.float32)) == g["min_filter_sha"]


def test_star_plugin_oracles_against_reference_source(oracle_mod):
    """max_filter / robot_centric_elevation restatements vs the reference's kernels (host build of their source,
    output stored in reference_cpu.npz)."""
    g = load_golden("reference_cpu")
    p = core_parameter(130)
    W = 130
    rng = np.random.default_rng(8)
    h = rng.standard_normal((W, W)).astype(np.float32)
    m = (rng.random((W, W)) < 0.3).astype(np.float32)
    # max_filter.py:100-113: every launch reads COPIES of the running arrays
    ours, _ = oracle_mod.max_filter(W, 1, 4, h, m)
    assert digest(np.nan_to_num(ours, nan=-7).astype(np.float32)) == g["max_filter_sha"]
    # robot_centric_elevation.py:118-121
    R = np.array([[0.9, 0.1, -0.2], [0.0, 1.0, 0.1], [0.15, -0.12, 0.97]], np.float32)
    assert digest(oracle_mod.robot_centric(W, p.resolution, 1.1, True, h, m, R)) == g["rce_thr_sha"]
    ours = oracle_mod.robot_centric(W, p.resolution, 1.1, False, h, m, R)
    # host build has no FMA contraction: last-ulp differences
    assert np.abs(ours.ravel()[g["rce_raw_cells"]] - g["rce_raw_vals"]).max() <= 5e-7 * max(1.0, g["rce_raw_absmax"])


def _drift_frames(n=5):
    out = []
    for f in range(n):
        pts, R, t = wl.lidar_cloud(0, f, n_rings=24, n_az=500, max_range=4.0)
        pts = pts.copy(); pts[:, 2] += np.float32(0.03 * (f % 2))     # alternating 3 cm bias -> non-zero mean error
        out.append((pts, R, t))
    return out


EXACT_LAYERS = [0, 1, 2, 4, 5, 6]


def test_drift_compensation_against_reference_source(oracle_mod):
    """EM.py:346-357 fires (error_cnt > min_height_drift_cnt, |mean| < max_drift): oracle vs the reference's kernels.
    reference_cpu.npz holds, per frame, the reference's state on a seeded sample of the cells on which input order
    and reverse order agree (each reference frame started from the oracle's state) and its mean error."""
    from oracle.configs import DRIFT_OVERRIDES
    g = load_golden("reference_cpu")
    p = core_parameter(130, **DRIFT_OVERRIDES)
    om = oracle_mod.OracleElevationMap(p)
    fired = 0
    for f, (pts, R, t) in enumerate(_drift_frames()):
        om.move_to(t, R); om.input_pointcloud(pts, ["x", "y", "z"], R, t, 0.02, 0.02)
        ours = om.elevation_map[EXACT_LAYERS].reshape(6, -1)[:, g[f"drift_cells_{f}"]]
        d = np.abs(ours - g[f"drift_vals_{f}"])
        assert d.max() <= 1e-6, (f, d.max(1))
        if om.stats.drift_applied:
            fired += 1
            assert abs(om.stats.mean_error - g[f"drift_mean_error_{f}"]) < 1e-6
        om.update_variance(); om.update_time()
    assert fired >= 3


FLAG_CASES = [
    dict(enable_edge_sharpen=False),
    dict(enable_visibility_cleanup=False),
    dict(enable_overlap_clearance=False, enable_drift_compensation=False),
    dict(max_ray_length=2.0, cleanup_step=0.01, cleanup_cos_thresh=0.5, wall_num_thresh=3, dilation_size=2,
         min_valid_distance=0.3, mahalanobis_thresh=1.0),
]


@pytest.mark.parametrize("flags", FLAG_CASES)
def test_flag_combinations_against_reference_source(oracle_mod, flags):
    """feature toggles and thresholds are baked into the reference's kernel source (one build per combination):
    three frames against its output stored in reference_cpu.npz, on a seeded sample of the order-independent cells"""
    g = load_golden("reference_cpu")
    k = FLAG_CASES.index(flags)
    p = core_parameter(130, **flags)
    om = oracle_mod.OracleElevationMap(p)
    for f in range(3):
        pts, R, t = wl.lidar_cloud(0, f, n_rings=24, n_az=500, max_range=4.0)
        om.move_to(t, R); om.input_pointcloud(pts, ["x", "y", "z"], R, t, 0.02, 0.02)
        ours = om.elevation_map[EXACT_LAYERS].reshape(6, -1)[:, g[f"flags{k}_cells_{f}"]]
        ref = g[f"flags{k}_vals_{f}"]
        for j, li in enumerate(EXACT_LAYERS):
            d = np.abs(ours[j] - ref[j])
            assert int((d > 1e-6).sum()) <= 3, (flags, f, li, float(d.max()))      # symmetric order-dependent patterns
        assert digest(om.last_point_record[0]) == g[f"flags{k}_point_idx_sha_{f}"]
        assert g[f"flags{k}_n_cmp_{f}"] > 0.9 * 130 * 130
        om.update_variance(); om.update_time()


def test_semantic_fusion_oracle_against_reference_source(oracle_mod):
    """SURVEY 8(f)2: the NumPy restatement of the point-channel fusions (average, class_average, color) against the
    reference's own kernel strings (fusion/pointcloud_average.py, pointcloud_class_average.py, pointcloud_color.py),
    compiled for the host by oracle/build_ref.py and run one element at a time in input order; their output is
    stored in reference_cpu.npz."""
    g = load_golden("reference_cpu")
    p = core_parameter(130)
    W = 130
    rng = np.random.default_rng(3)
    pts, R, t = wl.uniform_cloud(0, 1, n=6000, half_extent=2.3)
    idx, valid, inside, _ = oracle_mod.point_index(p, pts, R, t)
    feats = np.stack([rng.random(len(pts), dtype=np.float32) * 3, rng.random(len(pts), dtype=np.float32),
                      rng.integers(0, 1 << 24, len(pts)).astype(np.uint32).view(np.float32)], 1)
    kinds = ["average", "class_average", "color"]
    cnt = np.bincount(idx[(valid > 0) & (inside > 0)], minlength=W * W).astype(np.float32)
    cnt[rng.random(W * W) < 0.3] = 0          # as if some cells' points had been rejected by the fusion (CK.py:174-179)
    sem_or = np.zeros((3, W, W), np.float32)
    for frame in range(2):                    # second frame exercises class_average's running mix
        oracle_mod.semantic_fuse(W, idx, valid, inside, feats, kinds, sem_or, cnt, alpha=0.5)
        assert digest(sem_or[2].view(np.uint32)) == g[f"sem_color_sha_{frame}"], "color"
        ours = sem_or[:2].reshape(2, -1)[:, g[f"sem_cells_{frame}"]]
        for k in (0, 1):
            d = np.abs(ours[k] - g[f"sem_vals_{frame}"][k])
            assert d.max() <= 2e-6 * max(1.0, float(g[f"sem_absmax_{frame}"][k])), (frame, kinds[k], float(d.max()))
