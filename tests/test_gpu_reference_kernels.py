"""The engine against the REFERENCE'S OWN kernels run on a B200 (tests/ref_gpu.py); their output is stored in
tests/golden/reference_gpu.npz (written by tests/golden/make_golden.py --gpu)."""
import numpy as np
import pytest

from helpers import digest, load_golden

pytestmark = pytest.mark.gpu


def _mk(param):
    from elevation_mapping_cupy_b200.elevation_mapping import ElevationMap
    return ElevationMap(param)


def test_indices_bit_identical_to_reference_gpu_kernels():
    from elevation_mapping_cupy_b200.parameter import Parameter, core_parameter
    from elevation_mapping_cupy_b200 import workloads as wl
    g = load_golden("reference_gpu")
    for tag, p, cloud in (("default202", Parameter(), "rand"), ("core1024", core_parameter(1024), "lidar")):
        p.update()
        em = _mk(p)
        if cloud == "rand":
            pts, R, t = wl.reference_test_cloud(3)
            pts = (pts * np.float32(9.0) - np.float32(4.5)).astype(np.float32)
        else:
            pts, R, t = wl.lidar_cloud(1, 2)
        em.input_pointcloud(pts, ["x", "y", "z"], R, t, 0, 0)
        idx, valid, inside = em.get_point_record(len(pts))
        ref_idx, ref_valid, ref_inside = g[f"index_{tag}_sha"]
        assert digest(idx.astype(np.int32)) == ref_idx, tag
        assert digest(valid.astype(np.uint8)) == ref_valid, tag
        assert digest(inside.astype(np.uint8)) == ref_inside, tag


def test_state_matches_reference_gpu_kernels_on_order_independent_cells():
    """Same pre-frame state in both; the reference GPU kernel was run three times per frame (its races resolve
    differently from launch to launch and for permuted inputs): cells on which those runs agree are order-
    independent, and there the engine must match to 1e-4 (BASELINE) -- in practice ~1e-6.  The stored fixture holds
    the first run's state on a seeded sample of those cells, with per cell whether its upper bound was stable over the
    three runs and whether its traversability window was free of unstable cells."""
    from elevation_mapping_cupy_b200.parameter import core_parameter
    from elevation_mapping_cupy_b200 import workloads as wl
    g = load_golden("reference_gpu")
    p = core_parameter(256)
    em = _mk(p)
    worst = 0.0
    worst_trav = 0.0
    for f in range(5):
        pts, R, t = wl.lidar_cloud(0, f, n_rings=32, n_az=625, max_range=8.0)
        em.move_to(t, R)
        em.input_pointcloud(pts, ["x", "y", "z"], R, t, 0.02, 0.02)
        state, _ = em.get_state()
        assert g[f"state_racy_mean_{f}"] < 0.06
        cells = g[f"state_cells_{f}"]
        ref = g[f"state_vals_{f}"]
        ours = state.reshape(7, -1)[:, cells]
        # height / variance / validity / time: three runs of a racy kernel can still agree on a cell whose outcome is
        # order-dependent (e.g. outlier-inlier-outlier in input order looks the same forward and reversed), so a
        # handful of cells may legitimately differ: the bar is <= 1e-4 on all but at most 0.1 % of the compared cells
        lim = max(1, len(cells) // 1000)
        for li in (0, 1, 2, 4):
            d = np.abs(ours[li] - ref[li])
            bad = int((d > 1e-4).sum())
            assert bad <= lim, (f, li, bad, float(d.max()))
            worst = max(worst, float(np.sort(d)[-(bad + 1)]))
        # traversability (layer 3): the reference computes it with torch / cuDNN convolutions (traversability_filter.py:
        # 15-42, TF32 off); it depends on the dilated upper bound within a 13 x 13 window, so compare where no racy or
        # upper-bound-unstable cell lies in that window
        clean = g[f"state_clean_{f}"]
        if clean.any():
            dt = np.abs(ours[3] - ref[3])[clean]
            assert float(dt.max()) <= 1e-4, (f, "traversability vs cuDNN", float(dt.max()))
            worst_trav = max(worst_trav, float(dt.max()))
        # upper_bound: the reference's check-then-store (CK.py:230-233,253-256) loses updates, so a carved cell
        # holds SOME ray's height; the engine holds the true minimum: never above any reference outcome, and
        # is_upper_bound identical wherever the three reference runs agree with each other
        ub_stable = g[f"state_ub_stable_{f}"]
        assert int((ours[6][ub_stable] != ref[6][ub_stable]).sum()) <= lim
        carved = ub_stable & (ours[6] > 0.5) & (ref[6] > 0.5)
        assert int((ours[5][carved] > g[f"state_ub_min_{f}"][carved] + 1e-6).sum()) <= lim
        # (upper_bound of a cell fused by several points is the new_h of an ARBITRARY one of them in the reference,
        # CK.py:191; the engine takes the last in input order -- not comparable cell by cell)
        em.update_variance(); em.update_time()
    print("largest abs difference vs reference GPU kernels over the accepted order-independent cells:", worst,
          "; traversability vs the cuDNN path:", worst_trav)
