"""Generates tests/golden/*.npz.  Needs the reference libraries oracle/build_ref.py builds into oracle/_ref/ from the
reference source: the "ref_*" arrays and reference_*.npz come from the REFERENCE'S OWN kernel source
(custom_kernels.py strings compiled for the host by oracle/build_ref.py and driven in the order of
elevation_mapping.py:316-391); the "oracle_*" arrays from oracle/emap_oracle.c.

    python tests/golden/make_golden.py            # host build of the reference kernels
    python tests/golden/make_golden.py --gpu      # its nvcc build, run on a B200 -> reference_gpu.npz

Inputs are regenerated from seeds by elevation_mapping_cupy_b200/workloads.py, so only outputs are stored.
The reference kernel is racy (SURVEY 3.5); `racy` marks the cells whose outcome differs between executing the
points in input order, in reverse order and in a fixed random order -- parity is asserted outside that mask.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from elevation_mapping_cupy_b200 import workloads as wl          # noqa: E402
from elevation_mapping_cupy_b200.parameter import Parameter, core_parameter   # noqa: E402
from oracle import oracle as O                                   # noqa: E402


def index_case(seed):
    """reference test shape (test_elevation_mapping.py:51-61), default parameters, 202^2 map"""
    p = Parameter(); p.update()
    pts, R, t = wl.reference_test_cloud(seed, n=20000)
    if seed % 2:
        pts = (pts * np.float32(9.0) - np.float32(4.5)).astype(np.float32)
    rm = O.RefKernelMap(p, "default202")
    rm.input_pointcloud(pts.copy(), ["x", "y", "z"], R, t, 0, 0)
    idx, valid, inside = rm.last_point_record
    return dict(idx=idx, valid=valid, inside=inside)


def frames_case(cell_n=130, n_frames=4, tag="core130"):
    p = core_parameter(cell_n)
    om = O.OracleElevationMap(p)
    out = {}
    perm_rng = np.random.default_rng(99)
    for f in range(n_frames):
        pts, R, t = wl.lidar_cloud(0, f, n_rings=24, n_az=500, max_range=4.0)
        refs = []
        for order in ("fwd", "rev", "perm"):
            rm = O.RefKernelMap(p, tag)
            rm.elevation_map = om.elevation_map.copy(); rm.normal_map = om.normal_map.copy()
            rm.center = om.center.copy(); rm.additive_mean_error = om.additive_mean_error
            pp = pts if order == "fwd" else (pts[::-1].copy() if order == "rev" else pts[perm_rng.permutation(len(pts))])
            rm.move_to(t, R)
            rm.input_pointcloud(pp, ["x", "y", "z"], R, t, 0.02, 0.02)
            refs.append(rm)
        om.move_to(t, R)
        om.input_pointcloud(pts, ["x", "y", "z"], R, t, 0.02, 0.02)
        racy = np.zeros((cell_n, cell_n), bool)
        for li in (0, 1, 2, 4, 5, 6):
            for other in refs[1:]:
                racy |= np.abs(refs[0].elevation_map[li] - other.elevation_map[li]) > 1e-6
        out[f"ref_state_{f}"] = refs[0].elevation_map.copy()
        out[f"ref_normal_{f}"] = refs[0].normal_map.copy()
        out[f"racy_{f}"] = racy
        out[f"oracle_state_{f}"] = om.elevation_map.copy()
        out[f"oracle_normal_{f}"] = om.normal_map.copy()
        out[f"ref_point_idx_{f}"] = refs[0].last_point_record[0]
        om.update_variance(); om.update_time()
    return out


def sample_cells(rng, candidates, k, focus=None):
    """A fixed, seeded sample of up to k flat cell indices out of the True cells of `candidates`: two thirds from the
    cells that also lie in `focus` (those carrying data), the rest uniform; sorted."""
    cand = np.flatnonzero(candidates)
    picked = np.zeros(0, np.int64)
    if focus is not None:
        f = np.flatnonzero(candidates & focus)
        picked = rng.choice(f, min(len(f), 2 * k // 3), replace=False)
    rest = np.setdiff1d(cand, picked)
    picked = np.concatenate([picked, rng.choice(rest, min(len(rest), k - len(picked)), replace=False)])
    return np.sort(picked).astype(np.uint16 if candidates.size <= 1 << 16 else np.int32)


def drift_frames(n=5):
    """tests/test_oracle_cpu.py: LiDAR frames with an alternating 3 cm bias (non-zero mean error)"""
    out = []
    for f in range(n):
        pts, R, t = wl.lidar_cloud(0, f, n_rings=24, n_az=500, max_range=4.0)
        pts = pts.copy(); pts[:, 2] += np.float32(0.03 * (f % 2))
        out.append((pts, R, t))
    return out


FLAG_CASES = [
    dict(enable_edge_sharpen=False),
    dict(enable_visibility_cleanup=False),
    dict(enable_overlap_clearance=False, enable_drift_compensation=False),
    dict(max_ray_length=2.0, cleanup_step=0.01, cleanup_cos_thresh=0.5, wall_num_thresh=3, dilation_size=2,
         min_valid_distance=0.3, mahalanobis_thresh=1.0),
]


def reference_cpu_case():
    """tests/test_oracle_cpu.py: the reference's kernel source compiled for the host (oracle/_ref/libref_cpu_*.so).
    Exact comparisons are stored as digests, tolerance comparisons as a seeded sample of the compared cells."""
    import ctypes as C
    from helpers import digest
    from oracle import build_ref
    from oracle.configs import REF_CONFIGS, DRIFT_OVERRIDES
    out = {}
    srng = np.random.default_rng(130)
    W = 130
    _p = O._p
    # dilation / normal / min_filter
    p = core_parameter(W)
    rm = O.RefKernelMap(p, "core130")
    rng = np.random.default_rng(3)
    h = rng.standard_normal((W, W)).astype(np.float32)
    mask = (rng.random((W, W)) < 0.15).astype(np.float32)
    mask[:, :4] = (rng.random((W, 4)) < 0.6); mask[:, -4:] = (rng.random((W, 4)) < 0.6)
    ref = np.zeros((W, W), np.float32); dummy = np.zeros((W, W), np.float32)
    rm.lib.ref_dilation_filter(C.c_longlong(W * W), _p(h), _p(mask), _p(ref), _p(dummy), C.c_int(0))
    out["dilation_sha"] = digest(ref)
    rm.elevation_map[2] = mask
    rm.update_normal(ref)
    nz = rm.normal_map != 0
    out["normal_nonzero_sha"] = digest(nz)
    cells = sample_cells(srng, nz.any(0), 600)
    out["normal_cells"] = cells
    out["normal_vals"] = rm.normal_map.reshape(3, -1)[:, cells]
    m2 = np.ones((W, W), np.float32); m2[5:-5:4, 5:-5:4] = 0
    rm.elevation_map[0] = h; rm.elevation_map[2] = m2
    out["min_filter_sha"] = digest(np.nan_to_num(rm.min_filter(1)).astype(np.float32))
    # max_filter / robot_centric_elevation
    rng = np.random.default_rng(8)
    h = rng.standard_normal((W, W)).astype(np.float32)
    m = (rng.random((W, W)) < 0.3).astype(np.float32)
    cur_h, cur_m = h.copy(), m.copy()
    for _ in range(4):
        ih, im = cur_h.copy(), cur_m.copy()
        rm.lib.ref_max_filter(C.c_longlong(W * W), _p(ih), _p(im), _p(cur_h), _p(cur_m), C.c_int(0))
        if (cur_m > 0.5).all():
            break
    out["max_filter_sha"] = digest(np.where(cur_m > 0.5, cur_h, np.float32(-7)).astype(np.float32))
    R = np.array([[0.9, 0.1, -0.2], [0.0, 1.0, 0.1], [0.15, -0.12, 0.97]], np.float32)
    for thr, fn in ((True, rm.lib.ref_base_elevation_thr), (False, rm.lib.ref_base_elevation_raw)):
        o = h.copy()
        fn(C.c_longlong(W * W), _p(h), _p(m), _p(np.ascontiguousarray(R.reshape(9))), _p(o), C.c_int(0))
        if thr:
            out["rce_thr_sha"] = digest(o)
        else:
            cells = sample_cells(srng, np.ones((W, W), bool), 500)
            out["rce_raw_cells"] = cells
            out["rce_raw_vals"] = o.ravel()[cells]
            out["rce_raw_absmax"] = float(np.abs(o).max())
    # drift compensation: both reference runs start every frame from the oracle's state
    p = core_parameter(W, **DRIFT_OVERRIDES)
    rf = O.RefKernelMap(p, "drift130"); rr = O.RefKernelMap(p, "drift130")
    om = O.OracleElevationMap(p)
    for f, (pts, R, t) in enumerate(drift_frames()):
        for m_ in (rf, rr):
            m_.elevation_map = om.elevation_map.copy(); m_.normal_map = om.normal_map.copy(); m_.center = om.center.copy()
            m_.additive_mean_error = om.additive_mean_error
        for m_, pp in ((om, pts), (rf, pts), (rr, pts[::-1].copy())):
            m_.move_to(t, R); m_.input_pointcloud(pp, ["x", "y", "z"], R, t, 0.02, 0.02)
        racy = np.zeros((W, W), bool)
        for li in (0, 1, 2, 4, 5, 6):
            racy |= np.abs(rf.elevation_map[li] - rr.elevation_map[li]) > 1e-6
        cells = sample_cells(srng, ~racy, 300, focus=rf.elevation_map[2] > 0.5)
        out[f"drift_cells_{f}"] = cells
        out[f"drift_vals_{f}"] = rf.elevation_map[[0, 1, 2, 4, 5, 6]].reshape(6, -1)[:, cells]
        out[f"drift_mean_error_{f}"] = float(np.ravel(rf.mean_error)[0])
        om.update_variance(); om.update_time()
    # feature toggles and thresholds (one reference build per combination)
    for i, flags in enumerate(FLAG_CASES):
        p = core_parameter(W, **flags)
        om = O.OracleElevationMap(p)
        for f in range(3):
            pts, R, t = wl.lidar_cloud(0, f, n_rings=24, n_az=500, max_range=4.0)
            refs = []
            for order in (1, -1):
                rm_ = O.RefKernelMap(p, None)
                rm_.elevation_map = om.elevation_map.copy(); rm_.normal_map = om.normal_map.copy(); rm_.center = om.center.copy()
                rm_.additive_mean_error = om.additive_mean_error
                rm_.move_to(t, R); rm_.input_pointcloud(pts[::order].copy(), ["x", "y", "z"], R, t, 0.02, 0.02)
                refs.append(rm_)
            om.move_to(t, R); om.input_pointcloud(pts, ["x", "y", "z"], R, t, 0.02, 0.02)
            racy = np.zeros((W, W), bool)
            for li in (0, 1, 2, 4, 5, 6):
                racy |= np.abs(refs[0].elevation_map[li] - refs[1].elevation_map[li]) > 1e-6
            cells = sample_cells(srng, ~racy, 300, focus=refs[0].elevation_map[2] > 0.5)
            out[f"flags{i}_n_cmp_{f}"] = int((~racy).sum())
            out[f"flags{i}_cells_{f}"] = cells
            out[f"flags{i}_vals_{f}"] = refs[0].elevation_map[[0, 1, 2, 4, 5, 6]].reshape(6, -1)[:, cells]
            out[f"flags{i}_point_idx_sha_{f}"] = digest(refs[0].last_point_record[0])
            om.update_variance(); om.update_time()
    # semantic point-channel fusion (average, class_average, color)
    L = C.CDLL(build_ref.build(REF_CONFIGS["core130"], tag="core130", gpu=False))
    p = core_parameter(W)
    rng = np.random.default_rng(3)
    pts, R, t = wl.uniform_cloud(0, 1, n=6000, half_extent=2.3)
    idx, valid, inside, _ = O.point_index(p, pts, R, t)
    feats = np.stack([rng.random(len(pts), dtype=np.float32) * 3, rng.random(len(pts), dtype=np.float32),
                      rng.integers(0, 1 << 24, len(pts)).astype(np.uint32).view(np.float32)], 1)
    pall = np.ascontiguousarray(np.concatenate([np.stack([idx, valid, inside], 1).astype(np.float32), feats], 1))
    cnt = np.bincount(idx[(valid > 0) & (inside > 0)], minlength=W * W).astype(np.float32)
    cnt[rng.random(W * W) < 0.3] = 0
    new_el = np.zeros((7, W, W), np.float32); new_el[2] = cnt.reshape(W, W)
    fp = lambda a: a.ctypes.data_as(C.c_void_p)
    dummy = np.zeros(16, np.float32)
    sem_ref = np.zeros((3, W, W), np.float32)
    for frame in range(2):
        newmap = np.zeros((3, W, W), np.float32)
        for k, kind in enumerate(["average", "class_average"]):
            chan = np.array([3 + k], np.int32); lay = np.array([k], np.int32); dims = np.array([pall.shape[1], 1], np.int32)
            L.ref_sem_sum(C.c_longlong(len(pts)), fp(pall), fp(dummy), fp(dummy), fp(chan), fp(lay), fp(dims), fp(sem_ref), fp(newmap), 0)
            fn = L.ref_sem_average if kind == "average" else L.ref_sem_class_average
            fn(C.c_longlong(W * W), fp(newmap), fp(chan), fp(lay), fp(dims), fp(new_el), fp(sem_ref), 0)
        color_map = np.zeros((4, W, W), np.uint32)
        chan = np.array([5], np.int32); lay = np.array([2], np.int32); dims = np.array([pall.shape[1], 1], np.int32)
        L.ref_sem_add_color(C.c_longlong(len(pts)), fp(pall), fp(dummy), fp(dummy), fp(chan), fp(lay), fp(dims), fp(color_map), 0)
        L.ref_sem_color_average(C.c_longlong(W * W), fp(color_map), fp(chan), fp(lay), fp(dims), fp(sem_ref), 0)
        out[f"sem_color_sha_{frame}"] = digest(sem_ref[2].view(np.uint32))
        cells = sample_cells(srng, np.ones((W, W), bool), 500, focus=(sem_ref[0] != 0) | (sem_ref[1] != 0))
        out[f"sem_cells_{frame}"] = cells
        out[f"sem_vals_{frame}"] = sem_ref[:2].reshape(2, -1)[:, cells]
        out[f"sem_absmax_{frame}"] = np.abs(sem_ref[:2]).reshape(2, -1).max(1)
    return out


def reference_gpu_case():
    """tests/test_gpu_reference_kernels.py: the reference's own CUDA kernels (oracle/_ref/libref_gpu_*.so, driven by
    tests/ref_gpu.py) on a B200.  Exact comparisons are stored as digests, tolerance comparisons as a seeded sample of
    the compared cells."""
    import torch
    from ref_gpu import RefGpuMap
    from helpers import digest
    from elevation_mapping_cupy_b200.elevation_mapping import ElevationMap
    out = {}
    for tag, p, cloud in (("default202", Parameter(), "rand"), ("core1024", core_parameter(1024), "lidar")):
        p.update()
        rg = RefGpuMap(p, tag)
        if cloud == "rand":
            pts, R, t = wl.reference_test_cloud(3)
            pts = (pts * np.float32(9.0) - np.float32(4.5)).astype(np.float32)
        else:
            pts, R, t = wl.lidar_cloud(1, 2)
        wb = rg.input_pointcloud(pts, R, t, 0, 0).cpu().numpy()
        out[f"index_{tag}_sha"] = np.array([digest(wb[:, 0].astype(np.int32)), digest(wb[:, 1].astype(np.uint8)),
                                            digest(wb[:, 2].astype(np.uint8))])
    # 5 LiDAR frames on a 256^2 map; each frame starts every reference run from the engine's pre-frame state
    p = core_parameter(256)
    em = ElevationMap(p)
    refs = [RefGpuMap(p, "core256") for _ in range(3)]
    rng = np.random.default_rng(4)
    srng = np.random.default_rng(256)
    from scipy import ndimage
    for f in range(5):
        pts, R, t = wl.lidar_cloud(0, f, n_rings=32, n_az=625, max_range=8.0)
        em.move_to(t, R)
        st, nm = em.get_state()
        outs = []
        for k, rg in enumerate(refs):
            rg.set_state(st, nm, em.center)
            pp = pts if k == 0 else (pts[::-1].copy() if k == 1 else pts[rng.permutation(len(pts))])
            rg.input_pointcloud(pp, R, t, 0.02, 0.02)
            outs.append(rg.elevation_map.cpu().numpy())
        em.input_pointcloud(pts, ["x", "y", "z"], R, t, 0.02, 0.02)
        state, _ = em.get_state()
        racy = np.zeros((256, 256), bool)
        for li in (0, 1, 2, 4):
            for o in outs[1:]:
                racy |= np.abs(outs[0][li] - o[li]) > 1e-6
        ub_stable = ~racy
        for o in outs[1:]:
            ub_stable &= (np.abs(outs[0][5] - o[5]) <= 1e-6) & (outs[0][6] == o[6])
        ub_ok = ub_stable & (np.abs(state[5] - outs[0][5]) <= 1e-6) & (state[6] == outs[0][6])
        clean = ndimage.minimum_filter(ub_ok.astype(np.uint8), size=13, mode="constant", cval=0).astype(bool)
        clean[:3, :] = clean[-3:, :] = False; clean[:, :3] = clean[:, -3:] = False
        cells = np.union1d(sample_cells(srng, ~racy, 600, focus=outs[0][2] > 0.5), sample_cells(srng, clean, 150))
        out[f"state_racy_mean_{f}"] = float(racy.mean())
        out[f"state_cells_{f}"] = cells
        out[f"state_vals_{f}"] = outs[0].reshape(7, -1)[:, cells]
        out[f"state_ub_min_{f}"] = np.min([o[5].ravel()[cells] for o in outs], axis=0)
        out[f"state_ub_stable_{f}"] = ub_stable.ravel()[cells]
        out[f"state_clean_{f}"] = clean.ravel()[cells]
        em.update_variance(); em.update_time()
    return out


if __name__ == "__main__":
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpu", action="store_true", help="write reference_gpu.npz (needs a B200 and oracle/_ref/libref_gpu_*.so)")
    ap.add_argument("--out", default=HERE)
    args = ap.parse_args()
    sys.path.insert(0, os.path.dirname(HERE))
    if args.gpu:
        np.savez_compressed(os.path.join(args.out, "reference_gpu.npz"), **reference_gpu_case())
    else:
        for seed in (0, 1):
            np.savez_compressed(os.path.join(args.out, f"index_default202_seed{seed}.npz"), **index_case(seed))
        np.savez_compressed(os.path.join(args.out, "frames_core130.npz"), **frames_case())
        np.savez_compressed(os.path.join(args.out, "reference_cpu.npz"), **reference_cpu_case())
    for f in sorted(os.listdir(args.out)):
        print(f, os.path.getsize(os.path.join(args.out, f)))
