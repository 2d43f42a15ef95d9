#!/usr/bin/env python
"""bench.py -- Mpoints/s fused + map-update frames/s of the fusion path (BASELINE.json metric).

A "step" is one frame = one ElevationMap.input_pointcloud() call = everything in the reference's
update_map_with_kernel (elevation_mapping.py:316-391): error count -> drift -> Kalman fusion ->
ray-cast cleanup -> average -> overlap clear -> dilation -> traversability -> normals.

Workload at N=1 = BASELINE.json configs[1]: 1024x1024 grid, 0.04 m, 200k-point LiDAR-like cloud per
frame, ray-cast + overlap clear on (SURVEY.md 8(d) "B").  At N>1 (torchrun, one rank per GPU) the
workload is configs[2] generalised: one 200k-point sensor per GPU fused into a replicated grid with
an NCCL all-reduce of the per-cell partials (weak scaling: per-GPU work fixed).

Between timed frames, untimed: move_to (recentre on the sensor), update_variance, update_time (the
reference runs these from timers) and an L2 flush (a 512 MB memset) -- say so in `config`.
`value`: inputs resident in HBM, each frame timed with CUDA events on the launching stream.
`e2e`:   the same frames through the public API with pinned HOST buffers: H2D copy of the cloud and a
         D2H read of the frame statistics inside the timed region.
`--impl reference` times the reference's own kernel source (oracle/_ref, compiled for the host by
oracle/build_ref.py with OpenMP + atomics) on all host threads, on a bounded sample of the workload.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

# torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU legs (rank 0 only) must use every host core
if os.environ.get("RANK", "0") == "0":
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Mpoints/s fused + map-update frames/s (1024^2 grid, 200k-pt LiDAR frames, raycast+overlap-clear on)"
N_FRAME_POOL = 8          # distinct synthetic frames, cycled
PTS_PER_SENSOR = 200000


def workload_string(n_sensors):
    """One description for both arms (the driver compares the two `config.workload` strings)."""
    return ("1024x1024 grid, 0.04 m, %d x 200k-pt LiDAR-like frame(s) per step, raycast+overlap-clear on, "
            "drift compensation on (BASELINE configs[%d])" % (n_sensors, 1 if n_sensors == 1 else 2))


def use_all_host_threads():
    """All host cores for the oracle / reference-source OpenMP loops, whatever the launcher exported."""
    from oracle import oracle as O
    n = os.cpu_count() or 1
    L = O.lib()
    L.oracle_set_threads(int(n))
    return int(L.oracle_max_threads())


def make_frames(n_sensors, sensor, n_pool):
    from elevation_mapping_cupy_b200 import workloads as wl
    out = []
    for f in range(n_pool):
        pts, R, t = wl.lidar_cloud(1 if n_sensors == 1 else 2, f, sensor=sensor, n_sensors=n_sensors)
        out.append((pts, R, t))
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self, t_begin=None, t_end=None):
        """Summary of the samples taken in [t_begin, t_end] (epoch seconds; the GPU-busy part of the run)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        try:
            self.thr.join(timeout=2)
        except Exception:
            pass
        import datetime
        sm, mx, reasons, n_all = [], [], set(), 0
        for r in self.rows:
            try:
                n_all += 1
                ts = datetime.datetime.strptime(r[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                if t_begin is not None and not (t_begin - 0.02 <= ts <= t_end + 0.02):
                    continue
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_total": n_all,
                "window_s": None if t_begin is None else round(t_end - t_begin, 3)}


def cpu_baseline_port(param, frames, max_seconds=20.0):
    """The oracle (C restatement, all host threads) on a bounded sample of the same workload."""
    from oracle import oracle as O
    cores = use_all_host_threads()
    om = O.OracleElevationMap(param, nthreads=cores)
    npts, t_total, n = 0, 0.0, 0
    t_begin = time.perf_counter()
    for pts, R, t in frames:
        om.move_to(t, R)
        t0 = time.perf_counter()
        om.input_pointcloud(pts, ["x", "y", "z"], R, t, 0.02, 0.02)
        t_total += time.perf_counter() - t0
        om.update_variance(); om.update_time()
        npts += len(pts); n += 1
        if time.perf_counter() - t_begin > max_seconds:
            break
    return {"value": npts / t_total / 1e6, "unit": "Mpoints/s", "cores": int(cores), "kind": "port",
            "sample": f"{n} frames of the same 200k-pt workload, oracle/emap_oracle.c with OpenMP", "frames_per_s": n / t_total}


def run_reference_arm(args):
    """Reference arm: the reference's own kernel source (oracle/_ref) on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    from elevation_mapping_cupy_b200.parameter import core_parameter
    from oracle import oracle as O
    param = core_parameter(1024)
    try:
        rm = O.RefKernelMap(param, "core1024", parallel=True)
    except Exception as e:       # prebuilt library absent
        return {"impl": "reference", "unavailable": f"oracle/_ref not built: {e}"[:200]}
    cores = use_all_host_threads()
    n_sensors = max(1, args.gpus)
    # bounded sample: the CPU needs ~0.2-1 s per 200k-point frame and sensor, so the number of timed steps is capped
    # such that the whole arm ends within a few minutes at any --gpus N; `steps` / `warmup` in the line are the counts
    # actually run (the requested ones are kept as requested_steps / requested_warmup)
    n_warm = min(args.warmup, 3)
    n_steps = max(1, min(args.steps, 24 // n_sensors if n_sensors > 1 else 20))
    pools = [make_frames(n_sensors, s, 2) for s in range(n_sensors)]
    times = []
    for it in range(n_warm + n_steps):
        f = it % len(pools[0])
        rm.move_to(pools[0][f][2], pools[0][f][1])
        t0 = time.perf_counter()
        for s in range(n_sensors):                       # the reference fuses sensors sequentially
            pts, R, t = pools[s][f]
            rm.input_pointcloud(pts, ["x", "y", "z"], R, t, 0.02, 0.02)
        dt = time.perf_counter() - t0
        rm.update_variance(); rm.update_time()
        if it >= n_warm:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    val = n_sensors * PTS_PER_SENSOR / (ms * 1e-3) / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Mpoints/s", "frames_per_s": 1e3 / ms, "n_gpus": args.gpus,
            "steps": n_steps, "warmup": n_warm, "requested_steps": args.steps, "requested_warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(n_sensors), "frames_per_s": 1e3 / ms,
                       "points_per_step": n_sensors * PTS_PER_SENSOR},
            "cpu_baseline": {"value": val, "unit": "Mpoints/s", "cores": int(cores), "kind": "reference",
                             "sample": f"{n_steps} timed steps ({n_warm} warm-up) of {n_sensors} x 200k-pt frame(s); reference kernel source (custom_kernels.py) compiled for the "
                                       "host by oracle/build_ref.py, OpenMP + CAS atomics; traversability via torch CPU conv"},
            "e2e": {"value": val, "unit": "Mpoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    return line


def _state_digest(em):
    import hashlib
    state, normal = em.get_state()
    h = hashlib.sha256(); h.update(state.tobytes()); h.update(normal.tobytes())
    return h.digest(), state, normal


def check_sharded_parity(torch, dist, em, sh, frames, poses0, dev_pts, world, rank, between, frame):
    """One CHECKED sharded frame after the timed loops: every rank hashes its 7+3 planes (replicas must be
    bit-identical), and rank 0 replays the frame as a single-GPU `input_sensors` of the concatenated clouds from
    the same pre-frame state and compares all planes bit for bit.  Raises SystemExit(3) on a mismatch."""
    from elevation_mapping_cupy_b200 import workloads as wl
    from elevation_mapping_cupy_b200.elevation_mapping import ElevationMap
    f = 1
    between(f)
    torch.cuda.synchronize()
    pre_state, pre_normal = em.get_state()
    center = em.center.astype(np.float64)
    frame(f, dev_pts[f])
    torch.cuda.synchronize()
    dig, state, normal = _state_digest(em)
    t = torch.frombuffer(bytearray(dig), dtype=torch.uint8).cuda()
    allt = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(allt, t)
    replicas_equal = all(bool((x == allt[0]).all().item()) for x in allt)
    equals_single = None
    if rank == 0:
        import contextlib
        with contextlib.redirect_stdout(sys.stderr):
            em1 = ElevationMap(em.param, device=em.device)
        em1.set_state(pre_state, pre_normal, center)
        clouds, Rs, ts = [], [], []
        for s in range(world):
            if s == 0:
                pts, R, tt = frames[f]
            else:
                pts, R, tt = wl.lidar_cloud(2, f, sensor=s, n_sensors=world)
            clouds.append(pts); Rs.append(R); ts.append(tt)
        em1.input_sensors(clouds, Rs, ts, 0.02, 0.02)
        s1, n1 = em1.get_state()
        equals_single = bool(np.array_equal(s1, state, equal_nan=True) and np.array_equal(n1, normal, equal_nan=True))
        em1.close()
    flag = torch.tensor([1 if (replicas_equal and equals_single is not False) else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    out = {"replicas_equal": replicas_equal, "equals_single_gpu": equals_single, "transport": sh.mode,
           "checked": "frame %d of the pool: sha256 of the 7+3 planes all-gathered over %d ranks; rank 0 replays the frame on one GPU "
                      "(input_sensors of the %d concatenated clouds, same pre-frame state) and compares every plane bit for bit" % (f, world, world)}
    if int(flag.item()) != 1:
        if rank == 0:
            sys.stderr.write("PARITY FAILURE at N=%d: %s\n" % (world, json.dumps(out)))
        raise SystemExit(3)
    return out


def reference_gpu_leg(torch, em, param, frames, dev_pts, between, ms_ours, flush):
    """The reference's own CUDA kernels (its CUDA-C strings compiled by nvcc for sm_100a into oracle/_ref by
    oracle/build_ref.py, launched as CuPy would: 128-thread blocks, one element per thread) + torch/cuDNN for the
    traversability filter, on the same GPU, same frames, same pre-frame state, same L2 flush -- the bar SURVEY 2.2 names."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    try:
        from ref_gpu import RefGpuMap
        rg = RefGpuMap(param, "core1024")
    except Exception as e:
        return {"unavailable": str(e)[:160]}
    times = []
    for it in range(3 + 10):
        f = it % len(frames)
        pts, R, t = frames[f]
        between(f)
        st, nm = em.get_state()
        rg.set_state(st, nm, em.center)
        if flush is not None:
            flush.zero_()
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); rg.input_pointcloud(pts, R, t, 0.02, 0.02, points_dev=dev_pts[f]); e1.record(); torch.cuda.synchronize()
        if it >= 3:
            times.append(e0.elapsed_time(e1))
        em.input_pointcloud(dev_pts[f], ["x", "y", "z"], R, t, 0.02, 0.02)
    ms_ref = float(np.mean(times))
    return {"ms_per_frame": ms_ref, "mpoints_per_s": PTS_PER_SENSOR / (ms_ref * 1e-3) / 1e6, "speedup": ms_ref / ms_ours,
            "steps": len(times), "note": "reference kernel source (custom_kernels.py strings) built by nvcc for sm_100a + torch/cuDNN "
            "traversability, incl. its 2 host syncs per frame; device-resident cloud, cold L2, CUDA events"}


class _QuietStdout:
    """stdout must carry exactly ONE JSON line: park fd 1 on stderr while libraries (NCCL banner, plugin
    loader prints) are chatty, and give it back for the final print."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *a):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def main():
    with _QuietStdout():
        line = _main()
    if line is not None:
        print(json.dumps(line), flush=True)
    return 0


def _main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-flush", action="store_true", help="keep the map L2-resident between frames (reported separately)")
    ap.add_argument("--config", default="B", choices=["B", "D", "E"],
                    help="BASELINE.json configuration: B = configs[1]/[2] (default, the headline metric), D = configs[3], E = configs[4]")
    ap.add_argument("--no-graph", action="store_true", help="config E: launch the frames eagerly instead of replaying CUDA graphs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the map state after the last timed step (elevation_map.npy (7,W,W), normal_map.npy "
                         "(3,W,W), float32) to DIR, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.config != "B":
        ap.error("--dump-outputs is supported for --config B only")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    from elevation_mapping_cupy_b200.parameter import core_parameter
    from elevation_mapping_cupy_b200.elevation_mapping import ElevationMap

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world != args.gpus:
        raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local_rank)
    # one explicit stream for everything (library kernels, torch memsets, NCCL ordering, timing events)
    torch.cuda.set_stream(torch.cuda.Stream())
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    if args.config != "B":
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_configs
        fn = bench_configs.run_config_d if args.config == "D" else bench_configs.run_config_e
        line = fn(args, torch, dist, rank, local_rank, world, sampler if rank == 0 else None)
        if dist is not None:
            dist.destroy_process_group()
        return line
    param = core_parameter(1024)
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):      # stdout carries exactly one JSON line
        em = ElevationMap(param, device=local_rank)
    frames = make_frames(world, rank, N_FRAME_POOL)
    frames0 = frames if rank == 0 or world == 1 else None
    sh = None
    if world > 1:
        from elevation_mapping_cupy_b200.sharded import ShardedElevationMap
        sh = ShardedElevationMap(em, static_offsets=(rank * PTS_PER_SENSOR, world * PTS_PER_SENSOR))
        # every replica recentres on sensor 0's pose
        from elevation_mapping_cupy_b200 import workloads as wl
        poses0 = [wl.lidar_pose(f, 0, world) for f in range(N_FRAME_POOL)]
    else:
        poses0 = [(R, t) for (_, R, t) in frames]

    dev_pts = [torch.from_numpy(p).cuda() for p, _, _ in frames]
    pin_pts = [torch.from_numpy(p).pin_memory() for p, _, _ in frames]
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream()      # the side stream made current below
    assert stream.cuda_stream != 0
    if sh is None:
        em._check(em._L.emap_set_stream(em._h, stream.cuda_stream))

    def between(f):
        R0, t0 = poses0[f]
        em.move_to(t0, R0)
        em.update_variance(); em.update_time()
        if not args.no_flush:
            flush.zero_()

    def frame(f, pts):
        _, R, t = frames[f]
        if sh is None:
            em.input_pointcloud(pts, ["x", "y", "z"], R, t, 0.02, 0.02)
        else:
            sh.input_sensors([pts], [R], [t], 0.02, 0.02, device_ptrs=pts.is_cuda, overlap_z=float(poses0[f][1][2]))

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    export_buf = np.zeros((param.cell_n - 2, param.cell_n - 2), np.float32)

    def run(n_warm, n_steps, host, export=False):
        src = pin_pts if host else dev_pts
        for it in range(n_warm):
            f = it % N_FRAME_POOL
            between(f); frame(f, src[f])
            if host:
                em.get_frame_stats()
            if export:
                em.get_map_with_name_ref("elevation", export_buf)
        barrier()
        evs, wall = [], 0.0
        launches0 = em.launch_count()
        for it in range(n_steps):
            f = (n_warm + it) % N_FRAME_POOL
            between(f)
            if host:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                frame(f, src[f])
                em.get_frame_stats()                     # D2H read of the step's result (syncs)
                if export:
                    em.get_map_with_name_ref("elevation", export_buf)     # EM.py:720-775: the layer a consumer reads
                wall += time.perf_counter() - t0
            else:
                e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                e0.record(stream); frame(f, src[f]); e1.record(stream)
                evs.append((e0, e1))
        launches = em.launch_count() - launches0
        barrier()
        if host:
            ms = 1e3 * wall / n_steps
        else:
            ms = sum(a.elapsed_time(b) for a, b in evs) / n_steps
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), launches

    # ---- device-resident arm (value); clocks are sampled from before the warm-up to the end of the e2e arm (the
    # sampler was started before the frames were built: nvidia-smi needs ~1 s to print its first row) and the
    # summary keeps the rows stamped inside that GPU-busy window
    t_busy0 = time.time()
    ms, launches = run(args.warmup, args.steps, host=False)
    if args.dump_outputs and rank == 0:
        # what a caller of the timed path receives after its last step: the fused map layers and the normals
        state, normal = em.get_state()
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "elevation_map.npy"), state)
        np.save(os.path.join(args.dump_outputs, "normal_map.npy"), normal)
    # launches inside the timed frames only (exclude move_to / ticks): count one frame precisely
    between(0); torch.cuda.synchronize(); l0 = em.launch_count(); frame(0, dev_pts[0]); torch.cuda.synchronize()
    launches_per_frame = em.launch_count() - l0

    # ---- per-stage device times (CUDA events inside the library, same stream) for the roofline
    em.enable_stage_timing(True)
    stage = np.zeros(8)
    n_st = min(20, max(5, args.steps // 5))
    for it in range(n_st):
        f = it % N_FRAME_POOL
        between(f); frame(f, dev_pts[f]); torch.cuda.synchronize()
        stage += em.stage_ms()
    stage /= n_st
    em.enable_stage_timing(False)
    em._check(em._L.emap_set_ray_counting(em._h, 1))
    between(0); frame(0, dev_pts[0]); st = em.get_frame_stats()
    em._check(em._L.emap_set_ray_counting(em._h, 0))

    # ---- end-to-end arm: pinned host buffers through the public API, stats read back every step
    ms_e2e, _ = run(max(3, args.warmup // 2), args.steps, host=True)
    # ---- the same with the caller-visible product crossing PCIe too: one exported layer per frame
    ms_e2e_x, _ = run(3, max(10, args.steps // 2), host=True, export=True)
    t_busy1 = time.time()
    clocks = sampler.stop(t_busy0, t_busy1) if rank == 0 else None

    parity_n = check_sharded_parity(torch, dist, em, sh, frames, poses0, dev_pts, world, rank, between, frame) if sh is not None else None
    ref_gpu = reference_gpu_leg(torch, em, param, frames, dev_pts, between, ms, flush if not args.no_flush else None) if sh is None else None

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return None

    n_total = world * PTS_PER_SENSOR
    value = n_total / (ms * 1e-3) / 1e6
    e2e = n_total / (ms_e2e * 1e-3) / 1e6
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    C = param.cell_n ** 2
    names = ["index+error", "drift", "fusion", "record", "raycast", "finalize", "post(dilate+cnn+normal)"]
    dom = int(np.argmax(stage[:7]))
    # algorithmic bytes per launch of each stage (DESIGN.md "bytes per unit")
    N = PTS_PER_SENSOR
    NV = int(st.n_valid_points)
    # compulsory bytes per launch with the layout of DESIGN.md section 3 (each input once, each output once)
    alg = {"index+error": 12 * N + 20 * N + 32 * NV + 16 * NV, "drift": 64, "fusion": 20 * N + 12 * NV + 28 * NV,
           "record": 28 * C + 8 * C, "raycast": 32 * NV + 8 * C, "finalize": 24 * C + 24 * C + 12 * C,
           "post(dilate+cnn+normal)": 12 * C + 20 * C}
    dom_name = names[dom]
    ach = alg[dom_name] / (stage[dom] * 1e-3) / 1e9 if stage[dom] > 0 else 0.0
    frame_bytes = 24 * N * world + 80 * C
    traffic = None          # dram__bytes_read+write of the dominant kernel per launch, from the committed ncu capture
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")))
        if tr.get("kernel") == dom_name:
            traffic = tr["dram_bytes_per_launch"]
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": dom_name, "achieved": ach, "peak": hbm, "unit": "GB/s",
                "frac": ach / hbm, "traffic": traffic, "peak_source": peak_src,
                "kernel_ms": float(stage[dom]), "kernel_share_of_frame": float(stage[dom] / max(stage[7], 1e-9)),
                "frame_algorithmic_bytes": frame_bytes,
                "frame_achieved_gbs": frame_bytes / (ms * 1e-3) / 1e9, "frame_frac": frame_bytes / (ms * 1e-3) / 1e9 / hbm,
                "stage_ms": {n: float(v) for n, v in zip(names + ["total"], stage)}}
    cpu = None
    if not args.no_cpu_baseline:
        cpu = cpu_baseline_port(param, frames0[:4])
    line = {"metric": METRIC, "value": value, "unit": "Mpoints/s", "frames_per_s": 1e3 / ms, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(world),
                       "frames_per_s": 1e3 / ms, "points_per_step": n_total,
                       "parallelism": "1 GPU" if world == 1 else (
                           f"{world} sensor shards, replicated grid, " + (
                               "per-cell reductions as NVLink multicast multimem.red inside the frame kernels (no NCCL call in the frame)"
                               if sh.mode == "multicast" else "NCCL integer all-reduce x3 per frame")),
                       "transport": "none" if sh is None else sh.mode,
                       "l2": "flushed between timed frames (512 MB memset, untimed)" if not args.no_flush else "warm (no flush)",
                       "untimed_between_frames": "move_to, update_variance, update_time",
                       "ray_steps_per_frame": int(st.ray_steps), "ray_cell_visits_per_frame": int(st.ray_visits),
                       "valid_points_per_frame": int(st.n_valid_points)},
            "e2e": {"value": e2e, "unit": "Mpoints/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": int(PTS_PER_SENSOR * 12),
                    "d2h_bytes_per_step": 72, "note": "pinned host cloud -> emap_input_pointcloud (H2D inside), frame stats read back",
                    "with_layer_export": {"value": n_total / (ms_e2e_x * 1e-3) / 1e6, "unit": "Mpoints/s", "ms_per_step": ms_e2e_x,
                                          "d2h_bytes_per_step": 72 + int(export_buf.nbytes),
                                          "note": "as above + get_map_with_name_ref('elevation') into host memory every frame"}},
            "parity_n": parity_n, "reference_gpu": ref_gpu,
            "gpu_launches": int(launches_per_frame * args.steps), "gpu_launches_per_frame": int(launches_per_frame),
            "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu}
    if dist is not None:
        dist.destroy_process_group()
    return line


if __name__ == "__main__":
    sys.exit(main())
