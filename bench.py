#!/usr/bin/env python
"""bench.py — measures the two hot paths on BASELINE.json's configurations.

    python bench.py --gpus N --steps K --warmup W            (this repo's CUDA path)
    python bench.py --impl reference --gpus N --steps K ...  (CPU reference arm: the oracle port)

Primary line (ONE JSON line on rank 0): point-to-plane ICP, 2M-point synthetic clouds,
30 iterations, r = 0.05 (BASELINE config 2).  A *step* is one 30-iteration registration.
  value   = ICP iterations/s with the clouds resident in HBM (iteration loop only; the
            search-index build is reported separately and is part of `e2e`)
  e2e     = the same metric through the C-ABI host-buffer entry point
            o3db_icp_point_to_plane_host (H2D of the clouds, index build, 30 iterations,
            final evaluation and D2H of the result inside the timed region)
The same line carries a "tsdf" object: VoxelBlockGrid TSDF integration of a synthetic
640x480 depth(+colour) sequence, 8 mm voxels, 16^3 blocks (BASELINE config 3), frames/s.

N > 1 (torchrun, one rank per GPU): weak scaling.  ICP: every rank owns a 2M-point shard of
the source, the target is replicated, one 30-double NCCL all-reduce per iteration
(value = N x 2M-point iteration equivalents / s).  TSDF: frames round-robin over N
independent volumes, no collective.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ICP_POINTS = 2_000_000
ICP_ITERS = 30
ICP_RADIUS = 0.05
TSDF_FRAMES = 1000
VOXEL, RES, TRUNC_MULT, DSCALE, DMAX = 0.008, 16, 8.0, 1000.0, 3.0
HBM_FALLBACK_GBS = 6650.0


def measured_hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel):
    """dram read+write bytes per launch from the committed ncu --set full summary, or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f).get(kernel)
    except Exception:
        return None


def icp_algorithmic_bytes(n, m):
    """SURVEY.md §8(d): compulsory HBM bytes of one ICP iteration."""
    h = min(max(m // 32, 1), 2 ** 25)
    return 12 * n + 12 * n + 12 * m + 12 * m + 4 * m + 4 * (h + 1) + 4 * n


def tsdf_algorithmic_bytes(blocks, color, width=640, height=480):
    """SURVEY.md §8(d): compulsory HBM bytes of one integrated frame."""
    s_vox = 12 if color else 6
    touch = (width // 4) * (height // 4) * 2 + 4 * (width // 4) * (height // 4) * 12
    return blocks * 4096 * 2 * s_vox + width * height * 2 + (width * height * 3 if color else 0) + blocks * 16 + touch


DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLE_BLOCKS = 128


def volume_outputs(L, v, stream, torch, prefix, color):
    """What a caller of the TSDF path receives: the key of every active block (sorted, since the hash map's slot order
    depends on insertion timing) and tsdf / weight (/ colour) of a fixed, seeded sample of those blocks."""
    from open3d_b200.t._libshim import device_view
    torch.cuda.synchronize()
    size = L.check(L.lib.o3db_vbg_size(v, stream))
    cap = L.lib.o3db_vbg_capacity(v)
    idx = torch.empty(size, dtype=torch.int32, device="cuda")
    L.check(L.lib.o3db_vbg_active_indices(v, idx.data_ptr(), size, stream))
    idx = idx.long()
    keys = device_view(L.lib.o3db_vbg_key_buffer(v), (cap, 3), torch.int32)[idx].cpu().numpy()
    order = np.lexsort((keys[:, 2], keys[:, 1], keys[:, 0]))
    pick = np.sort(np.random.default_rng(0).choice(size, min(size, DUMP_SAMPLE_BLOCKS), replace=False))
    slots = idx[torch.from_numpy(order[pick]).cuda()]
    vox = RES ** 3
    out = {f"{prefix}_block_keys": keys[order].astype(np.float64),
           f"{prefix}_sample_block_keys": keys[order[pick]].astype(np.float64),
           f"{prefix}_sample_tsdf": device_view(L.lib.o3db_vbg_tsdf_buffer(v), (cap, vox), torch.float32)[slots],
           f"{prefix}_sample_weight": device_view(L.lib.o3db_vbg_weight_buffer(v), (cap, vox), torch.uint16)
           .view(torch.int16)[slots].int().bitwise_and(0xFFFF).float()}
    if color:
        out[f"{prefix}_sample_color"] = device_view(L.lib.o3db_vbg_color_buffer(v), (cap, vox, 3), torch.uint16) \
            .view(torch.int16)[slots].int().bitwise_and(0xFFFF).float()
    return out


def write_outputs(dirname, arrays):
    """--dump-outputs: one DIR/<name>.npy per array; doubles and integers as float64, everything else as float32."""
    os.makedirs(dirname, exist_ok=True)
    conv = {}
    for name, a in arrays.items():
        a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
        exact64 = a.dtype == np.float64 or (a.dtype.kind in "iu" and a.dtype.itemsize > 2)
        conv[name] = np.ascontiguousarray(a, np.float64 if exact64 else np.float32)
    total = sum(a.nbytes for a in conv.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    for name, a in conv.items():
        np.save(os.path.join(dirname, f"{name}.npy"), a)


class ClockSampler:
    """Samples SM clocks / throttle reasons during the timed region (B200_PROFILING.md): NVML in-process
    every 5 ms (the timed region is tens of milliseconds), nvidia-smi as a fallback."""

    def __init__(self, index=0):
        self.index = index
        self.rows = []   # (sm_mhz, sm_max_mhz, power_w, reasons_bitmask)
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        sm = n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self._h, n.NVML_CLOCK_SM)
        pw = n.nvmlDeviceGetPowerUsage(self._h) / 1000.0
        rs = n.nvmlDeviceGetCurrentClocksEventReasons(self._h) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") \
            else n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        self.rows.append((float(sm), float(mx), pw, int(rs)))

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout
        p = [x.strip() for x in out.strip().split(",")]
        if len(p) >= 7:
            bits = 0
            for i, b in enumerate((0x8, 0x40, 0x20, 0x4)):   # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
                if p[3 + i].lower().startswith("active"):
                    bits |= b
            self.rows.append((float(p[0]), float(p[1]), float(p[2]), bits))

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop.wait(0.005 if self._nvml is not None else 0.2)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(r[0] for r in self.rows)
        bits = 0
        for r in self.rows:
            bits |= r[3]
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        reasons = [n for b, n in names.items() if bits & b]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.rows[0][1], "reasons": reasons, "samples": len(self.rows),
                "power_w_max": max(r[2] for r in self.rows), "source": "nvml" if self._nvml is not None else "nvidia-smi"}


# ----------------------------------------------------------------------------------------------
# reference arm (CPU): the oracle port, timed on the host cores
# ----------------------------------------------------------------------------------------------

_CPU_THREADS = None


def use_all_host_cores():
    """The CPU legs run on the host's cores whatever OMP_NUM_THREADS the launcher exported (torchrun sets it
    to 1 for its workers — round 1's N>=2 reference lines were timed on one thread because of it).  "All
    cores" is not always "all hardware threads": with SMT siblings or a cgroup quota below the affinity mask
    an OpenMP team that large runs several times SLOWER.  So the candidates (every hardware thread the cgroup
    grants; one thread per physical core) are timed once on a small ICP problem and the fastest is used for
    every CPU leg of this process — the reference gets its best configuration."""
    global _CPU_THREADS
    import oracle
    if _CPU_THREADS is None:
        from tests.synth import make_icp_pair
        cands = oracle.thread_candidates()
        best = (None, 0.0)
        if len(cands) > 1:
            src, tgt, nrm, _ = make_icp_pair(300_000, seed=5)
            for t in cands:
                oracle.set_num_threads(t)
                rate = 0.0
                for _ in range(2):
                    r = oracle.icp_p2plane(src, tgt, nrm, ICP_RADIUS, max_iteration=2, relative_fitness=0,
                                           relative_rmse=0, accumulate_f64=False)
                    rate = max(rate, 2 / r.loop_seconds)
                if rate > best[1]:
                    best = (t, rate)
        _CPU_THREADS = best[0] or cands[0]
    return oracle.set_num_threads(_CPU_THREADS)


def cpu_icp_baseline(src, tgt, nrm, iters, reps=5):
    """ICP iterations/s of the CPU restatement on all host threads (loop only, like `value`):
    one warm-up run, then the MEDIAN of `reps` repetitions (BASELINE.md §3).  Returns (median, last result, rates)."""
    import oracle
    use_all_host_cores()
    rates, r = [], None
    for k in range(reps + 1):
        r = oracle.icp_p2plane(src, tgt, nrm, ICP_RADIUS, max_iteration=iters, relative_fitness=0, relative_rmse=0,
                               accumulate_f64=False)
        if k > 0:
            rates.append(iters / r.loop_seconds)
    return float(np.median(rates)), r, rates


def cpu_tsdf_baseline(frames, color):
    """frames/s of the CPU restatement of Model::Integrate on all host threads."""
    import oracle
    from tests.synth import PRIMESENSE_K
    cap = 60000
    keys = np.zeros((cap, 3), np.int32)
    tsdf = np.zeros((cap, RES ** 3), np.float32)
    wt = np.zeros((cap, RES ** 3), np.uint16)
    colbuf = np.zeros((cap, RES ** 3, 3), np.uint16) if color else None
    size = 0
    t0 = time.perf_counter()
    for (E, depth, col) in frames:
        want = oracle.depth_touch(depth, PRIMESENSE_K, E, RES, VOXEL, VOXEL * TRUNC_MULT, DSCALE, DMAX, 4)
        bi, _, size, _ = oracle.hashmap_activate(keys, size, want)
        oracle.tsdf_integrate(depth, col if color else None, bi, keys, tsdf, wt, colbuf, PRIMESENSE_K, PRIMESENSE_K, E,
                              RES, VOXEL, VOXEL * TRUNC_MULT, DSCALE, DMAX)
    return len(frames) / (time.perf_counter() - t0)


def _ref_lib():
    """oracle/_ref/libo3dref.so: the reference's own VoxelBlockGridCPU.cpp / VoxelBlockGridImpl.h compiled unmodified
    (oracle/ref_shim/ref_shim_vbg.cpp; ParallelFor on OpenMP).  None if it was not built (no /root/reference)."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle", "_ref", "libo3dref.so")
    if not os.path.exists(path):
        return None
    try:
        L = C.CDLL(path)
        L.ref_depth_touch.restype = C.c_int64
        L.ref_depth_touch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_float,
                                      C.c_float, C.c_float, C.c_float, C.c_int, C.c_void_p, C.c_int64]
        L.ref_integrate.restype = None
        L.ref_integrate.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p,
                                    C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_int, C.c_float, C.c_float, C.c_float, C.c_float]
        L.ref_num_threads.restype = C.c_int
        return L
    except (OSError, AttributeError):
        return None


def cpu_tsdf_reference(frames, color, R):
    """frames/s of the REFERENCE's DepthTouchCPU + IntegrateCPU (compiled from /root/reference) on all host threads;
    HashMap::Activate in between is the oracle's (upstream's is a TBB container, absent here)."""
    import oracle
    from tests.synth import PRIMESENSE_K
    cap = 60000
    keys = np.zeros((cap, 3), np.int32)
    tsdf = np.zeros((cap, RES ** 3), np.float32)
    wt = np.zeros((cap, RES ** 3), np.uint16)
    colbuf = np.zeros((cap, RES ** 3, 3), np.uint16) if color else None
    K9 = np.ascontiguousarray(np.asarray(PRIMESENSE_K, np.float64).reshape(9))
    touched = np.zeros((76800, 3), np.int32)
    size = 0
    t0 = time.perf_counter()
    for (E, depth, col) in frames:
        Ef = np.ascontiguousarray(np.asarray(E, np.float64).reshape(16))
        n = R.ref_depth_touch(depth.ctypes.data, 0, 480, 640, K9.ctypes.data, Ef.ctypes.data, RES, VOXEL,
                              VOXEL * TRUNC_MULT, DSCALE, DMAX, 4, touched.ctypes.data, len(touched))
        bi, _, size, _ = oracle.hashmap_activate(keys, size, touched[:n])
        bi = np.ascontiguousarray(bi, np.int32)
        R.ref_integrate(depth.ctypes.data, col.ctypes.data if color else None, 0, 480, 640, bi.ctypes.data, len(bi),
                        keys.ctypes.data, cap, tsdf.ctypes.data, wt.ctypes.data,
                        colbuf.ctypes.data if color else None, K9.ctypes.data, K9.ctypes.data, Ef.ctypes.data, RES,
                        VOXEL, VOXEL * TRUNC_MULT, DSCALE, DMAX)
    return len(frames) / (time.perf_counter() - t0)


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path cannot be built here
    (Eigen/TBB/nanoflann/stdgpu are download-time dependencies, SURVEY.md §8c), so this arm
    times the oracle port on all host threads.  Each step is a bounded sample of the workload:
    2 ICP iterations on the full 2M-point clouds; `value` is the MEDIAN of the per-step rates
    (one untimed full-size warm-up step first)."""
    if rank != 0:
        return
    if args.metric == "tsdf":
        return run_reference_tsdf(args)
    import oracle
    from tests.synth import make_icp_pair
    cores = use_all_host_cores()
    sample_iters = 2
    src, tgt, nrm, _ = make_icp_pair(ICP_POINTS, seed=2)
    for _ in range(max(args.warmup, 1)):
        oracle.icp_p2plane(src, tgt, nrm, ICP_RADIUS, max_iteration=1, relative_fitness=0, relative_rmse=0,
                           accumulate_f64=False)
    t0 = time.perf_counter()
    rates = []
    for _ in range(args.steps):
        r = oracle.icp_p2plane(src, tgt, nrm, ICP_RADIUS, max_iteration=sample_iters, relative_fitness=0,
                               relative_rmse=0, accumulate_f64=False)
        rates.append(sample_iters / r.loop_seconds)
    wall = time.perf_counter() - t0
    value = float(np.median(rates))
    sample = (f"{sample_iters} iterations on the full 2M-point clouds per step (loop time only, f32 accumulation); "
              f"median of {len(rates)} steps, min {min(rates):.1f} max {max(rates):.1f}")
    line = {"impl": "reference", "metric": "icp_iters_per_sec_2M_pts", "value": value, "unit": "iters/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": icp_config(args.gpus),
            "cpu_baseline": {"value": value, "unit": "iters/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def tsdf_cpu_frames(n_sample, F=TSDF_FRAMES):
    """A bounded sample of the config-3 trajectory for the CPU legs: (extrinsic, depth, colour) numpy triples."""
    import oracle
    from tests.synth import camera_pose, render_depth
    idx = list(range(0, F, max(1, F // n_sample)))[:n_sample]
    frames = []
    for i in idx:
        T = camera_pose(i, n_frames=F)
        d, c = render_depth(T, with_color=True)
        frames.append((oracle.inverse_transformation(T), d.numpy(), c.numpy()))
    return frames


def cpu_tsdf_best(frames, reps=5):
    """frames/s of the CPU TSDF path on all host threads, for depth-only and depth+colour: the FASTER of the
    reference's own DepthTouchCPU + IntegrateCPU (oracle/_ref, `kind: reference`) and the OpenMP port
    (`kind: port`) is the baseline, the other is kept beside it.  One warm-up + median of `reps` repetitions."""
    import oracle
    cores = use_all_host_cores()

    def med(fn):
        fn()
        return float(np.median([fn() for _ in range(reps)]))

    port = {c: med(lambda c=c: cpu_tsdf_baseline(frames, c)) for c in (False, True)}
    ref = None
    R = None
    try:
        R = _ref_lib()
        if R is not None:
            cpu_tsdf_reference(frames[:1], False, R)       # must not take the bench down
            ref = {c: med(lambda c=c: cpu_tsdf_reference(frames, c, R)) for c in (False, True)}
    except Exception as e:                                # noqa: BLE001
        print(f"[bench] reference-compiled TSDF baseline unavailable: {e}", file=sys.stderr)
        ref = None
    use_ref = ref is not None and ref[False] >= port[False]
    best = ref if use_ref else port
    out = {"value": best[False], "value_with_color": best[True], "unit": "frames/s", "cores": cores,
           "kind": "reference" if use_ref else "port",
           "sample": f"{len(frames)} frames spread over the trajectory (DepthTouch + HashMap::Activate + Integrate), "
                     f"median of {reps} repetitions after a warm-up; the faster of the reference-compiled kernels "
                     "(oracle/_ref: VoxelBlockGridCPU.cpp unmodified, OpenMP ParallelFor stand-in for TBB) and the "
                     "OpenMP port is reported",
           "port_value": port[False], "port_value_with_color": port[True]}
    if ref is not None:
        out["reference_compiled_value"] = ref[False]
        out["reference_compiled_value_with_color"] = ref[True]
    return out


def tsdf_config(world, F=TSDF_FRAMES):
    return {"workload": "voxel_block_grid_tsdf_integrate", "frames": F, "image": "640x480 u16 depth (+u8 colour)",
            "voxel_size": VOXEL, "block_resolution": RES, "trunc_voxel_multiplier": TRUNC_MULT,
            "initial_block_capacity": 40000, "baseline_config": "configs[2]",
            "l2_policy": "each frame touches a different part of a multi-GB volume; inputs larger than L2 over the sequence",
            "parallelism": f"frames round-robin over {world} independent volumes" if world > 1 else "single GPU"}


def run_reference_tsdf(args):
    """--impl reference --metric tsdf: the CPU TSDF path (see cpu_tsdf_best) on a bounded sample per step."""
    frames = tsdf_cpu_frames(12, args.tsdf_frames)
    t0 = time.perf_counter()
    cpu = cpu_tsdf_best(frames, reps=max(args.steps, 5))
    wall = time.perf_counter() - t0
    line = {"impl": "reference", "metric": "tsdf_frames_per_sec_640x480", "value": cpu["value"], "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": tsdf_config(args.gpus, args.tsdf_frames), "cpu_baseline": cpu,
            "e2e": {"value": cpu["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def icp_config(n_gpus):
    return {"workload": "point_to_plane_icp", "points_source_per_gpu": ICP_POINTS, "points_target": ICP_POINTS,
            "iterations_per_step": ICP_ITERS, "max_correspondence_distance": ICP_RADIUS, "voxel_size": 0.02,
            "baseline_config": "configs[1]: PointToPlane ICP, 2M-pt synthetic clouds, 30 iters, voxel_size=0.02",
            "note": "clouds are generated on a jittered 2 cm lattice (already voxel-size 0.02, down-sample = identity)",
            "l2_policy": "L2 flushed (256 MiB write) before every timed step; working set ~= L2 size",
            "parallelism": f"source-sharded x{n_gpus}, target replicated, 30-double all-reduce per iteration"
            if n_gpus > 1 else "single GPU"}


# ----------------------------------------------------------------------------------------------
# this repo's arm
# ----------------------------------------------------------------------------------------------

def bench_config3(args, rank, world, comm, torch, barrier, max_over_ranks):
    """BASELINE configs[3]: MultiScaleICP with TransformationEstimationForColoredICP, 3 scales, a 5M-point pair; with N
    ranks the source of every level is split by rows, one 30-double exchange per iteration (SURVEY 8e).  One run,
    through the public API (open3d_b200.t.pipelines.registration.multi_scale_icp)."""
    import open3d_b200 as o3d
    from tests.synth import make_colors, make_icp_pair
    reg = o3d.t.pipelines.registration
    n = int(args.config3_points)
    src, tgt, nrm, T_gt = make_icp_pair(n, seed=11)
    sc = make_colors((np.c_[src.astype(np.float64), np.ones(len(src))] @ T_gt.T)[:, :3], 1)
    tc = make_colors(tgt, 1)
    s = o3d.t.geometry.PointCloud(src).set_point_colors(sc)
    t = o3d.t.geometry.PointCloud(tgt).set_point_normals(nrm).set_point_colors(tc)
    voxels, radii, iters = [0.08, 0.04, 0.02], [0.16, 0.08, 0.05], [20, 15, 10]
    crits = [reg.ICPConvergenceCriteria(0, 0, k) for k in iters]
    est = reg.TransformationEstimationForColoredICP()
    levels = []
    runs = []
    for rep in range(2):                      # first run warms allocator pools / NCCL / IPC mappings
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        res = reg.multi_scale_icp(s, t, voxels, crits, radii, np.eye(4), est, None, comm)
        torch.cuda.synchronize()
        runs.append(max_over_ranks(time.perf_counter() - t0))
    total_iters = int(res.num_iterations)
    return {"workload": "multi-scale ColoredICP, 3 scales (voxel 0.08 / 0.04 / 0.02, radius 0.16 / 0.08 / 0.05, "
                        f"{iters} iterations), {len(src)} source x {len(tgt)} target points, source rows split over "
                        f"{world} GPU(s), pyramid + colour gradients built inside the call",
            "baseline_config": "configs[3]", "n_gpus": world, "seconds_total": runs[-1], "seconds_first_run": runs[0],
            "iterations": total_iters, "iters_per_sec_end_to_end": total_iters / runs[-1],
            "fitness": float(res.fitness), "inlier_rmse": float(res.inlier_rmse),
            "transformation_error_vs_ground_truth": float(np.abs(np.asarray(res.transformation) - T_gt).max()),
            "timing": "wall clock around multi_scale_icp (voxel pyramid, colour gradients, index builds, all iterations, "
                      "final evaluation), max over ranks"}


def main():
    # NCCL announces its version on stdout at VERSION level; keep stdout to the one JSON line
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--metric", default="icp", choices=["icp", "tsdf"],
                    help="icp (default): the primary line, BASELINE configs[1], with the TSDF numbers in a nested object; "
                         "tsdf: the same one-line schema with BASELINE configs[2] (TSDF frames/s) as the top-level metric")
    ap.add_argument("--skip-tsdf", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--tsdf-frames", type=int, default=TSDF_FRAMES)
    ap.add_argument("--cell-scale", type=float, default=0.0)
    ap.add_argument("--config3", action="store_true",
                    help="also run BASELINE configs[3] once (multi-scale ColoredICP, 3 scales, 5M points, source split over the "
                         "ranks); always on for N > 1")
    ap.add_argument("--config3-points", type=int, default=5_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step of each timed path returned to its caller "
                         "as DIR/<name>.npy (the inputs are seeded: two builds can be compared output for output)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from open3d_b200 import _lib as L
    from tests.synth import PRIMESENSE_K, camera_pose, make_icp_pair, render_depth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: open3d_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    comm = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        from open3d_b200.distributed import Communicator
        comm = Communicator(rank, world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    stream = int(torch.cuda.current_stream().cuda_stream)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def flush_l2():
        flush_buf.fill_(1)

    peak, peak_src = measured_hbm_peak()

    # ------------------------------------------------------------------ ICP
    src, tgt, nrm, T_gt = make_icp_pair(ICP_POINTS, seed=2)
    if world > 1:   # this rank's shard: an independent sampling of the same moved surface
        src = make_icp_pair(ICP_POINTS, seed=2 + 7919 * rank)[0]
    n, m = len(src), len(tgt)
    d_src, d_tgt, d_nrm = (torch.from_numpy(a).cuda() for a in (src, tgt, nrm))
    opt = L.IcpOptions()
    opt.max_correspondence_distance = ICP_RADIUS
    opt.max_iteration = ICP_ITERS
    opt.relative_fitness = opt.relative_rmse = 0.0          # all 30 iterations run (SURVEY §8d config 2)
    opt.kernel = L.RobustKernel(0, 1.0, 1.0)
    opt.cell_scale = args.cell_scale
    T0 = np.eye(4)
    h = C.c_void_p()
    ev = lambda: torch.cuda.Event(enable_timing=True)
    e0, e1 = ev(), ev()
    barrier()
    e0.record()
    L.check(L.lib.o3db_icp_create(d_src.data_ptr(), n, d_tgt.data_ptr(), d_nrm.data_ptr(), m, L.dptr(T0), C.byref(opt),
                                  comm.handle if comm else None, stream, C.byref(h)))
    e1.record()
    torch.cuda.synchronize()
    build_ms = e0.elapsed_time(e1)
    res = L.IcpResult()

    def icp_step(timed):
        """One registration: reset (untimed), 30 iterations + final evaluation (timed)."""
        L.check(L.lib.o3db_icp_reset(h, stream))
        flush_l2()
        a, b, c = ev(), ev(), ev()
        a.record()
        L.check(L.lib.o3db_icp_iterate(h, ICP_ITERS, stream))
        b.record()
        L.check(L.lib.o3db_icp_finish(h, C.byref(res), None, None, stream))   # syncs; reads the result back
        c.record()
        torch.cuda.synchronize()
        return a.elapsed_time(c), a.elapsed_time(b)

    for _ in range(args.warmup):
        icp_step(False)
    barrier()
    launches0 = L.launch_count()
    wall0 = time.perf_counter()
    with ClockSampler(local_rank) as clocks:
        step_ms, loop_ms = 0.0, 0.0
        for _ in range(args.steps):
            s, l = icp_step(True)
            step_ms += s
            loop_ms += l
        barrier()
    icp_wall = time.perf_counter() - wall0
    icp_launches = L.launch_count() - launches0
    step_ms = max_over_ranks(step_ms)
    loop_ms = max_over_ranks(loop_ms)
    icp_value = world * ICP_ITERS * args.steps / (step_ms * 1e-3)
    kern_ms = loop_ms / (ICP_ITERS * args.steps)          # average launch duration of icp_iteration_kernel
    alg = icp_algorithmic_bytes(n, m)
    icp_roof = {"bound": "hbm", "kernel": "icp_iteration_kernel", "achieved": alg / (kern_ms * 1e-3) / 1e9,
                "peak": peak, "unit": "GB/s", "frac": alg / (kern_ms * 1e-3) / 1e9 / peak,
                "traffic": ncu_traffic("icp_iteration_kernel"), "algorithmic_bytes_per_launch": alg,
                "avg_launch_us": kern_ms * 1e3, "peak_source": peak_src}
    final = {"fitness": res.fitness, "inlier_rmse": res.inlier_rmse, "num_iterations": res.num_iterations,
             "transformation_error_vs_ground_truth": float(np.abs(np.array(res.transformation).reshape(4, 4) - T_gt).max())}
    dump = {"icp_transformation": np.array(res.transformation).reshape(4, 4),
            "icp_fitness": np.float64([res.fitness]), "icp_inlier_rmse": np.float64([res.inlier_rmse]),
            "icp_num_iterations": np.float64([res.num_iterations]),
            "icp_num_correspondences": np.float64([res.num_correspondences])}
    L.lib.o3db_icp_destroy(h)

    # e2e: host buffers (pinned) through the C ABI, everything inside the timed region
    hs, ht, hn = (torch.from_numpy(a).pin_memory() for a in (src, tgt, nrm))
    res2 = L.IcpResult()
    e2e_ms = 0.0
    if world == 1:
        for i in range(2 + args.steps):
            flush_l2()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            L.check(L.lib.o3db_icp_point_to_plane_host(hs.data_ptr(), n, ht.data_ptr(), hn.data_ptr(), m, L.dptr(T0),
                                                       C.byref(opt), C.byref(res2), None, None))
            torch.cuda.synchronize()
            if i >= 2:
                e2e_ms += 1e3 * (time.perf_counter() - t0)
        icp_e2e = {"value": ICP_ITERS * args.steps / (e2e_ms * 1e-3), "unit": "iters/s",
                   "h2d_bytes_per_step": int(n * 12 + m * 24), "d2h_bytes_per_step": C.sizeof(L.IcpResult),
                   "ms_per_step": e2e_ms / args.steps,
                   "path": "o3db_icp_point_to_plane_host: H2D + index build + 30 iterations + evaluation + D2H"}
    else:
        # N ranks: every rank uploads its source shard + the replicated target from pinned memory, builds
        # its index, runs the 30 all-reduced iterations and reads the result back
        for i in range(2 + args.steps):
            flush_l2()
            barrier()
            t0 = time.perf_counter()
            ds, dt, dn = hs.cuda(non_blocking=True), ht.cuda(non_blocking=True), hn.cuda(non_blocking=True)
            h2 = C.c_void_p()
            L.check(L.lib.o3db_icp_create(ds.data_ptr(), n, dt.data_ptr(), dn.data_ptr(), m, L.dptr(T0), C.byref(opt),
                                          comm.handle, stream, C.byref(h2)))
            L.check(L.lib.o3db_icp_iterate(h2, ICP_ITERS, stream))
            L.check(L.lib.o3db_icp_finish(h2, C.byref(res2), None, None, stream))
            torch.cuda.synchronize()
            dt_ms = 1e3 * (time.perf_counter() - t0)
            L.lib.o3db_icp_destroy(h2)
            if i >= 2:
                e2e_ms += max_over_ranks(dt_ms)
        icp_e2e = {"value": world * ICP_ITERS * args.steps / (e2e_ms * 1e-3), "unit": "iters/s",
                   "h2d_bytes_per_step": int(n * 12 + m * 24) * world, "d2h_bytes_per_step": C.sizeof(L.IcpResult) * world,
                   "ms_per_step": e2e_ms / args.steps,
                   "path": "per rank: pinned H2D of shard + target, o3db_icp_create(comm) + iterate + finish, D2H result"}

    # ------------------------------------------- multi-GPU extras: transport, strong scaling, configs[3]
    multi = None
    if world > 1:
        transport = ("in-kernel exchange over NVLink peer memory (one kernel per iteration)"
                     if L.lib.o3db_comm_uses_peer_memory(comm.handle) else
                     "ncclAllReduce(30 x f64) + finalize kernel per iteration")
        # strong scaling (SURVEY 8e's actual partition): ONE 2M-point registration, its source split over the ranks
        from open3d_b200.distributed import shard_range
        full = make_icp_pair(ICP_POINTS, seed=2)[0]
        b, e = shard_range(len(full), rank, world)
        d_shard = torch.from_numpy(np.ascontiguousarray(full[b:e])).cuda()
        hs_ = C.c_void_p()
        L.check(L.lib.o3db_icp_create(d_shard.data_ptr(), e - b, d_tgt.data_ptr(), d_nrm.data_ptr(), m, L.dptr(T0), C.byref(opt),
                                      comm.handle, stream, C.byref(hs_)))
        rs = L.IcpResult()

        def strong_step():
            L.check(L.lib.o3db_icp_reset(hs_, stream))
            flush_l2()
            a, c = ev(), ev()
            a.record()
            L.check(L.lib.o3db_icp_iterate(hs_, ICP_ITERS, stream))
            L.check(L.lib.o3db_icp_finish(hs_, C.byref(rs), None, None, stream))
            c.record()
            torch.cuda.synchronize()
            return a.elapsed_time(c)
        for _ in range(args.warmup):
            strong_step()
        barrier()
        strong_ms = max_over_ranks(sum(strong_step() for _ in range(args.steps)))
        L.lib.o3db_icp_destroy(hs_)
        multi = {"transport": transport,
                 "strong_scaling": {"value": ICP_ITERS * args.steps / (strong_ms * 1e-3), "unit": "iters/s",
                                    "ms_per_step": strong_ms / args.steps, "points_source_total": int(len(full)),
                                    "points_source_per_gpu": int(e - b), "scaling": "strong",
                                    "workload": "ONE 2M-point registration (BASELINE configs[1]), source rows split over the ranks, "
                                                "target replicated",
                                    "fitness": rs.fitness, "inlier_rmse": rs.inlier_rmse}}
    if world > 1 or args.config3:
        try:
            cfg3 = bench_config3(args, rank, world, comm, torch, barrier, max_over_ranks)
        except Exception as exc:   # reported, never hidden; the primary line must survive
            cfg3 = {"error": f"{type(exc).__name__}: {exc}"}
        multi = dict(multi or {}, config3=cfg3)

    # ----------------------------------------------------------------- TSDF
    tsdf = None
    if not args.skip_tsdf:
        tsdf = bench_tsdf(args, rank, world, local_rank, L, torch, stream, barrier, max_over_ranks, peak, peak_src,
                          dump if args.dump_outputs else None)

    # ---------------------------------------------------------- CPU baseline
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        import oracle
        v, r, rates = cpu_icp_baseline(src, tgt, nrm, 3, reps=5)
        cpu = {"value": v, "unit": "iters/s", "cores": oracle.num_threads(), "kind": "port",
               "sample": "3 iterations on the full 2M-point clouds (iteration loop only; OpenMP port of the "
                         "reference CPU path, f32 accumulation); median of 5 repetitions after one warm-up, "
                         f"min {min(rates):.1f} max {max(rates):.1f}",
               "build_seconds": r.build_seconds}
        if tsdf is not None:
            tsdf["cpu_baseline"] = cpu_tsdf_best(tsdf_cpu_frames(12, args.tsdf_frames), reps=5)

    if rank == 0:
        icp_line = {"metric": "icp_iters_per_sec_2M_pts", "value": icp_value, "unit": "iters/s", "n_gpus": world,
                    "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms / args.steps,
                    "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                    "config": icp_config(world), "correspondences_per_sec": icp_value * ICP_POINTS,
                    "index_build_ms": build_ms, "result": final, "roofline": icp_roof, "cpu_baseline": cpu,
                    "e2e": icp_e2e, "gpu_launches": int(icp_launches), "clocks": clocks.summary(),
                    "wall_s_timed_region": icp_wall}
        if multi is not None:
            icp_line["multi_gpu"] = multi
        if args.metric == "tsdf" and tsdf is not None:
            # same one-line schema, BASELINE configs[2] on top: depth-only integration is `value` (the config names
            # depth frames), the depth+colour run and everything else sit beside it; the ICP line rides along nested
            d = tsdf["depth_only"]
            line = {"metric": tsdf["metric"], "value": d["value"], "unit": "frames/s", "n_gpus": world,
                    "steps": args.steps, "warmup": args.warmup, "ms_per_step": d["ms_per_frame"] * tsdf["config"]["frames"] / world,
                    "higher_is_better": True, "scaling": tsdf["scaling"], "vs_baseline": None, "dtype": "f32",
                    "data": "synthetic", "config": tsdf["config"], "roofline": d["roofline"],
                    "cpu_baseline": tsdf.get("cpu_baseline"), "e2e": d["e2e"], "gpu_launches": d["gpu_launches"],
                    "clocks": tsdf.get("clocks"), "depth_color": tsdf["depth_color"], "raycast": tsdf.get("raycast"),
                    "dense_slam": tsdf.get("dense_slam"), "icp": icp_line}
        else:
            line = dict(icp_line, tsdf=tsdf)
        if args.dump_outputs:
            write_outputs(args.dump_outputs, dump)
        print(json.dumps(line), flush=True)
    if world > 1:
        comm.close()
        dist.destroy_process_group()


def bench_tsdf(args, rank, world, local_rank, L, torch, stream, barrier, max_over_ranks, peak, peak_src, dump=None):
    """`dump` (a dict, or None): receives the volume of the last timed device pass of each variant, the last ray cast
    and the dense-SLAM loop's final pose."""
    from tests.synth import PRIMESENSE_K, camera_pose, render_depth
    F = args.tsdf_frames
    mine = list(range(rank, F, world))                      # frames round-robin over independent volumes
    K = np.ascontiguousarray(PRIMESENSE_K)
    poses, exts = [], []
    for i in mine:
        T = camera_pose(i, n_frames=F)
        E = np.eye(4)
        E[:3, :3] = T[:3, :3].T
        E[:3, 3] = -(T[:3, :3].T @ T[:3, 3])
        poses.append(T)
        exts.append(np.ascontiguousarray(E))
    depth_dev, color_dev = [], []
    for T in poses:
        d, c = render_depth(T, device="cuda", with_color=True)
        depth_dev.append(d.contiguous())
        color_dev.append(c.contiguous())
    depth_host = torch.stack(depth_dev).cpu().pin_memory()
    color_host = torch.stack(color_dev).cpu().pin_memory()
    torch.cuda.synchronize()
    ext_all = np.ascontiguousarray(np.stack(exts).reshape(-1, 16))
    PtrArr = C.c_void_p * len(mine)
    dev_ptrs = PtrArr(*[t.data_ptr() for t in depth_dev])
    dev_cptrs = PtrArr(*[t.data_ptr() for t in color_dev])
    host_ptrs = PtrArr(*[depth_host[j].data_ptr() for j in range(len(mine))])
    host_cptrs = PtrArr(*[color_host[j].data_ptr() for j in range(len(mine))])
    out = {}
    steps, warmup = args.steps, 1
    for color in (False, True):
        name = "depth_color" if color else "depth_only"
        results = {}
        for mode in ("device", "host"):
            tot_ms, launches, touch_ms, integ_ms, nfr, blocks = 0.0, 0, 0.0, 0.0, 0, 0
            exec_ms, exec_launches = 0.0, 0
            # device mode runs one extra, untimed pass with per-kernel CUDA events (they perturb the
            # pipeline, so the pass that feeds `value` runs without them)
            n_pass = warmup + steps + (1 if mode == "device" else 0)
            for it in range(n_pass):
                v = C.c_void_p()
                L.check(L.lib.o3db_vbg_create(VOXEL, RES, 40000, 1, stream, C.byref(v)))   # default_config.yml:26
                profiled = mode == "device" and it == n_pass - 1
                timed = it >= warmup and not profiled
                if profiled:
                    L.check(L.lib.o3db_vbg_profile(v, 1))
                barrier()
                l0 = L.launch_count()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0 = time.perf_counter()
                a.record()
                dptrs = dev_ptrs if mode == "device" else host_ptrs
                cptrs = (dev_cptrs if mode == "device" else host_cptrs) if color else None
                L.check(L.lib.o3db_vbg_integrate_sequence(v, len(mine), dptrs, L.DEPTH_U16, cptrs, L.COLOR_U8, 480, 640,
                                                          L.dptr(K), L.dptr(ext_all), DSCALE, DMAX, TRUNC_MULT,
                                                          0 if mode == "device" else 1, stream))
                b.record()
                size = L.check(L.lib.o3db_vbg_size(v, stream))      # D2H read of the step's result (block count)
                torch.cuda.synchronize()
                wall = 1e3 * (time.perf_counter() - t0)
                if timed:
                    tot_ms += a.elapsed_time(b) if mode == "device" else wall
                    launches += L.launch_count() - l0
                    blocks = int(size)
                    if mode == "device":       # device-timer duration of the integrate launches of the TIMED passes
                        em, el = C.c_double(0), C.c_int64(0)
                        L.check(L.lib.o3db_vbg_exec_stats(v, C.byref(em), C.byref(el), 1, stream))
                        exec_ms += em.value
                        exec_launches += el.value
                        if dump is not None and rank == 0 and it == warmup + steps - 1:
                            dump.update(volume_outputs(L, v, stream, torch, f"tsdf_{name}", color))
                if profiled:
                    if True:
                        tm, im, nf = C.c_double(0), C.c_double(0), C.c_int64(0)
                        L.check(L.lib.o3db_vbg_profile_read(v, C.byref(tm), C.byref(im), C.byref(nf)))
                        touch_ms += tm.value
                        integ_ms += im.value
                        nfr += nf.value
                L.lib.o3db_vbg_destroy(v)
            tot_ms = max_over_ranks(tot_ms)
            results[mode] = {"frames_per_sec": F * steps / (tot_ms * 1e-3),
                             "ms_per_frame": tot_ms / (len(mine) * steps), "launches": launches, "blocks_total": blocks,
                             "touch_ms": touch_ms, "integrate_ms": integ_ms, "profiled_frames": nfr,
                             "exec_ms": exec_ms, "exec_launches": exec_launches}
        dev, host = results["device"], results["host"]
        entry = {"value": dev["frames_per_sec"], "unit": "frames/s", "ms_per_frame": dev["ms_per_frame"],
                 "gpu_launches": dev["launches"], "blocks_in_volume_after_sequence": dev["blocks_total"],
                 "e2e": {"value": host["frames_per_sec"], "unit": "frames/s",
                         "h2d_bytes_per_step": 640 * 480 * (2 + (3 if color else 0)) * len(mine),
                         "d2h_bytes_per_step": 64,
                         "path": "o3db_vbg_integrate_sequence(host images): per frame pinned H2D + touch + integrate; block-count read-back per sequence"}}
        out[name] = entry
        out[name]["_dev"] = dev
    # mean touched blocks per frame (needed by the byte model) — measured on the device with the
    # stand-alone GetUniqueBlockCoordinates entry point on a sample of frames
    v = C.c_void_p()
    L.check(L.lib.o3db_vbg_create(VOXEL, RES, 1000, 0, stream, C.byref(v)))
    cnts = []
    nb = C.c_int64(0)
    for j in range(0, len(mine), max(1, len(mine) // 50)):
        L.check(L.lib.o3db_vbg_unique_block_coordinates(v, depth_dev[j].data_ptr(), L.DEPTH_U16, 480, 640, L.dptr(K),
                                                        L.dptr(exts[j]), DSCALE, DMAX, TRUNC_MULT, None, 0,
                                                        C.byref(nb), stream))
        cnts.append(nb.value)
    L.lib.o3db_vbg_destroy(v)
    mean_blocks = float(np.mean(cnts))
    for color in (False, True):
        name = "depth_color" if color else "depth_only"
        dev = out[name].pop("_dev")
        alg = tsdf_algorithmic_bytes(mean_blocks, color)
        k_ms = dev["integrate_ms"] / max(dev["profiled_frames"], 1)
        x_ms = dev["exec_ms"] / max(dev["exec_launches"], 1)
        out[name]["roofline"] = {"bound": "hbm", "kernel": "integrate16_kernel", "achieved": alg / (k_ms * 1e-3) / 1e9,
                                 "peak": peak, "unit": "GB/s", "frac": alg / (k_ms * 1e-3) / 1e9 / peak,
                                 "avg_exec_us_device_timer": x_ms * 1e3,
                                 "frac_device_timer": (alg / (x_ms * 1e-3) / 1e9 / peak) if x_ms > 0 else None,
                                 "timing_note": "avg_launch_us / frac: CUDA events around every kernel in an extra, untimed pass "
                                                "(the events sit between the frame's two kernels and disable their programmatic "
                                                "overlap, so each interval also contains an un-hidden launch latency); "
                                                "avg_exec_us_device_timer: %globaltimer of the last CTA's end minus the earliest "
                                                "CTA's start, accumulated by the kernel itself during the TIMED passes",
                                 "traffic": ncu_traffic("integrate_kernel_color" if color else "integrate_kernel"),
                                 "algorithmic_bytes_per_launch": alg, "avg_launch_us": k_ms * 1e3,
                                 "touch_kernel_avg_us": 1e3 * dev["touch_ms"] / max(dev["profiled_frames"], 1),
                                 "mean_touched_blocks_per_frame": mean_blocks, "peak_source": peak_src,
                                 "model_note": "algorithmic bytes = every voxel of every touched block read AND written "
                                               "(SURVEY 8d): an upper bound, voxels behind the truncation band are read "
                                               "but not written; `traffic` is the ncu cold-cache DRAM figure (writes still "
                                               "in L2 at the end of a replay are not counted by ncu)",
                                 "frame_frac_end_to_end": alg / (dev["ms_per_frame"] * 1e-3) / 1e9 / peak}
    # slam::Model::SynthesizeModelFrame (EstimateRange + RayCast of the last frame's frustum, depth + colour),
    # SURVEY 8f #4: reported beside the integration numbers, not part of `value`
    if rank == 0:
        v = C.c_void_p()
        L.check(L.lib.o3db_vbg_create(VOXEL, RES, 40000, 1, stream, C.byref(v)))
        nseq = min(60, len(mine))
        L.check(L.lib.o3db_vbg_integrate_sequence(v, nseq, dev_ptrs, L.DEPTH_U16, dev_cptrs, L.COLOR_U8, 480, 640,
                                                  L.dptr(K), L.dptr(ext_all), DSCALE, DMAX, TRUNC_MULT, 0, stream))
        rd = torch.empty((480, 640, 1), dtype=torch.float32, device="cuda")
        rc = torch.empty((480, 640, 3), dtype=torch.float32, device="cuda")
        ro = L.RaycastOutputs()
        ro.depth, ro.color = rd.data_ptr(), rc.data_ptr()
        E_last = exts[nseq - 1]
        reps = 20

        def cast():
            L.check(L.lib.o3db_vbg_ray_cast(v, None, 0, L.dptr(K), L.dptr(E_last), 640, 480, C.byref(ro), DSCALE, 0.1, DMAX,
                                            3.0, TRUNC_MULT, 8, None, stream))
        for _ in range(3):
            cast()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = L.launch_count()
        a.record()
        for _ in range(reps):
            cast()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / reps
        if dump is not None:
            dump.update(raycast_depth=rd.clone(), raycast_color=rc.clone())
        out["raycast"] = {"workload": "slam::Model::SynthesizeModelFrame 640x480 depth+color after 60 fused frames",
                          "ms_per_frame": ms, "frames_per_sec": 1e3 / ms, "rays_per_sec": 640 * 480 / (ms * 1e-3),
                          "hit_fraction": float((rd > 0).float().mean()), "gpu_launches_per_frame":
                          (L.launch_count() - l0) / reps}
        L.lib.o3db_vbg_destroy(v)
    # BASELINE configs[4]: the full slam::Model loop of dense_slam.py — track_frame_to_model (RGB-D odometry against
    # the ray-cast model frame) -> update_frame_pose -> integrate -> synthesize_model_frame — on consecutive
    # frames, poses estimated by the tracker.  Every rank runs its own segment of the trajectory on its own model
    # (frame-parallel replicas).  Wall-clock with a synchronize on both sides: the loop needs the odometry result on
    # the host every frame (pose = pose @ T), as the reference's API does.
    import open3d_b200
    slam = open3d_b200.t.pipelines.slam
    # Every rank tracks the SAME trackable segment (frames 0..S-1) into its own volume — independent replicas, which is
    # what "frame-parallel" means for a loop whose frames depend on each other.  (Other stretches of the synthetic
    # trajectory face a single flat wall, where point-to-plane odometry is singular in the reference's CPU path as
    # well: the oracle loop raises at frame 501 exactly like the CUDA path.)
    S = max(10, min(100, F // max(world, 1)))
    seg = [k for k in range(S)]
    seg_frames = []
    for i in seg:
        d, c = render_depth(camera_pose(i, n_frames=F), device="cuda", with_color=True)
        seg_frames.append((d.contiguous(), c.contiguous()))

    def slam_loop(n_frames, model=None):
        T0 = camera_pose(seg[0], n_frames=F)
        if model is None:
            model = slam.Model(VOXEL, RES, 40000, T0)
        pose = T0.copy()
        rc_frame = slam.Frame(480, 640, K)
        for n in range(n_frames):
            fr = slam.Frame(480, 640, K)
            fr.set_data("depth", seg_frames[n][0])
            fr.set_data("color", seg_frames[n][1])
            if n > 0:
                res = model.track_frame_to_model(fr, rc_frame, DSCALE, DMAX, 0.07)
                pose = pose @ res.transformation
            model.update_frame_pose(n, pose)
            model.integrate(fr, DSCALE, DMAX, TRUNC_MULT)
            model.synthesize_model_frame(rc_frame, DSCALE, 0.1, DMAX, TRUNC_MULT, False)
        torch.cuda.synchronize()
        return pose

    slam_err = None
    pose = camera_pose(seg[0], n_frames=F)
    l0, t0 = L.launch_count(), time.perf_counter()
    barrier()                                  # (no collective inside the try: a rank that loses track must not hang the others)
    try:
        slam_loop(min(8, S))                   # warm-up (allocator pools, pinned blocks)
        # The volume (a 1.9 GB allocation + clear) is built before the clock starts: configs[4] amortises it over 5000
        # frames, this bounded segment would charge it to 100.  It stays alive until the clock has stopped.
        timed_model = slam.Model(VOXEL, RES, 40000, camera_pose(seg[0], n_frames=F))
        torch.cuda.synchronize()
        l0 = L.launch_count()
        t0 = time.perf_counter()
        pose = slam_loop(S, timed_model)
    except RuntimeError as e:                  # tracking lost: reported, never hidden
        slam_err = str(e)
    slam_ms = max_over_ranks(1e3 * (time.perf_counter() - t0))
    timed_model = None
    if max_over_ranks(1.0 if slam_err else 0.0) > 0 and not slam_err:
        slam_err = "tracking failed on another rank"      # its clock is meaningless: report, never average over it
    gt = camera_pose(seg[-1], n_frames=F)
    if dump is not None and rank == 0 and not slam_err:
        dump["dense_slam_final_pose"] = pose
    out["dense_slam"] = {"error": slam_err} if slam_err else {"workload": "slam::Model loop (odometry PointToPlane {6,3,1} + integrate + ray cast), "
                                     f"{S} consecutive 640x480 RGB-D frames per GPU, poses estimated",
                         "baseline_config": "configs[4] (bounded segment)", "frames_per_sec": world * S / (slam_ms * 1e-3),
                         "ms_per_frame": slam_ms / S, "gpu_launches_per_frame": (L.launch_count() - l0) / S,
                         "final_pose_translation_error_mm": float(1e3 * np.linalg.norm(pose[:3, 3] - gt[:3, 3])),
                         "timing": "wall clock, host in the loop (one odometry result read-back per frame); the volume is "
                                   "allocated before the clock starts (configs[4] amortises it over 5000 frames)"}
    out["metric"] = "tsdf_frames_per_sec_640x480"
    out["config"] = tsdf_config(world, F)
    out["higher_is_better"] = True
    out["scaling"] = "weak" if world == 1 else "strong (fixed 1000-frame sequence split over volumes)"

    return out


if __name__ == "__main__":
    main()
