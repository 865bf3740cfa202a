#!/usr/bin/env python
"""bench.py — registration residuals/s + pose-graph solve ms (BASELINE.json metric).

A "step" is one full evaluation of the registration hot path over every registration
constraint of the pose graph: per point transform -> 8-voxel brick gather -> trilinear
interpolation -> residual -> two 1x4 Jacobians -> in-kernel reduction to the per-constraint
normal-equation blocks -> assembly of the global J^T J / J^T r (+ one exchange of the packed
normal equations over NVLink for N > 1).

Workloads
  config2  BASELINE.json configs[1]: 50 submaps / 200 overlapping pairs (x2 mirrored residual
           blocks) / 10k isosurface points per block, 0.20 m voxels.  Headline at N = 1.
  config4  BASELINE.json configs[3]: 200 submaps / 1500 pairs / 20k points / 0.10 m voxels, every
           submap shared by all ranks, constraints sharded (STRONG scaling).  Headline at N > 1;
           at N = 1 it is measured as a second leg and reported inside the kept dicts
           (`e2e.config4`, `roofline.config4`) so the 1 -> 8 curve has its own N = 1 point.
At N > 1 rank 0 re-evaluates the full problem on one GPU (vgx_comm_suspend) and the line carries
`e2e.parity_vs_single_rank`; the run fails when it exceeds 1e-12.

  python bench.py --gpus 1 --steps 20 --warmup 3
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference      # restated reference CPU path on the host cores
"""
import argparse
import json
import os
import pickle
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ALGO_BYTES_PER_RESIDUAL = 84  # SURVEY.md §8(d): 20 B point + 8 corners x (4 B distance + 4 B weight)
ALGO_BYTES_PER_TSDF_UPDATE = 16
_REAL_STDOUT = sys.stdout

WORKLOADS = {
    # name: (submaps, pairs, points, voxel size, seed, BASELINE.json configs index)
    "config2": dict(submaps=50, pairs=200, points=10000, voxel_size=0.2, seed=2, baseline_index=1),
    "config4": dict(submaps=200, pairs=1500, points=20000, voxel_size=0.1, seed=4, baseline_index=3),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto", "config2", "config4", "stream", "rgbd"],
                    help="auto: config2 at N = 1 (+ a config4 leg), config4 (strong scaling) at N > 1")
    ap.add_argument("--submaps", type=int, default=None)
    ap.add_argument("--pairs", type=int, default=None)
    ap.add_argument("--points", type=int, default=None)
    ap.add_argument("--voxel-size", type=float, default=None)
    ap.add_argument("--no-extras", action="store_true", help="skip solve / TSDF / CPU baseline / config4 legs")
    ap.add_argument("--no-config4", action="store_true", help="N = 1: skip the config4 leg")
    ap.add_argument("--no-stream", action="store_true", help="N = 1: skip the streaming (configs[2]) leg")
    ap.add_argument("--stream-scans", type=int, default=40)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU baseline budget")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the cost, gradient and H of the timed evaluation as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload in ("stream", "rgbd")):
        ap.error("--dump-outputs applies to the registration evaluation (--impl b200, workload auto / config2 / config4)")
    return args


def workload_params(name, args):
    w = dict(WORKLOADS[name])
    for k, a in (("submaps", args.submaps), ("pairs", args.pairs), ("points", args.points),
                 ("voxel_size", args.voxel_size)):
        if a is not None:
            w[k] = a
    w["name"] = name
    return w


# --------------------------------------------------------------------------- workload
def build_scene(w, rank=0, wait_s=1500.0):
    """Seeded synthetic scene, cached in /tmp (generation is host-side numpy, forked workers: must
    run before this process touches CUDA).  Under torchrun only rank 0 generates; the others wait
    for the cache file."""
    from voxgraph_b200 import synth
    key = "vgx_scene_v3_%s_s%d_p%d_k%d_v%g.pkl" % (w["name"], w["submaps"], w["pairs"], w["points"],
                                                   w["voxel_size"])
    path = os.path.join("/tmp", key)

    def load():
        try:
            with open(path, "rb") as f:
                return pickle.load(f)
        except Exception:
            return None

    sc = load() if os.path.exists(path) else None
    if sc is not None:
        return sc
    if rank != 0:
        t0 = time.time()
        while time.time() - t0 < wait_s:
            if os.path.exists(path):
                sc = load()
                if sc is not None:
                    return sc
            time.sleep(1.0)
        raise RuntimeError("rank %d: scene cache %s did not appear" % (rank, path))
    workers = max(1, min(64, (os.cpu_count() or 2) - 2))
    sc = synth.make_scene(seed=w["seed"], n_submaps=w["submaps"], n_points=w["points"],
                          voxel_size=w["voxel_size"], max_pairs=w["pairs"],
                          trunc=0.6 if abs(w["voxel_size"] - 0.2) < 1e-9 else None,
                          drift=(0.03, 0.005, 0.002), workers=workers)
    try:
        tmp = path + ".%d" % os.getpid()
        with open(tmp, "wb") as f:
            pickle.dump(sc, f, protocol=4)
        os.replace(tmp, path)
    except Exception:
        pass
    return sc


def _scan_job(job):
    from voxgraph_b200 import synth
    world, pose, kind, seed = job
    if kind == "lidar":
        return synth.lidar_scan(world, pose, n_beams=64, n_azimuth=1024, seed=seed, max_range=16.0)
    return synth.depth_scan(world, pose, seed=seed)


def build_stream(kind, n_scans, rank=0, wait_s=900.0):
    """Synthetic sensor stream (SURVEY §8d cfg 3 / cfg 5): the sensor moves at 2 m/s through the hall;
    kind = "lidar": 64 x 1024 beams @ 10 Hz; "rgbd": 640 x 480 depth @ 30 Hz (<= 5 m).  Odometry =
    ground truth + integrated drift.  Host-side numpy ray casting, forked workers, cached in /tmp."""
    from voxgraph_b200 import synth
    path = "/tmp/vgx_stream_v3_%s_%d.pkl" % (kind, n_scans)

    def load():
        try:
            with open(path, "rb") as f:
                return pickle.load(f)
        except Exception:
            return None
    st = load() if os.path.exists(path) else None
    if st is not None:
        return st
    if rank != 0:
        t0 = time.time()
        while time.time() - t0 < wait_s:
            st = load() if os.path.exists(path) else None
            if st is not None:
                return st
            time.sleep(1.0)
        raise RuntimeError("stream cache %s did not appear" % path)
    world = synth.make_world(3, size_xy=(120.0, 80.0), n_clutter=400, n_walls=24)
    hz = 10.0 if kind == "lidar" else 30.0
    dt = 1.0 / hz
    rng = np.random.default_rng(3)
    # a gentle arc through the hall at 2 m/s
    s_arc = np.arange(n_scans) * dt * 2.0
    x = 20.0 + s_arc * np.cos(0.15) ; y = 20.0 + s_arc * np.sin(0.15) + 3.0 * np.sin(s_arc / 9.0)
    yaw = np.arctan2(np.gradient(y), np.gradient(x)) if n_scans > 1 else np.zeros(1)
    gt = np.stack([x, y, np.full(n_scans, 1.2), yaw], -1)
    odo = gt.copy()
    drift = np.cumsum(rng.normal(0, 1.0, (n_scans, 4)) * np.array([0.02, 0.02, 0.001, 0.002]), 0)
    odo += drift
    import multiprocessing as mp
    workers = max(1, min(64, (os.cpu_count() or 2) - 2))
    jobs = [(world, gt[k], kind, 100 + k) for k in range(n_scans)]
    with mp.get_context("fork").Pool(min(workers, n_scans)) as pool:
        scans = pool.map(_scan_job, jobs, chunksize=1)
    st = {"kind": kind, "hz": hz, "gt": gt, "odom": odo, "scans": [np.ascontiguousarray(p, np.float32) for p in scans]}
    try:
        tmp = path + ".%d" % os.getpid()
        with open(tmp, "wb") as f:
            pickle.dump(st, f, protocol=4)
        os.replace(tmp, path)
    except Exception:
        pass
    return st


def stream_leg(ctx, api, st, voxel_size, scans_per_submap, peak, cpu_scans=3):
    """BASELINE configs[2]-shaped run: scans -> TSDF integration (Fast, as voxgraph) -> every
    `scans_per_submap` scans: finish the submap on the device (view + registration points + OBB),
    overlap detection, registration constraints, LM solve - the reference's
    VoxgraphMapper::pointcloudCallback order (voxgraph_mapper.cpp:202-265, 457-524)."""
    from oracle import oracle as o
    from voxgraph_b200 import mapper as vm
    hz = st["hz"]
    trunc = 3.0 * voxel_size
    cfg = vm.MapperConfig(voxel_size=voxel_size, submap_creation_interval=scans_per_submap / hz,
                          capacity_blocks=16384 if voxel_size >= 0.1 else 32768,
                          tsdf=dict(default_truncation_distance=trunc,
                                    max_ray_length_m=16.0 if st["kind"] == "lidar" else 5.0))
    # warm-up: module load, scratch growth
    ctx.submap_create(9 * 10 ** 5, voxel_size, 16, cfg.capacity_blocks)
    wcfg = ctx.tsdf_config(mode=1, default_truncation_distance=trunc)
    for k in range(2):
        ctx.tsdf_integrate(9 * 10 ** 5, np.array([1, 0, 0, 0, 0, 0, 0], np.float32), st["scans"][k], wcfg)
    ctx.submap_free(9 * 10 ** 5)
    # ... and one throw-away pass through two submap switches (finish, overlap, constraints, solve):
    # first launches of those kernels load their modules and grow the scratch buffers
    wm = vm.VoxgraphMapper(ctx, cfg, first_submap_id=3 * 10 ** 5)
    for k in range(min(len(st["scans"]), 2 * scans_per_submap + 1)):
        wm.pointcloudCallback(k / hz, st["odom"][k], st["scans"][k])
    ctx.synchronize()
    for i in wm.submap_ids:
        ctx.submap_free(i)
    del wm
    m = vm.VoxgraphMapper(ctx, cfg, first_submap_id=2 * 10 ** 5)
    n = len(st["scans"])
    ctx.profile_reset(); ctx.profile_enable(True)
    per_scan = []
    t_all = time.time()
    for k in range(n):
        t0 = time.time()
        m.pointcloudCallback(k / hz, st["odom"][k], st["scans"][k])
        per_scan.append(time.time() - t0)
    ctx.synchronize()
    wall = time.time() - t_all
    k_ms, k_n = ctx.profile_get(2)
    ctx.profile_enable(False)
    upd = sum(int(s.voxel_updates) for s in m.scan_stats)
    rays = sum(int(p.shape[0]) for p in st["scans"])
    switch = [t for t in m.timings if t.get("finish_ms", 0) > 0]
    integ = np.array([per_scan[k] for k in range(n) if k % scans_per_submap != 0] or per_scan)
    # drift correction: optimised submap origins vs the ground-truth sensor pose at their creation
    ids = m.submap_ids
    err_odo = err_opt = err_opt_tight = tight_iters = None
    if len(ids) >= 2:
        starts = [int(round(m.submap_start[i] * hz)) for i in ids]
        gt0 = st["gt"][starts]
        odo0 = st["odom"][starts]
        opt = np.array([m.submap_pose[i] for i in ids])
        # express everything relative to the first submap (gauge)
        err_odo = float(np.abs((odo0[:, :2] - odo0[0, :2]) - (gt0[:, :2] - gt0[0, :2])).mean())
        err_opt = float(np.abs((opt[:, :2] - opt[0, :2]) - (gt0[:, :2] - gt0[0, :2])).mean())
        # the reference's parameter_tolerance 3e-3 is relative to |x| (tens of metres here): a step
        # below ~5 cm ends the solve unapplied.  One more solve at 1e-8 shows what registration recovers.
        m.pose_graph.solver_options.parameter_tolerance = 1e-8
        m.pose_graph.solver_options.function_tolerance = 1e-12
        m.pose_graph.solver_options.max_num_iterations = 50
        st_tight = m.pose_graph.optimize()
        opt_t = np.array([m.pose_graph.getSubmapPoses()[i] for i in ids])
        err_opt_tight = float(np.abs((opt_t[:, :2] - opt_t[0, :2]) - (gt0[:, :2] - gt0[0, :2])).mean())
        tight_iters = int(st_tight.iterations)
    # CPU: the restated Fast integrator, all cores (voxblox: hardware_concurrency) and one thread
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    nt = max(1, min(cores, 64))
    lay = o.Layer(voxel_size, 16)
    oc = o.tsdf_config(mode=1, default_truncation_distance=trunc,
                       max_ray_length_m=16.0 if st["kind"] == "lidar" else 5.0)
    T0 = np.array([1, 0, 0, 0, 0, 0, 0], np.float32)
    o.tsdf_integrate_mt(lay, oc, T0, st["scans"][0], nt)
    cpu_ms = []
    cpu_upd = 0
    for k in range(min(cpu_scans, n)):
        t0 = time.time(); so = o.tsdf_integrate_mt(lay, oc, T0, st["scans"][k], nt); cpu_ms.append((time.time() - t0) * 1e3)
        cpu_upd += int(so.voxel_updates)
    for i in ids:
        ctx.submap_free(i)
    return {"stream": "%s, %d scans @ %g Hz, %.2f m voxels, trunc %.2f m, new submap every %d scans" % (
                st["kind"], n, hz, voxel_size, trunc, scans_per_submap),
            "rays_per_scan": rays // n, "voxel_updates_per_scan": upd // n,
            "scans_per_s_e2e": n / wall, "realtime_factor": (n / wall) / hz,
            "integrate_ms_per_scan_e2e_median": float(np.median(integ) * 1e3),
            "integrate_kernel_ms_per_scan": k_ms / max(n, 1),
            "updates_per_s_e2e": upd / wall,
            "updates_per_s_kernel": upd / (k_ms * 1e-3) if k_ms > 0 else None,
            "frac_of_hbm_peak_kernel": (upd * ALGO_BYTES_PER_TSDF_UPDATE / (k_ms * 1e-3) / 1e9 / peak) if k_ms > 0 else None,
            "submaps": len(ids),
            "submap_switch": {"finish_ms_median": float(np.median([t["finish_ms"] for t in switch])) if switch else None,
                              "overlap_ms_median": float(np.median([t["overlap_ms"] for t in switch])) if switch else None,
                              "optimize_ms_median": float(np.median([t.get("optimize_ms", 0.0) for t in switch])) if switch else None,
                              "pairs_last": switch[-1]["pairs"] if switch else 0,
                              "isosurface_points_last": switch[-1].get("isosurface_points") if switch else None,
                              "blocks_last": switch[-1].get("finished_blocks") if switch else None},
            "switch_timings_ms": [{k: (round(v, 3) if isinstance(v, float) else v) for k, v in t.items()} for t in m.timings],
            "submap_origin_xy_error_odometry_m": err_odo, "submap_origin_xy_error_optimised_m": err_opt,
            "submap_origin_xy_error_optimised_tight_m": err_opt_tight, "lm_iterations_tight": tight_iters,
            "cpu_reference_integrate_ms_per_scan_mt": float(np.median(cpu_ms)), "cpu_reference_threads": nt,
            "cpu_reference_updates_per_s_mt": cpu_upd / (sum(cpu_ms) * 1e-3)}


class _DevMem:
    """Foreign device memory as a __cuda_array_interface__ object (zero-copy torch view)."""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2}


def run_rgbd(args):
    """BASELINE configs[4]: dense RGB-D 640 x 480 @ 30 Hz, 0.05 m voxels, concurrent integration and
    registration on 2 GPUs.  Rank 0 integrates the frames (Fast scheduling) and finishes a submap every
    `frames_per_submap` frames; the finished submap's bricks cross NVLink ONCE (device pointers from
    vgx_submap_peek_device, NCCL send/recv) to rank 1, which extracts its registration points, detects
    overlaps, rebuilds the registration constraints and solves the pose graph while rank 0 keeps
    integrating - SURVEY §8e "replicas by role".  Prints one JSON line (rank 0)."""
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != 2:
        raise SystemExit("--workload rgbd needs exactly 2 ranks (torchrun --nproc-per-node 2)")
    n_frames = args.stream_scans if args.stream_scans != 40 else 90
    fps, per_submap, vs = 30.0, 30, 0.05
    st = build_stream("rgbd", n_frames, rank)
    import torch
    import torch.distributed as dist
    from voxgraph_b200 import api, mapper as vm
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = api.Context(local_rank)
    dev = torch.device("cuda", local_rank)
    n_sub = (n_frames + per_submap - 1) // per_submap
    trunc = 3 * vs
    out = {}
    def send_submap(sid, origin, pending):
        ctx.submap_finish(sid)
        pi, pd, nb = ctx.submap_peek_device(sid)
        dist.send(torch.tensor([sid, nb] + [float(v) for v in origin], dtype=torch.float64, device=dev), 1)
        ti = torch.as_tensor(_DevMem(pi, 3 * nb, "<i4"), device=dev)
        td = torch.as_tensor(_DevMem(pd, 2 * 4096 * nb, "<f4"), device=dev)
        pending += [dist.isend(ti, 1), dist.isend(td, 1)]     # the bricks cross NVLink once
        return nb

    def integrate_pass(frames, per_sub, id_base, tcfg):
        """rank 0: integrate `frames` frames, hand every finished submap to rank 1."""
        dist.barrier(); torch.cuda.synchronize()
        t_all = time.time()
        per_frame, sends, upd, pending = [], [], 0, []
        sid, origin, made = id_base - 1, None, []
        for k in range(frames):
            if k % per_sub == 0:
                if origin is not None:
                    t0 = time.time()
                    nb = send_submap(sid, origin, pending)
                    sends.append(((time.time() - t0) * 1e3, nb))
                sid += 1
                origin = st["odom"][k].copy()
                ctx.submap_create(sid, vs, 16, 16384)
                made.append(sid)
            t0 = time.time()
            T_S_C = vm._compose4(vm._inverse4(origin), st["odom"][k])
            s_ = ctx.tsdf_integrate(sid, vm._pose4_to_T(T_S_C), st["scans"][k], tcfg)
            per_frame.append(time.time() - t0)
            upd += int(s_.voxel_updates)
        send_submap(sid, origin, pending)
        t_int = time.time() - t_all
        for p in pending:
            p.wait()
        dist.send(torch.tensor([-1, 0, 0, 0, 0, 0], dtype=torch.float64, device=dev), 1)
        res = torch.zeros(8, dtype=torch.float64, device=dev)
        dist.recv(res, 1)
        torch.cuda.synchronize()
        t_total = time.time() - t_all
        for i in made:
            ctx.submap_free(i)
        return t_int, t_total, res.cpu().numpy(), per_frame, sends, upd

    def register_pass():
        """rank 1: receive finished submaps, extract, detect overlaps, constrain, solve."""
        pg = api.PoseGraph(ctx)
        ids, poses = [], {}
        busy = 0.0
        last = [0, 0.0, 0]
        prev_origin = None
        dist.barrier(); torch.cuda.synchronize()
        while True:
            hdr = torch.zeros(6, dtype=torch.float64, device=dev)
            dist.recv(hdr, 0)
            h = hdr.cpu().numpy()
            sid, nb = int(h[0]), int(h[1])
            if sid < 0:
                break
            ti = torch.empty(3 * nb, dtype=torch.int32, device=dev)
            td = torch.empty(2 * 4096 * nb, dtype=torch.float32, device=dev)
            dist.recv(ti, 0); dist.recv(td, 0)
            torch.cuda.synchronize()
            t0 = time.time()
            ctx.submap_upload_device(sid, vs, 16, nb, ti.data_ptr(), td.data_ptr())
            ctx.submap_extract_points(sid, None)
            origin = h[2:6].copy()
            pg.addSubmapNode(api.SubmapNodeConfig(sid, origin, set_constant=(not ids)))
            if ids:
                T12 = vm._compose4(vm._inverse4(prev_origin), origin)
                pg.addRelativePoseConstraint(api.RelativePoseConstraintConfig(ids[-1], sid, T12,
                                                                              np.diag([1.0, 1.0, 2500.0, 2500.0])))
            ids.append(sid); poses[sid] = origin; prev_origin = origin
            if len(ids) >= 2:
                pg.resetRegistrationConstraints()
                T = np.array([vm._pose4_to_T(poses[i]) for i in ids], np.float32)
                pairs = ctx.find_overlapping_pairs(ids, T)
                for (a, b) in pairs:
                    pg.addRegistrationConstraint(api.RegistrationConstraintConfig(a, b))
                t1 = time.time()
                summ = pg.optimize()
                for i, p in pg.getSubmapPoses().items():
                    poses[i] = p
                last = [len(pairs), (time.time() - t1) * 1e3, summ.iterations]
            ctx.synchronize()
            busy += time.time() - t0
        dist.send(torch.tensor([busy, last[0], last[1], last[2], 0, 0, 0, 0], dtype=torch.float64, device=dev), 0)
        pg.resetRegistrationConstraints()
        for i in ids:
            ctx.submap_free(i)

    if rank == 0:
        tcfg = ctx.tsdf_config(mode=1, default_truncation_distance=trunc, max_ray_length_m=5.0)
        # rehearsal (untimed): 3 short submaps through the whole hand-over -> NCCL channels, kernel
        # modules and scratch buffers exist on both GPUs before the timed pass
        integrate_pass(min(n_frames, 9), 3, 10 ** 5, tcfg)
        t_int, t_total, res, per_frame, sends, upd = integrate_pass(n_frames, per_submap, 0, tcfg)
        pts_per_frame = int(np.mean([p.shape[0] for p in st["scans"]]))
        line = {"metric": "rgbd_frames_per_s", "value": n_frames / t_total, "unit": "frames/s", "n_gpus": 2,
                "steps": n_frames, "warmup": 9, "ms_per_step": t_total / n_frames * 1e3, "higher_is_better": True,
                "scaling": "replicas by role (GPU 0 integrates, GPU 1 registers)", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": "BASELINE configs[4]: dense RGB-D 640x480 @ 30 Hz, 0.05 m voxels, "
                                       "%d frames, new submap every %d frames, concurrent integration + "
                                       "registration on 2 GPUs" % (n_frames, per_submap),
                           "points_per_frame": pts_per_frame, "voxel_size": vs, "submaps": n_sub},
                "e2e": {"value": n_frames / t_total, "unit": "frames/s", "realtime_factor_vs_30hz": n_frames / t_total / fps,
                        "integrate_ms_per_frame_median": float(np.median(per_frame) * 1e3),
                        "voxel_updates_per_s": upd / t_int,
                        "integration_wall_s": t_int, "total_wall_s": t_total,
                        "registration_busy_s_on_gpu1": float(res[0]),
                        "sequential_estimate_s": t_int + float(res[0]),
                        "overlap_gain": (t_int + float(res[0])) / t_total,
                        "submap_hand_over_ms": [round(a, 3) for (a, b) in sends],
                        "submap_blocks": [b for (a, b) in sends],
                        "submap_bytes_over_nvlink": [int(b) * (4096 * 8 + 12) for (a, b) in sends],
                        "registration_pairs_last": int(res[1]), "optimize_ms_last": float(res[2]),
                        "lm_iterations_last": int(res[3]), "h2d_bytes_per_step": pts_per_frame * 12,
                        "d2h_bytes_per_step": 32},
                "gpu_launches": int(ctx.launch_count)}
        _REAL_STDOUT.write(json.dumps(line) + "\n"); _REAL_STDOUT.flush()
    else:
        register_pass()
        register_pass()
    dist.barrier()
    ctx.close()
    dist.destroy_process_group()


def run_stream(args):
    """--workload stream: BASELINE configs[2] on its own (64 x 1024 LiDAR @ 10 Hz, 0.15 m voxels)."""
    st = build_stream("lidar", args.stream_scans, 0)
    import torch
    from voxgraph_b200 import api
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback)")
    ctx = api.Context(0)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.exists(peaks_path) else 6650.0
    r = stream_leg(ctx, api, st, 0.15, 10, peak)
    line = {"metric": "stream_scans_per_s", "value": r["scans_per_s_e2e"], "unit": "scans/s", "n_gpus": 1,
            "steps": args.stream_scans, "warmup": 2, "ms_per_step": 1e3 / r["scans_per_s_e2e"],
            "higher_is_better": True, "scaling": "replicas only", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": "BASELINE configs[2]: " + r["stream"]},
            "e2e": {"value": r["scans_per_s_e2e"], "unit": "scans/s", "h2d_bytes_per_step": r["rays_per_scan"] * 12,
                    "d2h_bytes_per_step": 32, "realtime_factor_vs_10hz": r["realtime_factor"]},
            "stream": r, "gpu_launches": int(ctx.launch_count)}
    _REAL_STDOUT.write(json.dumps(line) + "\n"); _REAL_STDOUT.flush()
    ctx.close()


def scene_problem(sc):
    """(ids, poses_init, poses_gt, pairs, odometry) of one scene."""
    ids = list(range(len(sc.submaps)))
    return ids, np.array(sc.poses_init), np.array(sc.poses_gt), list(sc.pairs), list(sc.odometry)


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for (_, r) in self.rows]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])); smax = float(f[1])
            except Exception:
                continue
            for k, nm in enumerate(names):
                if len(f) > 3 + k and f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- CPU reference arm
def oracle_graph(sc, max_residuals=None):
    from oracle import oracle as o
    ids, pinit, pgt, pairs, odo = scene_problem(sc)
    layers = {}
    g = o.Graph()
    for k, i in enumerate(ids):
        g.add_node(i, pinit[k], constant=(k == 0))
    L = o.sqrt_information(sc.odom_information)
    for (i, j, t, y) in odo:
        g.add_relative(i, j, t, y, L)
    R = 0

    def layer(i):
        if i not in layers:
            s = sc.submaps[i]
            layers[i] = o.Layer.from_blocks(s.voxel_size, s.vps, s.block_idx, s.distance, s.weight)
        return layers[i]
    for (i, j) in pairs:
        a, b = sc.submaps[i], sc.submaps[j]
        g.add_registration(i, j, layer(j), a.points_xyz, a.points_distance, a.points_weight)
        g.add_registration(j, i, layer(i), b.points_xyz, b.points_distance, b.points_weight)
        R += 2 * a.points_xyz.shape[0]
        if max_residuals is not None and R >= max_residuals:
            break
    g._layers = layers   # keep the layers alive
    return g, o


def cpu_reference(sc, budget_s, reps=7):
    """Times the restated reference CPU path (oracle; worker threads pinned to distinct cores) on a
    bounded sample of the workload: median of `reps` evaluations with all host cores and with the
    reference's own num_threads = 4 (pose_graph.cpp:96)."""
    cores = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        pass
    R_full = 2 * len(sc.pairs) * sc.submaps[0].points_xyz.shape[0]
    g, o = oracle_graph(sc, max_residuals=min(R_full, 400000))    # probe on <= 400 k residuals
    R = g.num_registration_residuals
    g.eval(num_threads=cores, want_H=True)                       # pool start-up, first touch
    t = time.time(); g.eval(num_threads=cores, want_H=True); one = time.time() - t
    per_res = one / max(R, 1)
    # all-core sample: as many residuals as fit in ~40 % of the budget over `reps` repetitions
    want = int(min(R_full, max(R, 0.4 * budget_s / (reps * per_res))))
    if want > R:
        g, o = oracle_graph(sc, max_residuals=want)
        R = g.num_registration_residuals
        g.eval(num_threads=cores, want_H=True)
    sample = ("all %d registration residuals of the workload per step" % R if R >= R_full else
              "first %d of %d registration residuals (%.0f%% of the constraints) per step" % (
                  R, R_full, 100.0 * R / R_full))
    ts = []
    for _ in range(reps):
        t0 = time.time(); g.eval(num_threads=cores, want_H=True); ts.append(time.time() - t0)
    dt = float(np.median(ts))
    nt4 = min(4, cores)
    g.eval(num_threads=nt4, want_H=True)
    ts4 = []
    for _ in range(max(3, reps // 2 + 1)):
        t0 = time.time(); g.eval(num_threads=nt4, want_H=True); ts4.append(time.time() - t0)
        if sum(ts4) > 0.5 * budget_s:
            break
    dt4 = float(np.median(ts4))
    return dict(value=R / dt, unit="residuals/s", cores=cores, kind="port", sample=sample,
                ms_per_step=dt * 1e3, value_4_threads=R / dt4, reps=reps, value_best=R / min(ts),
                spread=float((max(ts) - min(ts)) / dt) if dt > 0 else None,
                note="restated reference (Ceres/voxblox/Eigen absent from the image; see DESIGN.md); "
                     "median of %d evaluations, worker threads pinned one per core" % reps)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wname = args.workload if args.workload != "auto" else ("config2" if args.gpus <= 1 else "config4")
    w = workload_params(wname, args)
    sc = build_scene(w)
    steps = max(1, args.steps); warmup = max(0, args.warmup)
    cb = cpu_reference(sc, budget_s=60.0, reps=max(5, min(steps, 9)))
    line = {"impl": "reference", "metric": "registration_residuals_per_s", "value": cb["value"],
            "unit": "residuals/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
            "scaling": "strong" if args.gpus > 1 else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(w, sc, args.gpus),
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample",
                                                "value_4_threads", "value_best", "spread", "note")},
            "e2e": {"value": cb["value"], "unit": "residuals/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _REAL_STDOUT.write(json.dumps(line) + "\n"); _REAL_STDOUT.flush()


def workload_config(w, sc, n_gpus):
    return {"workload": "BASELINE configs[%d]: %d submaps / %d overlapping pairs (x2 mirrored residual "
                        "blocks) / %d isosurface points per block, %.2f m voxels, 16^3-voxel bricks%s"
                        % (w["baseline_index"], len(sc.submaps), len(sc.pairs), w["points"], w["voxel_size"],
                           "" if n_gpus == 1 else "; every submap resident on all %d GPUs, constraints "
                           "sharded over the ranks (strong scaling)" % n_gpus),
            "name": w["name"], "submaps": len(sc.submaps), "pairs": len(sc.pairs),
            "points_per_constraint": w["points"], "voxel_size": w["voxel_size"],
            "registration_point_type": "isosurface", "sampling_ratio": -1,
            "l2": "inputs (points + reading bricks) exceed the 126 MB L2; no explicit flush in the bracketed region",
            "parallelism": ("constraints sharded x%d; packed H/g blocks summed by a one-shot NVLink "
                            "peer-memory all-gather-reduce (CUDA IPC), NCCL all-reduce as fallback" % n_gpus)
            if n_gpus > 1 else "single GPU"}


# --------------------------------------------------------------------------- GPU arm
class Problem:
    """One workload resident on this rank's GPU + its pose graph."""

    def __init__(self, ctx, api, sc, id_base=0):
        self.ctx, self.sc = ctx, sc
        self.ids, self.pinit, self.pgt, self.pairs, self.odo = scene_problem(sc)
        self.id_base = id_base
        t_up = time.time()
        self.bricks_bytes = 0
        for k, sid in enumerate(self.ids):
            s = sc.submaps[sid]
            ctx.submap_upload(id_base + sid, s.voxel_size, s.vps, s.block_idx, s.distance, s.weight)
            ctx.submap_upload_points(id_base + sid, api.K_ISOSURFACE_POINTS, s.points_xyz,
                                     s.points_distance, s.points_weight)
            self.bricks_bytes += s.num_blocks * s.vps ** 3 * 32
        self.upload_s = time.time() - t_up
        self.api = api
        self.n_nodes = len(self.ids)
        self.build_graph()

    def build_graph(self):
        api, sc, b = self.api, self.sc, self.id_base
        pg = api.PoseGraph(self.ctx)
        for k, sid in enumerate(self.ids):
            pg.addSubmapNode(api.SubmapNodeConfig(b + sid, self.pinit[k], set_constant=(k == 0)))
        for (i, j, t, y) in self.odo:
            pg.addRelativePoseConstraint(api.RelativePoseConstraintConfig(b + i, b + j, np.array([*t, y]),
                                                                          sc.odom_information))
        for (i, j) in self.pairs:
            pg.addRegistrationConstraint(api.RegistrationConstraintConfig(b + i, b + j))
        pg._sync()
        self.pg = pg
        self.r_local, self.r_global = self.ctx.graph_num_registration_residuals()
        self.packed_len = 4 + 20 * self.n_nodes + 16 * len(
            set((min(a, c), max(a, c)) for (a, c) in list(self.pairs) + [(i, j) for (i, j, _, _) in self.odo]))

    def free(self):
        for sid in self.ids:
            self.ctx.submap_free(self.id_base + sid)


def measure(P, args, torch, dist, world, stream, want_cpu_pose_check=None, want_outputs=False):
    """Device-resident throughput, end-to-end call, roofline split and the pose-graph solve of one
    resident problem.  Every rank takes part (each evaluation contains the exchange).
    want_outputs: out["outputs"] = what a caller of the timed evaluation receives (cost, gradient, H)."""
    ctx = P.ctx

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    out = {}
    ctx.graph_set_poses(P.pinit)
    for _ in range(max(args.warmup, 3)):
        ctx.graph_eval_async()
    barrier()
    launches0 = ctx.launch_count
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(args.steps):
            ctx.graph_eval_async()
        e1.record(stream)
    barrier()
    ms_step = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    out["ms_per_step"] = ms_step
    out["value"] = P.r_global / (ms_step * 1e-3)
    out["gpu_launches"] = int(ctx.launch_count - launches0)
    if want_outputs:
        # vgx_graph_eval enqueues the evaluation each timed step enqueued, at the same poses (its sums
        # run in a fixed order, so it repeats the last step bit for bit) and copies the result back
        _, cost, g, H = ctx.graph_eval(P.n_nodes, want_H=True)
        out["outputs"] = {"cost": np.array([cost]), "gradient": g, "H": H}

    # ---- end to end through the public call with host buffers
    e2e_steps = max(3, min(args.steps, 10))
    poses_host = P.pinit.copy()
    for _ in range(2):
        ctx.graph_set_poses(poses_host); ctx.graph_eval(P.n_nodes, want_H=False)
    barrier()
    t0 = time.time()
    for k in range(e2e_steps):
        poses_host[1:, 0] += 1e-6            # new poses every step (H2D inside the timed region)
        ctx.graph_set_poses(poses_host)
        ctx.graph_eval(P.n_nodes, want_H=False)   # D2H of cost / gradient / H blocks
    barrier()
    e2e_s = max_over_ranks((time.time() - t0) / e2e_steps)
    out["e2e"] = {"value": P.r_global / e2e_s, "unit": "residuals/s", "ms_per_step": e2e_s * 1e3,
                  "h2d_bytes_per_step": int(P.n_nodes * 32), "d2h_bytes_per_step": int(P.packed_len * 8),
                  "call": "vgx_graph_set_poses + vgx_graph_eval (fused reduce mode; host poses in, host "
                          "cost/gradient/H-blocks out)"}
    ctx.graph_set_poses(P.pinit)

    # ---- roofline of the dominant kernel (per-kernel CUDA events on the ctx stream)
    barrier()
    ctx.profile_reset(); ctx.profile_enable(True)
    n_prof = max(3, min(args.steps, 10))
    for _ in range(n_prof):
        ctx.graph_eval_async()
    ctx.synchronize()
    k_ms, k_n = ctx.profile_get(0)
    parts = {name: ctx.profile_get(w)[0] for name, w in (("pose_setup", 6), ("constraint_sums", 7),
                                                         ("assemble_exchange", 8), ("other", 5))}
    ctx.profile_enable(False)
    barrier()
    kern_ms = k_ms / max(k_n, 1)
    out["kernel_ms"] = kern_ms
    out["other_kernels_ms_per_step"] = sum(parts.values()) / max(k_n, 1)
    # per-kernel events, each kernel run to completion before the next starts (no programmatic
    # overlap, and at N > 1 the exchange figure includes the ranks' skew): where the step's
    # microseconds outside the reduce kernel are
    out["step_breakdown_us"] = dict({"reg_reduce": kern_ms * 1e3},
                                    **{k: v / max(k_n, 1) * 1e3 for k, v in parts.items()})

    # ---- pose-graph solve wall time (second half of the metric)
    if not args.no_extras:
        solve = {}
        for name, kw in (("reference_options", {}),
                         ("tight", dict(parameter_tolerance=1e-6, function_tolerance=1e-9,
                                        max_num_iterations=50, max_solver_time_s=60.0))):
            ms, summ, x = [], None, None
            for rep in range(3):
                ctx.graph_set_poses(P.pinit)
                barrier()
                t0 = time.time()
                x, summ = ctx.graph_solve(P.n_nodes, ctx.solver_options(**kw))
                ms.append((time.time() - t0) * 1e3)
            d = {"solve_ms": max_over_ranks(float(np.median(ms))), "lm_iterations": summ.iterations,
                 "successful_steps": summ.num_successful_steps, "residual_evaluations": summ.num_residual_evals,
                 "termination": summ.termination, "initial_cost": summ.initial_cost,
                 "final_cost": summ.final_cost,
                 "unknowns": 4 * (P.n_nodes - 1),
                 "mean_xy_error_before_m": float(np.abs(P.pinit[:, :2] - P.pgt[:, :2]).mean()),
                 "mean_xy_error_after_m": float(np.abs(x[:, :2] - P.pgt[:, :2]).mean()),
                 "options": ("Ceres defaults + parameter_tolerance 3e-3, max_solver_time 4 s (pose_graph.cpp:91-97)"
                             if not kw else "parameter_tolerance 1e-6, function_tolerance 1e-9, <= 50 iterations")}
            d["_x"] = x
            solve[name] = d
        ctx.graph_set_poses(P.pinit)
        out["solve"] = solve
    return out


DUMP_LIMIT_BYTES = 60 * 10 ** 6   # array data; with the .npy headers the files stay under 64 MB


def write_outputs(out_dir, arrays):
    """DIR/<name>.npy (float64) per array.  A dense H too large for DUMP_LIMIT_BYTES is replaced by
    a fixed, seeded sample of its entries: H_sample.npy (values) and H_sample_index.npy (flat
    row-major indices, exact in float64)."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, np.float64) for k, v in arrays.items()}
    H = arrays.pop("H")
    budget = DUMP_LIMIT_BYTES - sum(a.nbytes for a in arrays.values())
    if H.nbytes <= budget:
        arrays["H"] = H
    else:
        n = budget // 16
        idx = np.sort(np.random.default_rng(0).choice(H.size, n, replace=False))
        arrays["H_sample"] = H.reshape(-1)[idx]
        arrays["H_sample_index"] = idx.astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def single_rank_parity(P, torch, dist, world, rank):
    """N > 1: rank 0 evaluates the FULL problem on its own GPU (communicator suspended, every
    constraint local) and compares it with the sharded + exchanged result every rank holds."""
    ctx = P.ctx
    ctx.graph_set_poses(P.pinit)
    ok, cost, g, _ = ctx.graph_eval(P.n_nodes, want_H=False)        # sharded, all ranks
    sums = P.pg.getVisualizationEdgeResiduals()                      # per-constraint (local ones only)
    res = None
    dist.barrier()
    if rank == 0:
        ctx.comm_suspend(True)
        ok1, cost1, g1, H1 = ctx.graph_eval(P.n_nodes, want_H=True)
        ctx.comm_suspend(False)
    dist.barrier()
    ok2, cost2, g2, H2 = ctx.graph_eval(P.n_nodes, want_H=True)      # sharded again (tables rebuilt on rank 0)
    if rank == 0:
        sg = max(np.abs(g1).max(), 1e-300); sh = max(np.abs(H1).max(), 1e-300)
        rel = max(abs(cost2 - cost1) / max(abs(cost1), 1e-300), float(np.abs(g2 - g1).max() / sg),
                  float(np.abs(H2 - H1).max() / sh))
        res = {"parity_vs_single_rank": rel, "cost_equal": bool(abs(cost2 - cost1) <= 1e-12 * abs(cost1)),
               "cost_sharded": cost2, "cost_single_rank": cost1, "tolerance": 1e-12,
               "how": "rank 0 re-evaluates all constraints on one GPU (vgx_comm_suspend) and compares cost, "
                      "gradient and every H block with the exchanged result: max relative error"}
    return res


def run_b200(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = world
    wname = args.workload if args.workload != "auto" else ("config2" if world == 1 else "config4")
    w_main = workload_params(wname, args)
    want_c4_leg = (world == 1 and wname == "config2" and not args.no_extras and not args.no_config4)
    # scenes first: generation forks worker processes and must precede CUDA initialisation
    sc = build_scene(w_main, rank)
    w_c4 = workload_params("config4", args) if want_c4_leg else None
    sc_c4 = None
    if want_c4_leg:
        try:
            sc_c4 = build_scene(w_c4, rank)
        except Exception as e:  # pragma: no cover
            sys.stderr.write("config4 leg skipped: %r\n" % (e,))

    want_stream = (world == 1 and not args.no_extras and not args.no_stream)
    st_lidar = None
    if want_stream:
        try:
            st_lidar = build_stream("lidar", args.stream_scans, rank)
        except Exception as e:  # pragma: no cover
            sys.stderr.write("stream leg skipped: %r\n" % (e,))

    import torch
    import torch.distributed as dist
    from voxgraph_b200 import api
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    ctx = api.Context(local_rank)
    comm_kind = None
    if world > 1:
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid = torch.from_numpy(api.comm_unique_id()).cuda()
        dist.broadcast(uid, 0)
        ctx.comm_init(world, rank, uid.cpu().numpy())
        if os.environ.get("VGX_COMM", "p2p") == "p2p":
            # NVLink peer-memory exchange of the packed normal equations (CUDA IPC); NCCL stays
            # initialised as the fallback path (VGX_COMM=nccl selects it)
            def all_gather_bytes(h):
                t = torch.from_numpy(h).cuda()
                out = torch.zeros(world * 64, dtype=torch.uint8, device="cuda")
                dist.all_gather_into_tensor(out, t)
                return out.cpu().numpy()
            api.p2p_setup(ctx, world, rank, all_gather_bytes, capacity_doubles=1 << 20)
            comm_kind = "nvlink-p2p one-shot all-gather-reduce (CUDA IPC)"
        else:
            comm_kind = "ncclAllReduce"

    stream = torch.cuda.ExternalStream(ctx.stream_ptr)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    t_load0 = time.time()
    P = Problem(ctx, api, sc)
    M = measure(P, args, torch, dist, world, stream, want_outputs=bool(args.dump_outputs))
    ms_step = M["ms_per_step"]
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, M.pop("outputs"))

    parity = None
    if world > 1:
        parity = single_rank_parity(P, torch, dist, world, rank)

    # keep the GPU under the same evaluation load long enough for nvidia-smi (100 ms period) to
    # see it: the clocks line covers warm-up + the timed bracket + e2e + this sustained tail
    # (iteration count derived from the rank-reduced step time: every rank must issue the same
    # number of evaluations, each one contains a collective)
    n_tail = int(min(20000, max(50, 0.6 / max(ms_step * 1e-3, 1e-6))))
    for k in range(n_tail):
        ctx.graph_eval_async()
        if k % 50 == 49:
            ctx.synchronize()
    ctx.synchronize()
    clocks = sampler.stop(t_load0, time.time()) if sampler else None
    if clocks is not None:
        clocks["window"] = "upload + warm-up + timed bracket + e2e + solve + 0.6 s of the same evaluation loop"

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"]); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak = 6650.0; peak_src = "fallback 6.65 TB/s (MEASURED_PEAKS.json absent)"

    def roofline_of(Pm, Mm):
        achieved = Pm.r_local * ALGO_BYTES_PER_RESIDUAL / (Mm["kernel_ms"] * 1e-3) / 1e9
        return {"bound": "hbm", "kernel": "reg_reduce_kernel<true>", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_residual": ALGO_BYTES_PER_RESIDUAL,
                "residuals_per_launch": int(Pm.r_local), "kernel_ms": Mm["kernel_ms"],
                "kernel_share_of_step": Mm["kernel_ms"] / Mm["ms_per_step"] if Mm["ms_per_step"] > 0 else None,
                "other_kernels_ms_per_step": Mm["other_kernels_ms_per_step"],
                "step_breakdown_us_serialised": Mm.get("step_breakdown_us")}

    roofline = roofline_of(P, M)
    prof_traffic = os.path.join(ROOT, "profiles", "reg_reduce_traffic.json")
    if os.path.exists(prof_traffic) and wname == "config2":
        try:
            roofline["traffic"] = json.load(open(prof_traffic)).get("dram_bytes_per_launch")
        except Exception:
            pass

    e2e = M["e2e"]
    extras = {}
    cpu = None
    if "solve" in M:
        extras["solve"] = M["solve"]
    if rank == 0 and not args.no_extras:
        # ---------------- CPU baseline (pinned threads, median) + the restated reference's solve
        cpu = cpu_reference(sc, budget_s=args.cpu_seconds)
        if world == 1 and "solve" in M:
            from oracle import oracle as o
            nt = min(4, os.cpu_count() or 1)   # pose_graph.cpp:96 num_threads = 4
            for name, kw in (("reference_options", {}),
                             ("tight", dict(parameter_tolerance=1e-6, function_tolerance=1e-9,
                                            max_num_iterations=50, max_solver_time_s=60.0))):
                try:
                    g, _ = oracle_graph(sc)
                    rc, so = g.solve(o.solver_options(num_threads=nt, **kw))
                    d = M["solve"][name]
                    d["cpu_reference_solve_ms"] = so.total_time_s * 1e3
                    d["cpu_reference_iterations"] = so.iterations
                    d["cpu_reference_final_cost"] = so.final_cost
                    d["cpu_reference_threads"] = nt
                    d["max_pose_diff_vs_cpu_reference"] = float(np.abs(d["_x"] - g.poses()).max())
                except Exception as e:  # pragma: no cover
                    M["solve"][name]["cpu_reference_error"] = repr(e)
    if "solve" in M:
        ref_opts = M["solve"]["reference_options"]
        # the second half of the metric rides in a dict the driver keeps
        e2e["solve_ms"] = ref_opts["solve_ms"]
        e2e["lm_iterations"] = ref_opts["lm_iterations"]
        e2e["solve_unknowns"] = ref_opts["unknowns"]
        e2e["solve_final_cost"] = ref_opts["final_cost"]
        e2e["solve_ms_tight"] = M["solve"]["tight"]["solve_ms"]
        e2e["lm_iterations_tight"] = M["solve"]["tight"]["lm_iterations"]
        if "max_pose_diff_vs_cpu_reference" in ref_opts:
            e2e["max_pose_diff_vs_cpu_reference"] = ref_opts["max_pose_diff_vs_cpu_reference"]
            e2e["cpu_reference_solve_ms"] = ref_opts["cpu_reference_solve_ms"]
    if parity is not None:
        e2e["parity_vs_single_rank"] = parity["parity_vs_single_rank"]
        e2e["cost_equal"] = parity["cost_equal"]
        roofline["parity_vs_single_rank"] = parity["parity_vs_single_rank"]
        extras["parity"] = parity

    # ---------------- TSDF integration (HP1), configs[2]-shaped scan, rank 0, N = 1 only
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            extras["tsdf"] = tsdf_leg(ctx, sc, peak)
            e2e["tsdf_fast_updates_per_s_e2e"] = extras["tsdf"]["fast"]["updates_per_s_e2e"]
            e2e["tsdf_ray_ordered_updates_per_s_e2e"] = extras["tsdf"]["simple_ray_ordered"]["updates_per_s_e2e"]
        except Exception as e:  # pragma: no cover
            extras["tsdf"] = {"error": repr(e)}

    # ---------------- streaming leg (BASELINE configs[2]): integrate -> finish -> register online
    if st_lidar is not None and rank == 0:
        try:
            extras["stream"] = stream_leg(ctx, api, st_lidar, 0.15, 10, peak)
            e2e["stream_scans_per_s"] = extras["stream"]["scans_per_s_e2e"]
            e2e["stream_realtime_factor_vs_10hz"] = extras["stream"]["realtime_factor"]
            e2e["stream_updates_per_s_e2e"] = extras["stream"]["updates_per_s_e2e"]
        except Exception as e:  # pragma: no cover
            extras["stream"] = {"error": repr(e)}

    # ---------------- config4 leg at N = 1 (the strong-scaling curve's own first point)
    if sc_c4 is not None:
        try:
            P.free()
            P4 = Problem(ctx, api, sc_c4, id_base=100000)
            M4 = measure(P4, args, torch, dist, world, stream)
            c4 = {"workload": workload_config(w_c4, sc_c4, 1)["workload"], "value": M4["value"],
                  "unit": "residuals/s", "ms_per_step": M4["ms_per_step"],
                  "residuals_per_step": int(P4.r_global), "e2e_value": M4["e2e"]["value"],
                  "upload_s": P4.upload_s}
            if "solve" in M4:
                c4["solve_ms"] = M4["solve"]["reference_options"]["solve_ms"]
                c4["lm_iterations"] = M4["solve"]["reference_options"]["lm_iterations"]
                c4["solve_unknowns"] = M4["solve"]["reference_options"]["unknowns"]
                c4["solve_ms_tight"] = M4["solve"]["tight"]["solve_ms"]
            e2e["config4"] = c4
            r4 = roofline_of(P4, M4)
            roofline["config4"] = {k: r4[k] for k in ("achieved", "frac", "kernel_ms", "residuals_per_launch",
                                                      "kernel_share_of_step")}
            P4.free()
        except Exception as e:  # pragma: no cover
            e2e["config4"] = {"error": repr(e)}
    for d in M.get("solve", {}).values():
        d.pop("_x", None)

    if rank == 0:
        if parity is not None and not (parity["parity_vs_single_rank"] <= 1e-12):
            sys.stderr.write("PARITY FAILURE vs single rank: %r\n" % (parity,))
        line = {"metric": "registration_residuals_per_s", "value": M["value"], "unit": "residuals/s",
                "n_gpus": n_gpus, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "strong" if wname == "config4" else "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(w_main, sc, n_gpus),
                "residuals_per_step": int(P.r_global), "gpu_launches": M["gpu_launches"],
                "clocks": clocks, "e2e": e2e, "roofline": roofline,
                "cpu_baseline": ({k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample",
                                                       "value_4_threads", "value_best", "spread", "note")}
                                 if cpu else None),
                "collective": comm_kind, "upload_s": P.upload_s,
                "resident_bytes": {"points": int(P.r_global // 2 * 20 // max(len(sc.pairs), 1) * len(sc.submaps)),
                                   "reading_bricks_view": int(P.bricks_bytes)}}
        line.update(extras)
        _REAL_STDOUT.write(json.dumps(line) + "\n"); _REAL_STDOUT.flush()
    failed = parity is not None and not (parity["parity_vs_single_rank"] <= 1e-12)
    if world > 1:
        dist.barrier()      # tear the peer mappings down together
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    if failed:
        sys.exit(3)


def tsdf_leg(ctx, sc, peak):
    """HP1 on a configs[2]-shaped scan (64 x 1024 LiDAR): the integrator the reference runs (Fast) and
    the ray-ordered Simple path, next to the restated reference on the host."""
    from oracle import oracle as o
    from voxgraph_b200 import synth
    wpose = np.array([sc.poses_gt[0][0], sc.poses_gt[0][1], 1.2, 0.3])
    pts = synth.lidar_scan(sc.world, wpose, n_beams=64, n_azimuth=1024, seed=3, miss_range=40.0)
    T = synth.pose_to_T([0, 0, 0, 0])
    out = {"rays": int(pts.shape[0]), "scan": "64x1024 LiDAR, 0.20 m voxels, trunc 0.6 m, max ray 16 m",
           "algorithmic_bytes_per_update": ALGO_BYTES_PER_TSDF_UPDATE}
    for name, kw in (("simple_ray_ordered", dict(mode=0)), ("fast", dict(mode=1))):
        cfg = ctx.tsdf_config(**kw)
        ctx.submap_create(10 ** 6, 0.2, 16, 8192)
        ctx.tsdf_integrate(10 ** 6, T, pts, cfg)      # allocates the blocks (warm-up)
        ctx.profile_reset(); ctx.profile_enable(True)
        reps = 3
        for _ in range(reps):
            st = ctx.tsdf_integrate(10 ** 6, T, pts, cfg)
        ims, inn = ctx.profile_get(2); ams, ann = ctx.profile_get(3)
        ctx.profile_enable(False)
        t0 = time.time()
        for _ in range(reps):
            st = ctx.tsdf_integrate(10 ** 6, T, pts, cfg)
        wall = (time.time() - t0) / reps
        kms = (ims + ams) / reps
        lay = o.Layer(0.2, 16)
        oc = o.tsdf_config(mode=kw["mode"])
        o.tsdf_integrate(lay, oc, T, pts)
        tc = time.time(); so = o.tsdf_integrate(lay, oc, T, pts); cpu_s = time.time() - tc
        # voxblox runs integrator_threads = hardware_concurrency: multi-threaded restatement, median of 3
        cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        nt = max(1, min(cores, 64))
        lay_mt = o.Layer(0.2, 16)
        o.tsdf_integrate_mt(lay_mt, oc, T, pts, nt)
        mt = []
        for _ in range(3):
            tc = time.time(); smt = o.tsdf_integrate_mt(lay_mt, oc, T, pts, nt); mt.append(time.time() - tc)
        cpu_mt_s = float(np.median(mt))
        out[name] = {
            "voxel_updates_per_scan": int(st.voxel_updates), "rays_cast": int(st.rays_cast),
            "kernels_ms": kms,
            "updates_per_s_kernels": st.voxel_updates / (kms * 1e-3),
            "scan_ms_e2e_host_points": wall * 1e3,
            "updates_per_s_e2e": st.voxel_updates / wall,
            "achieved_gbs": st.voxel_updates * ALGO_BYTES_PER_TSDF_UPDATE / (kms * 1e-3) / 1e9,
            "frac_of_hbm_peak": st.voxel_updates * ALGO_BYTES_PER_TSDF_UPDATE / (kms * 1e-3) / 1e9 / peak,
            "saturated_batches": int(st.saturated_batches),
            "cpu_reference_scan_ms_1_thread": cpu_s * 1e3,
            "cpu_reference_updates_per_s_1_thread": so.voxel_updates / cpu_s,
            "cpu_reference_scan_ms_mt": cpu_mt_s * 1e3, "cpu_reference_threads_mt": nt,
            "cpu_reference_updates_per_s_mt": smt.voxel_updates / cpu_mt_s}
        ctx.submap_free(10 ** 6)
    return out


def main():
    args = parse_args()
    # Libraries (NCCL banner, torchrun) may print to stdout; the contract is ONE JSON line there.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "rgbd":
        run_rgbd(args)
    elif args.workload == "stream":
        run_stream(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
