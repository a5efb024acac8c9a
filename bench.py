#!/usr/bin/env python
"""bench.py — depth-frames/s (and Mvoxel-updates/s) of the semantic TSDF integrator hot path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload fast5|merged2|fast10] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one synthetic 640x480 depth+label frame (BASELINE.json
configs[1] by default: 5 cm voxels, 21 classes, `fast` integrator).  Every step integrates a DIFFERENT
frame of the synthetic trajectory into the same growing map (the frames are generated before the timed
region; for `value` they are already resident in HBM).  One JSON line is printed by rank 0.

  value     whole-job depth-frames/s with inputs resident in HBM (device entry point of the C-ABI),
            timed with CUDA events on the launching stream, max over ranks
  e2e       the same through the host-buffer C-ABI call (ksg_integrate_depth): pinned staging + H2D copy of
            depth+label and the D2H read of the frame counters inside the timed region
  roofline  tile-apply kernel: algorithmic bytes (updates * (34 + 8C) + pixels * 5) / its device time
  cpu_baseline  the reference's CPU path timed on this box's host cores: the faster of (a) the oracle port and (b) the reference's
            own integrator sources built against stand-in dependency headers (oracle/_ref), each at its best thread count
  --impl reference   times that CPU path alone and prints the same line shape

Multi-GPU (torchrun, one rank per GPU): the path shards by sequence - every rank integrates its own camera
stream into its own map (independent robots / sequences), no data-path collective; "scaling": "weak".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from kimera_semantics_b200 import synth  # noqa: E402
from kimera_semantics_b200.capi import (KSG_INTEGRATOR_FAST, KSG_INTEGRATOR_MERGED, default_config)  # noqa: E402

WORKLOADS = {
    # name: (integrator, width, height, voxel size, classes, max_updates, max_blocks)
    "fast5": (KSG_INTEGRATOR_FAST, 640, 480, 0.05, 21, 0, 8192),        # BASELINE.json configs[1] (headline)
    "merged2": (KSG_INTEGRATOR_MERGED, 640, 480, 0.02, 21, 80 << 20, 32768),  # configs[2]
    "merged5": (KSG_INTEGRATOR_MERGED, 640, 480, 0.05, 21, 16 << 20, 8192),
    "fast10": (KSG_INTEGRATOR_FAST, 320, 240, 0.10, 5, 0, 4096),        # configs[0] geometry
    "fast5_720p_c150": (KSG_INTEGRATOR_FAST, 1280, 720, 0.05, 150, 0, 2048),   # configs[3]: ADE20K-size label set, frame-per-GPU batches
    "merged1_4k_c40": (KSG_INTEGRATOR_MERGED, 3840, 2160, 0.01, 40, 1500 << 20, 65536),   # configs[4]: 4K / 1 cm, spatially sharded
}


def make_cfg(workload, device=0, threads=1):
    itype, w, h, vs, C, max_updates, max_blocks = WORKLOADS[workload]
    cfg = default_config(itype, vs, 16, C)
    cfg.dynamic_label[C - 1] = 1
    cfg.max_points = w * h
    cfg.max_updates = max_updates
    cfg.max_blocks = max_blocks
    cfg.device = device
    cfg.integrator_threads = threads
    return cfg


def gen_frames(workload, n, rank=0):
    _, w, h, _, C, _, _ = WORKLOADS[workload]
    cam = synth.make_camera(w, h)
    out = []
    for f in range(n):
        # every rank follows its own trajectory (phase shift) -> independent sequences
        T = synth.pose(f, phase=-2.967 + 0.37 * rank)
        depth, label, T = synth.frame(cam, f, C, seed=rank, T_G_C=T)
        out.append((depth, label, T))
    return cam, out


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []
        self._stop = threading.Event()
        self._th = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()

    def stop(self):
        self._stop.set()
        if self._th:
            self._th.join(timeout=6)
        sm = [float(s[1]) for s in self.samples if len(s) > 2 and s[1].replace(".", "").isdigit()]
        mx = [float(s[2]) for s in self.samples if len(s) > 2 and s[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for k, nme in enumerate(names):
                if len(s) > 5 + k and s[5 + k].lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


CPU_ARMS = {
    "port": "oracle port of the reference integrator (oracle/ks_oracle.cpp, timing build -O3 -march=x86-64-v3)",
    "reference": "the reference's own integrator sources (semantic_tsdf_integrator_{fast,merged}.cpp, semantic_integrator_base.cpp, "
                 "color.cpp) compiled -O3 -march=x86-64-v3 against stand-in Eigen/glog/voxblox headers (oracle/_ref, see oracle/ref_hybrid.cpp)",
}


def cpu_arms(workload):
    """Which CPU implementations can be timed on this box: the port always, the reference-source build when its prebuilt
    library travelled with the snapshot and the workload has the reference's compile-time 21 labels (common.h:27)."""
    arms = ["port"]
    try:
        from oracle import ref_py
        if ref_py.available(fast_build=True) and WORKLOADS[workload][4] == ref_py.load(fast_build=True).kref_num_labels():
            arms.append("reference")
    except Exception:
        pass
    return arms


class _ReferenceSourceArm:
    """Feeds depth+label frames to the reference boundary integratePointCloud(T_G_C, points_C, colors): back-projection and the
    label -> colour encoding happen outside the timed span, exactly as the ROS front end does them before the call."""

    def __init__(self, cfg, cam):
        from oracle.ref_py import RefHybridIntegrator
        self.integ = RefHybridIntegrator(cfg, fast_build=True)
        self.cam = cam
        self.pal = np.array([[cfg.label_color[l][k] for k in range(4)] for l in range(256)], np.uint8)

    def integrate_depth(self, T, depth, label, K):
        xyz, pix = synth.backproject(depth, self.cam)
        self.integ.integrate_points(T, xyz, rgba=np.ascontiguousarray(self.pal[label.reshape(-1)[pix]]))
        return None

    def last_integrate_seconds(self):
        return self.integ.last_integrate_seconds()

    def export(self):
        return self.integ.export()

    def close(self):
        self.integ.close()


def make_cpu_integrator(arm, workload, cam, threads):
    cfg = make_cfg(workload, threads=threads)
    if arm == "reference":
        return _ReferenceSourceArm(cfg, cam)
    from oracle.oracle_py import OracleIntegrator
    return OracleIntegrator(cfg, fast_build=True)   # merged: bundle order of cfg (default = the reference's unordered_map walk)


def cpu_baseline(workload, frames, cam, threads, budget_s=20.0, max_frames=40, arm="port", updates_per_frame=None):
    """One CPU arm on a bounded sample of the same frames. Timed span = integratePointCloud body."""
    integ = make_cpu_integrator(arm, workload, cam, threads)
    t_total, updates, n = 0.0, 0, 0
    t0 = time.time()
    for depth, label, T in frames[:max_frames]:
        st = integ.integrate_depth(T, depth, label, cam.K)
        t_total += integ.last_integrate_seconds()
        if st is not None:
            updates += st.voxel_updates
        elif updates_per_frame is not None:   # the reference's code does not count; the port's count of the same frame applies
            updates += updates_per_frame[n]
        n += 1
        if time.time() - t0 > budget_s:
            break
    integ.close()
    return {"frames": n, "seconds": t_total, "fps": n / t_total if t_total > 0 else 0.0,
            "mupdates_per_s": updates / t_total / 1e6 if t_total > 0 else 0.0}


def best_cpu_arm(workload, frames, cam):
    """The reference spawns config.integrator_threads threads per frame (default hardware_concurrency) that contend on 4096
    striped mutexes and two atomic hash sets; on many-core hosts that is slower than a few threads.  Calibrate every available
    arm on a few frames at several thread counts and keep the fastest (arm, threads) pair - the most favourable CPU number."""
    cores = os.cpu_count() or 1
    cands = sorted({1, 4, 16, cores} & set(range(1, cores + 1)) | {1})
    res = {}
    for arm in cpu_arms(workload):
        for t in cands:
            res[(arm, t)] = cpu_baseline(workload, frames, cam, t, budget_s=5.0, max_frames=4, arm=arm)["fps"]
    best = max(res, key=res.get)
    return best[0], best[1], {f"{a}@{t}": v for (a, t), v in res.items()}


def ncu_traffic(workload, tag="apply"):
    """dram__bytes_read.sum + dram__bytes_write.sum of one frame's launches of the phase `tag` ("apply": the update kernel(s), "solve3": the
    persistent solve kernel of `fast`, "sort": the radix sort passes of `merged`), from the newest committed `ncu --set full` capture
    (profiles/r*/prof_<tag>_<workload>*.raw.csv; one row per launch, summed) -> (bytes or None, which capture).  A capture describes the
    kernels of the commit it was taken at; the directory carries the round."""
    import csv
    import glob
    cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*", f"prof_{tag}_{workload}*.raw.csv")))
    for path in reversed(cands):
        try:
            rows = [r for r in csv.reader(open(path)) if r]
            hdr, units, launches = rows[0], rows[1], rows[2:]
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            tot = 0.0
            for vals in launches:
                for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    k = hdr.index(name)
                    tot += float(vals[k].replace(",", "")) * scale.get(units[k], 1.0)
            return tot, os.path.relpath(path, ROOT) + f" (ncu --set full, {len(launches)} launch(es) of one frame)"
        except Exception:
            continue
    return None, None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, exp, seed=0):
    """--dump-outputs: the map a caller of the timed path holds after its last step, as DIR/<name>.npy in float32 / float64, at most
    DUMP_BYTES in all.  Blocks are sorted by block index, so that the files do not depend on allocation order; every block index is
    written, the voxel fields for a fixed, seeded sample of the observed voxels (all of them when they fit)."""
    os.makedirs(out_dir, exist_ok=True)
    order = np.lexsort(exp["block_index"].T[::-1])
    blocks = exp["block_index"][order].astype(np.float64)
    b, v = np.nonzero(exp["tsdf_weight"][order] > 0)
    C = exp["sem_priors"].shape[-1]
    per_voxel = 8 * 2 + 4 * (3 + 4 + 4 + C)
    n_max = (DUMP_BYTES - blocks.nbytes - 8) // per_voxel
    observed = len(b)
    if observed > n_max:
        keep = np.sort(np.random.default_rng(seed).choice(observed, n_max, replace=False))
        b, v = b[keep], v[keep]
    rows = order[b]
    arrays = {"block_index": blocks, "observed_voxels": np.array([observed], np.float64),
              "voxel_index": np.stack([b, v], axis=1).astype(np.float64),     # (row of block_index, voxel within the block)
              "tsdf_distance": exp["tsdf_distance"][rows, v], "tsdf_weight": exp["tsdf_weight"][rows, v],
              "tsdf_rgba": exp["tsdf_rgba"][rows, v].astype(np.float32), "sem_label": exp["sem_label"][rows, v].astype(np.float32),
              "sem_priors": exp["sem_priors"][rows, v], "sem_rgba": exp["sem_rgba"][rows, v].astype(np.float32)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path - the faster of the oracle port and the reference-source
    build (oracle/_ref), at the thread count that is fastest on this host."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    itype, w, h, vs, C, _, _ = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    n = args.warmup + args.steps
    cam, frames = gen_frames(args.workload, n)
    arm, threads, calib = best_cpu_arm(args.workload, frames[args.warmup:], cam)
    integ = make_cpu_integrator(arm, args.workload, cam, threads)
    counter = make_cpu_integrator("port", args.workload, cam, 1) if arm != "port" else None   # untimed: counts voxel updates
    t_total, updates = 0.0, 0
    for i, (depth, label, T) in enumerate(frames):
        st = integ.integrate_depth(T, depth, label, cam.K)
        if counter is not None:
            st = counter.integrate_depth(T, depth, label, cam.K)
        if i >= args.warmup:
            t_total += integ.last_integrate_seconds()
            updates += st.voxel_updates
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, integ.export())
    integ.close()
    fps = args.steps / t_total
    line = {
        "impl": "reference", "metric": "depth_frames_per_s", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "mvoxel_updates_per_s": updates / t_total / 1e6,
        "config": {"workload": f"{w}x{h} depth+label stream, {vs * 100:.0f} cm voxels, {C} classes, "
                               f"{'fast' if itype == KSG_INTEGRATOR_FAST else 'merged'} integrator (BASELINE.json configs)",
                   "name": args.workload},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": arm, "host_cores": cores,
                         "implementation": CPU_ARMS[arm], "calibration_fps": calib,
                         "sample": f"{args.steps} frames after {args.warmup} warm-up; fastest (implementation, integrator_threads) pair of the "
                                   f"calibration = {arm} with {threads} threads (the host has {cores} cores)"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def shim_e2e(workload, frames, cam, warmup=5, timed=30):
    """Throughput through the drop-in C++ classes (SemanticTsdfIntegratorFactory::create + integratePointCloud on host std::vector clouds),
    eager (the reference's contract: host layers updated when the call returns) and lazy layer sync - kimera_semantics_b200/cpp/shim_bench."""
    import tempfile
    exe = os.path.join(ROOT, "kimera_semantics_b200", "cpp", "shim_bench")
    itype, w, h, vs, C, max_updates, max_blocks = WORKLOADS[workload]
    if not os.path.exists(exe) or C != 21:       # the shim keeps the reference's compile-time label count (common.h:27)
        return None
    cfg = make_cfg(workload)
    pal = np.array([[cfg.label_color[l][k] for k in range(4)] for l in range(C)], np.uint8)
    n = min(len(frames), warmup + timed)
    out = {}
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "frames.bin")
        with open(path, "wb") as f:
            f.write(np.int32(n).tobytes()); f.write(np.float32(vs).tobytes()); f.write(np.int32(16).tobytes())
            f.write(np.int32(C).tobytes())
            for l in range(C):
                f.write(bytes([int(pal[l, 0]), int(pal[l, 1]), int(pal[l, 2]), int(pal[l, 3]), l]))
            f.write(np.int32(1).tobytes()); f.write(bytes([C - 1]))
            for depth, label, T in frames[:n]:
                xyz, pix = synth.backproject(depth, cam)
                f.write(np.int32(len(xyz)).tobytes())
                f.write(np.ascontiguousarray(T, np.float32).tobytes())
                f.write(np.ascontiguousarray(xyz, np.float32).tobytes())
                f.write(np.ascontiguousarray(pal[label.reshape(-1)[pix]]).tobytes())
        env = dict(os.environ, KSG_MAX_POINTS=str(w * h), KSG_MAX_BLOCKS=str(max_blocks))
        if max_updates:
            env["KSG_MAX_UPDATES"] = str(max_updates)
        for mode in ("eager", "lazy"):
            try:
                r = subprocess.run([exe, "fast" if itype == KSG_INTEGRATOR_FAST else "merged", path, str(warmup), mode], capture_output=True, text=True,
                                   env=env, timeout=600)
                out[mode] = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"error": (r.stderr or r.stdout)[-300:]}
            except Exception as e:      # noqa: BLE001
                out[mode] = {"error": str(e)}
    return out


def measure(args, workload, steps, warmup, ctx, with_cpu, profile_frames):
    """Every leg of one workload on this rank; rank 0 gets the result dictionary (the others None)."""
    import torch
    import torch.distributed as dist
    from kimera_semantics_b200.capi import Integrator
    world, rank, local_rank = ctx["world"], ctx["rank"], ctx["local_rank"]
    itype, w, h, vs, C, _, _ = WORKLOADS[workload]
    n = warmup + steps
    spatial = args.sharding == "spatial" and world > 1
    # sequence mode (replicas): every rank integrates the SAME synthetic stream into its own map - weak scaling means fixed work per GPU
    # (rank-specific trajectories differ by up to 10 % in voxel updates per frame, which the max over ranks then reports as lost efficiency:
    # profiles/r02/bench_seq_fast5_n8.json, 18.4 K frames/s = 0.92 x 8 x the 1-GPU rate); KSG_BENCH_RANK_STREAMS=1 restores one trajectory per rank
    cam, frames = gen_frames(workload, n, rank if (not spatial and os.environ.get("KSG_BENCH_RANK_STREAMS")) else 0)
    P = w * h

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident leg (value) ----------------
    d_depth = [torch.from_numpy(f[0]).cuda() for f in frames]
    d_label = [torch.from_numpy(f[1]).cuda() for f in frames]
    total_in = sum(t.numel() * t.element_size() for t in d_depth + d_label)
    cfg = make_cfg(workload, device=local_rank)
    cfg.merged_bundle_order = 1 if args.merged_bundle_order == "libstdcxx" else 0
    cfg.hot_voxel_mode = int(args.hot_voxels)
    if spatial:
        cfg.shard_rank, cfg.shard_count = rank, world
    integ = Integrator(cfg)
    # a real (non-default) stream: the library treats a NULL stream handle as "use my own stream", on which torch events would not be ordered
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0
    for i in range(warmup):
        integ.integrate_depth_device(frames[i][2], d_depth[i].data_ptr(), d_label[i].data_ptr(), w, h, cam.K, stream)
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    integ.set_profiling(False)  # resets the launch counters
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # timed region: K frames enqueued back to back on the launching stream.  No per-frame statistics are requested, so the `fast`
    # driver never blocks the host inside the region (its frame has no read-back); the voxel-update count of exactly these frames
    # is taken from an identical untimed replay below.
    ev0.record(tstream)
    for i in range(warmup, n):
        integ.integrate_depth_device(frames[i][2], d_depth[i].data_ptr(), d_label[i].data_ptr(), w, h, cam.K, stream)
    ev1.record(tstream)
    barrier()
    integ.sync()
    ms = ev0.elapsed_time(ev1)
    prof = integ.get_profile()
    launches, libcalls = prof["kernel_launches"], prof["library_calls"]
    clocks = sampler.stop() if rank == 0 else None
    blocks = integ.num_blocks()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, integ.export())
    if args.quick:
        integ.close()
        return {"workload": workload, "value": steps / (ms / 1e3), "ms_per_step": ms / steps, "quick": True,
                "env": {k: v for k, v in os.environ.items() if k.startswith("KSG_")}}

    # ---------------- per-phase profiling pass + untimed replay of the timed frames (separate map, not part of `value`) ----------------
    integ.close()
    integ = Integrator(cfg)
    npf = min(profile_frames, steps)
    for i in range(warmup):
        integ.integrate_depth_device(frames[i][2], d_depth[i].data_ptr(), d_label[i].data_ptr(), w, h, cam.K, stream)
    integ.set_profiling(True)
    p_updates = 0
    timeline = None
    for i in range(warmup, warmup + npf):
        st = integ.integrate_depth_device(frames[i][2], d_depth[i].data_ptr(), d_label[i].data_ptr(), w, h, cam.K, stream, want_stats=True)
        p_updates += st.voxel_updates
    if itype == KSG_INTEGRATOR_FAST:
        timeline = integ.fast_timeline()
    prof = integ.get_profile()
    integ.set_profiling(False)
    updates = p_updates
    for i in range(warmup + npf, n):       # rest of the replay: same frames as the timed region -> their voxel updates
        st = integ.integrate_depth_device(frames[i][2], d_depth[i].data_ptr(), d_label[i].data_ptr(), w, h, cam.K, stream, want_stats=True)
        updates += st.voxel_updates
    integ.close()
    t = torch.tensor([ms, float(updates)], device="cuda", dtype=torch.float64)
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms, updates_all = float(tmax[0]), float(tsum[1])
    else:
        updates_all = float(updates)
    jobs = 1 if spatial else world          # spatial: every rank works on the same frames
    if spatial:
        updates_all = float(updates)
    value = jobs * steps / (ms / 1e3)
    mups = updates_all / (ms / 1e3) / 1e6
    nprof = max(1, prof["frames"])
    phase_ms = {k: prof[k] / nprof for k in Integrator.PHASES}
    alg_bytes = (p_updates / max(1, npf)) * (34 + 8 * C) + P * 5
    peak, peak_kind = peaks()
    # the kernel that carries the roofline number: the phase with the largest share of the frame
    kernel_of_phase = ({"classify+start_set": "k_fast_count + k_fast_classify + k_fast_start_eval (+ compaction / ray set-up inside k_fast_solve3)",
                        "fixpoint|bundling": "k_fast_solve3 (observed-set sweeps)", "ray_emit": "k_fast_solve3 (table commit + block allocation)",
                        "record_sort": "k_fast_solve3 (records -> tile segments)", "alloc+tile_heads": "-", "tile_apply": "k_tile_apply_fast"}
                       if itype == KSG_INTEGRATOR_FAST else
                       {"classify+start_set": "k_classify", "fixpoint|bundling": "bundle sort + k_bundle_order + k_bundle_merge", "ray_emit": "k_emit_merged",
                        "record_sort": "cub::DeviceRadixSort (stable, voxel bits only)", "alloc+tile_heads": "k_block_init + k_voxel_heads",
                        "tile_apply": "k_voxel_apply_long + k_voxel_apply_short (+ hot-voxel pre-pass)"})
    shares = {k: v for k, v in phase_ms.items() if k != "frame"}
    top_phase = max(shares, key=shares.get)
    top_ms = shares[top_phase]
    apply_ms = phase_ms["tile_apply"]
    frame_ms = phase_ms["frame"] if phase_ms["frame"] > 0 else ms / steps
    ach = lambda t_ms: alg_bytes / (t_ms / 1e3) / 1e9 if t_ms > 0 else 0.0

    # ---------------- end-to-end legs (host buffers through the C-ABI) ----------------
    barrier()
    # the step's inputs live in page-locked host memory (the contract's "pinned host memory"); the library copies from it
    pin_d = [torch.from_numpy(f[0]).pin_memory() for f in frames]
    pin_l = [torch.from_numpy(f[1]).pin_memory() for f in frames]
    hd = [t.numpy() for t in pin_d]
    hl = [t.numpy() for t in pin_l]
    e2e = {}
    for mode in ("pipelined", "sync"):
        passes = []
        for _pass in range(2):   # two identical passes of exactly K timed steps each (fresh map); the faster one is reported:
            integ = Integrator(cfg)   # the box is shared and a single ~70 ms host stall triples a 75 ms wall-clock region
            got = []
            if spatial:
                # rank 0 owns the camera stream: H2D on rank 0, NCCL broadcast of depth + label to every rank, then all ranks integrate
                buf_d = torch.empty((h, w), dtype=torch.float32, device="cuda")
                buf_l = torch.empty((h, w), dtype=torch.uint8, device="cuda")

                def run(lo, hi):
                    for i in range(lo, hi):
                        if rank == 0:
                            buf_d.copy_(pin_d[i], non_blocking=True)
                            buf_l.copy_(pin_l[i], non_blocking=True)
                        dist.broadcast(buf_d, 0)
                        dist.broadcast(buf_l, 0)
                        got.append(integ.integrate_depth_device(frames[i][2], buf_d.data_ptr(), buf_l.data_ptr(), w, h, cam.K, stream, want_stats=True))
            elif mode == "sync":
                def run(lo, hi):      # the reference's calling convention: the call returns when the frame is integrated
                    for i in range(lo, hi):
                        got.append(integ.integrate_depth(frames[i][2], hd[i], hl[i], cam.K))
            else:
                def run(lo, hi):      # camera-stream convention: submit frame i, then collect frame i-1 (its H2D overlaps frame i-1's kernels)
                    for i in range(lo, hi):
                        integ.integrate_depth_async(frames[i][2], hd[i], hl[i], cam.K)
                        if i > lo:
                            got.append(integ.wait_frame())
                    got.append(integ.wait_frame())
            run(0, warmup)
            barrier()
            t0 = time.perf_counter()
            run(warmup, n)
            integ.sync()
            passes.append(time.perf_counter() - t0)
            integ.close()
        te = torch.tensor([min(passes)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e[mode] = {"value": jobs * steps / float(te[0]), "pass_seconds": passes}
        if spatial:
            e2e["sync"] = e2e[mode]
            break

    # ---------------- several independent sequences on ONE GPU (how far the machine is from full at this frame size) ----------------
    multi = None
    if world == 1 and args.sequences_per_gpu > 1 and itype == KSG_INTEGRATOR_FAST:
        K = args.sequences_per_gpu
        integs = [Integrator(cfg) for _ in range(K)]
        streams = [torch.cuda.Stream() for _ in range(K)]
        for i in range(warmup):
            for k in range(K):
                integs[k].integrate_depth_device(frames[i][2], d_depth[i].data_ptr(), d_label[i].data_ptr(), w, h, cam.K, streams[k].cuda_stream)
        torch.cuda.synchronize()
        e0 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        e1 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        t0 = time.perf_counter()
        for k in range(K):
            e0[k].record(streams[k])
        for i in range(warmup, n):
            for k in range(K):
                integs[k].integrate_depth_device(frames[i][2], d_depth[i].data_ptr(), d_label[i].data_ptr(), w, h, cam.K, streams[k].cuda_stream)
        for k in range(K):
            e1[k].record(streams[k])
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        span = max(e0[0].elapsed_time(e1[k]) for k in range(K))
        for it in integs:
            it.sync()
            it.close()
        multi = {"sequences": K, "value": K * steps / (span / 1e3), "unit": "frames/s", "wall_value": K * steps / wall,
                 "note": "K integrators (own map each) fed round-robin on K streams of one GPU; device time from the first stream's start to the last stream's end"}

    if rank != 0:
        return None
    cpu = None
    if with_cpu:
        cores = os.cpu_count() or 1
        arm, threads, calib = best_cpu_arm(workload, frames[warmup:], cam)
        c_all = cpu_baseline(workload, frames[warmup:], cam, threads, arm=arm)
        cpu = {"value": c_all["fps"], "unit": "frames/s", "cores": threads, "kind": arm, "host_cores": cores,
               "implementation": CPU_ARMS[arm],
               "sample": f"{c_all['frames']} frames of the same stream (from the first timed frame, empty map); fastest (implementation, "
                         f"integrator_threads) pair of the calibration = {arm} with {threads} threads",
               "calibration_fps": calib}
        if arm == "port":
            cpu["mvoxel_updates_per_s"] = c_all["mupdates_per_s"]
    head = e2e.get("pipelined", e2e["sync"])
    tag_of_phase = ({"tile_apply": "apply"} if itype == KSG_INTEGRATOR_FAST else {"tile_apply": "apply", "record_sort": "sort"})
    traffic, traffic_src = ncu_traffic(workload, tag_of_phase.get(top_phase, "solve3" if itype == KSG_INTEGRATOR_FAST else top_phase))
    shim = shim_e2e(workload, frames[warmup:], cam) if (world == 1 and args.shim_e2e) else None
    return {
        "metric": "depth_frames_per_s", "value": value, "unit": "frames/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong" if spatial else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "mvoxel_updates_per_s": mups,
        "config": {"workload": f"{w}x{h} depth+label stream, {vs * 100:.0f} cm voxels, {C} classes, "
                               f"{'fast' if itype == KSG_INTEGRATOR_FAST else 'merged'} integrator (BASELINE.json configs)",
                   "name": workload, "voxels_per_side": 16, "frames_distinct": n, "merged_bundle_order": args.merged_bundle_order,
                   "hot_voxel_mode": int(args.hot_voxels),
                   "l2_policy": f"every step reads a different frame ({total_in / 1e6:.0f} MB of inputs cycled, larger than the 126 MB L2 "
                                "when steps >= 90) and a different part of the map; no explicit flush",
                   "parallelism": ("one map spatially sharded by tile owner over the GPUs; frames broadcast from rank 0 with NCCL" if spatial
                                   else "one sequence + map per GPU (the same synthetic stream on every rank), no collective") if world > 1 else "single GPU",
                   "map_blocks_after_run": blocks},
        "clocks": clocks,
        "e2e": {"value": head["value"], "unit": "frames/s", "h2d_bytes_per_step": P * 5,
                # fast: one copy of the frame counters (152 B) + the driver state with the solve kernel's time marks (568 B) per frame;
                # merged: the frame counters twice (record count for the sort, end of frame)
                "d2h_bytes_per_step": 152 + 568 if itype == KSG_INTEGRATOR_FAST else 2 * 152,
                "mode": "pipelined" if "pipelined" in e2e else "sync",
                "sync_value": e2e["sync"]["value"],
                "note": "host frames in page-locked memory through the C-ABI.  `value`: ksg_integrate_depth_async + ksg_wait_frame - frame i is "
                        "submitted (H2D of depth+label on a copy stream, then its kernels), then the statistics of frame i-1 are read back "
                        "(one D2H of the counter blocks per step); `sync_value`: ksg_integrate_depth, which returns when the frame is "
                        "integrated (the reference's calling convention).  Wall clock, faster of two identical K-step passes",
                "pass_seconds": head["pass_seconds"], "sync_pass_seconds": e2e["sync"]["pass_seconds"]},
        "gpu_launches": int(launches),
        "library_calls": int(libcalls),
        "multi_sequence": multi,
        "e2e_shim": None if shim is None else {
            "eager": shim.get("eager"), "lazy": shim.get("lazy"), "unit": "frames/s (field fps)",
            "note": "the reference's own call: SemanticTsdfIntegratorFactory::create + integratePointCloud(T_G_C, points_C, colors) on host clouds "
                    "through the C++ drop-in classes; eager = host Layer<TsdfVoxel> / Layer<SemanticVoxel> refreshed inside every call (the "
                    "reference's contract), lazy = refreshed once at the end (inside the measured span); clouds are back-projected before timing"},
        "roofline": {"bound": "hbm", "achieved": ach(top_ms), "peak": peak, "unit": "GB/s", "frac": ach(top_ms) / peak if peak else None,
                     "kernel": kernel_of_phase[top_phase], "phase": top_phase, "kernel_ms": top_ms,
                     "frame_frac": ach(frame_ms) / peak if peak else None, "frame_ms": frame_ms,
                     "tile_apply_frac": ach(apply_ms) / peak if peak and apply_ms > 0 else None, "tile_apply_ms": apply_ms,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_kind": peak_kind,
                     "algorithmic_bytes_per_launch": alg_bytes,
                     "note": "algorithmic bytes of one frame = updates * (34 + 8 C) + pixels * 5 (SURVEY.md 8d); `frac` divides them by the duration of "
                             "the phase with the largest share of the frame (`kernel`), `frame_frac` by the whole frame, `tile_apply_frac` by the update "
                             "kernel alone; durations are device-timed inside the library (CUDA events; clock64 marks inside the persistent kernel)",
                     "phase_ms_per_frame": phase_ms,
                     "solve_kernel_timeline_last_profiled_frame": timeline},
        "cpu_baseline": cpu,
    }


def measure_frame_batches(args, workload, steps, warmup, ctx):
    """--sharding frames: ONE camera stream, batches of N frames, one frame per GPU (SURVEY.md 8e row 1, BASELINE configs[3]).  Every rank
    holds a replica of the map; per batch it integrates its frame into an EMPTY delta map, the deltas (blocks in pool layout + block keys)
    are all-gathered with NCCL, and every rank merges the N deltas into its replica in frame order (ksg_merge_blocks_device).  A step = one
    batch = N frames.  Rank r's delta integrator is ONE integrator object for the whole run (frames r, r + N, ...) whose layers are emptied
    between its frames (ksg_clear_map = Layer::removeAllBlocks on a live reference integrator)."""
    import torch
    import torch.distributed as dist
    from kimera_semantics_b200.capi import Integrator
    world, rank, local_rank = ctx["world"], ctx["rank"], ctx["local_rank"]
    itype, w, h, vs, C, _, _ = WORKLOADS[workload]
    nb_batches = warmup + steps
    cam = synth.make_camera(w, h)
    mine = []
    for k in range(nb_batches):                       # frame k * N + rank of the single trajectory
        f = k * world + rank
        depth, label, T = synth.frame(cam, f, C, seed=0, T_G_C=synth.pose(f, phase=-2.967))
        mine.append((torch.from_numpy(depth).cuda(), torch.from_numpy(label).cuda(), T))
    cfg = make_cfg(workload, device=local_rank)
    base, delta = Integrator(cfg), Integrator(cfg)
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    _, stride, _, _ = delta.device_map_view()
    # `fast`: voxel-granular deltas (the update log of the frame = exactly the voxels of the delta map: 32 + 4 C bytes per touched voxel);
    # `merged` (no update log): whole blocks in pool layout
    by_voxels = itype == KSG_INTEGRATOR_FAST and not os.environ.get("KSG_FRAMES_BY_BLOCKS")
    if by_voxels:
        delta.set_update_log(max(1 << 18, w * h))
        stride = 32 + 4 * C
    cap_blocks = 0
    send_pool = recv_pool = send_keys = recv_keys = None
    counts = torch.zeros(world, dtype=torch.int64, device="cuda")
    t_int = t_xchg = t_merge = 0.0
    bytes_moved = 0
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(4)]

    def one_batch(k, timed):
        nonlocal cap_blocks, send_pool, recv_pool, send_keys, recv_keys, t_int, t_xchg, t_merge, bytes_moved
        d, l, T = mine[k]
        evs[0].record(tstream)
        delta.clear_map()       # empties the delta map, keeps the integrator (its per-scan approximate sets) - see ksg_clear_map
        delta.integrate_depth_device(T, d.data_ptr(), l.data_ptr(), w, h, cam.K, stream)
        nb = delta.update_log_size() if by_voxels else delta.device_map_view()[0]
        evs[1].record(tstream)
        mine_n = torch.tensor([nb], dtype=torch.int64, device="cuda")
        dist.all_gather_into_tensor(counts, mine_n)
        cs = [int(x) for x in counts.tolist()]
        mx = max(cs)
        if mx > cap_blocks:
            cap_blocks = int(mx * 1.25) + 8
            send_pool = torch.empty(cap_blocks * stride, dtype=torch.uint8, device="cuda")
            recv_pool = torch.empty(world * cap_blocks * stride, dtype=torch.uint8, device="cuda")
            send_keys = torch.empty(cap_blocks, dtype=torch.int64, device="cuda")
            recv_keys = torch.empty(world * cap_blocks, dtype=torch.int64, device="cuda")
        if by_voxels:
            # send_pool = [mx entries of 32 B | mx rows of C floats]; the gathered buffer keeps that layout per rank, so entries and rows of
            # rank g start at g * mx * stride and g * mx * stride + mx * 32: two all-gathers keep both arrays dense for the merge
            heads_s, rows_s = send_pool[: mx * 32], send_pool[cap_blocks * 32: cap_blocks * 32 + mx * 4 * C]
            heads_r, rows_r = recv_pool[: world * mx * 32], recv_pool[world * cap_blocks * 32: world * cap_blocks * 32 + world * mx * 4 * C]
            delta.copy_update_log_device(heads_s.data_ptr(), rows_s.data_ptr(), mx, stream)
            dist.all_gather_into_tensor(heads_r, heads_s)
            dist.all_gather_into_tensor(rows_r, rows_s)
            evs[2].record(tstream)
            base.merge_voxels_device(cs, mx, heads_r.data_ptr(), rows_r.data_ptr(), stream)      # the N deltas in frame order, one call
        else:
            delta.copy_map_device(send_pool.data_ptr(), send_keys.data_ptr(), stream)
            sp, rp = send_pool[: mx * stride], recv_pool[: world * mx * stride]
            sk, rk = send_keys[:mx], recv_keys[: world * mx]
            dist.all_gather_into_tensor(rp, sp)
            dist.all_gather_into_tensor(rk, sk)
            evs[2].record(tstream)
            for g in range(world):                      # frame order
                base.merge_blocks_device(cs[g], rk[g * mx:].data_ptr(), rp[g * mx * stride:].data_ptr(), stream)
        evs[3].record(tstream)
        torch.cuda.synchronize()
        if timed:
            t_int += evs[0].elapsed_time(evs[1]); t_xchg += evs[1].elapsed_time(evs[2]); t_merge += evs[2].elapsed_time(evs[3])
            bytes_moved += world * mx * (stride + 8)

    for k in range(warmup):
        one_batch(k, False)
    torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(tstream)
    for k in range(warmup, nb_batches):
        one_batch(k, True)
    e1.record(tstream)
    torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms, wall * 1e3], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, wall_ms = float(t[0]), float(t[1])
    blocks = base.num_blocks()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, base.export())
    base.close(); delta.close()
    if rank != 0:
        return None
    frames_total = steps * world
    return {
        "metric": "depth_frames_per_s", "value": frames_total / (ms / 1e3), "unit": "frames/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{w}x{h} depth+label stream, {vs * 100:.0f} cm voxels, {C} classes, "
                               f"{'fast' if itype == KSG_INTEGRATOR_FAST else 'merged'} integrator, batches of {world} frames, one frame per GPU (BASELINE.json configs[3] shape)",
                   "name": workload, "parallelism": "frame-per-GPU batches: delta maps all-gathered with NCCL, merged into every rank's replica in frame order",
                   "map_blocks_after_run": blocks},
        "e2e": {"value": frames_total / (wall_ms / 1e3), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 152 * (1 + world),
                "note": "wall clock of the same loop (frames resident on the device; the per-batch host work - block counts, launches - is inside)"},
        "collective": {"kind": "ncclAllGather (torch.distributed all_gather_into_tensor) of " +
                               ("the frames' update logs: one 32-byte entry + C floats per touched voxel" if by_voxels else "block keys + blocks in pool layout"),
                       "bytes_per_step": bytes_moved / max(1, steps),
                       "limiting": ("integration of the own frame; the exchange is %d B per touched voxel" % stride) if by_voxels
                                   else "the all-gather of whole blocks: block_stride = %d B at C = %d" % (stride, C)},
        "phase_ms_per_step": {"integrate_own_frame": t_int / steps, "all_gather": t_xchg / steps, "merge_all_deltas": t_merge / steps},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--workload", default="fast5", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--hot-voxels", type=int, default=0, choices=[0, 1, 2],
                    help="merged workloads: ksg_config.hot_voxel_mode (1 = parallel pre-pass for the semantic rows of hot voxels, 2 = + TSDF fixed-point check)")
    ap.add_argument("--merged-bundle-order", default="libstdcxx", choices=["canonical", "libstdcxx"],
                    help="merged workloads: bundle order (ksg_config.merged_bundle_order); libstdcxx = the reference's unordered_map order")
    ap.add_argument("--sharding", default="sequence", choices=["sequence", "spatial", "frames"],
                    help="N > 1: sequence = one stream + map per rank (weak scaling, default); spatial = ONE stream and map, every rank "
                         "receives every frame (NCCL broadcast from rank 0) and applies only the tiles it owns (strong scaling); frames = ONE "
                         "stream, batches of N frames, one frame per GPU into an empty delta map, NCCL all-gather of the deltas, every rank "
                         "merges them into its replica of the map in frame order (SURVEY.md 8e row 1, BASELINE configs[3])")
    ap.add_argument("--profile-frames", type=int, default=20, help="frames of the separate per-phase profiling pass")
    ap.add_argument("--sequences-per-gpu", type=int, default=4, help="N = 1, fast: also measure K independent sequences on one GPU (0/1: skip)")
    ap.add_argument("--quick", action="store_true", help="development aid: only the device-resident `value` leg, printed as a short line")
    ap.add_argument("--shim-e2e", type=int, default=1, help="N = 1: also time the C++ drop-in classes end to end (eager / lazy layer sync); 0 = skip")
    ap.add_argument("--extra-workloads", default="merged2", help="comma list of further workloads measured (briefly) into `workloads` at N = 1; '' = none")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the map they built (rank 0's) as DIR/<name>.npy: every block index and the voxel "
                         "fields of a seeded sample of the observed voxels, at most 64 MB; the inputs are the same on every run")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the integrator has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # NCCL announces its version on the process's stdout when the communicator is created: keep stdout = the one JSON line
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    ctx = {"world": world, "rank": rank, "local_rank": local_rank}
    if args.sharding == "frames" and world > 1:
        line = measure_frame_batches(args, args.workload, args.steps, args.warmup, ctx)
        if rank == 0:
            print(json.dumps(line), flush=True)
        dist.destroy_process_group()
        return
    line = measure(args, args.workload, args.steps, args.warmup, ctx, not args.no_cpu_baseline, args.profile_frames)
    if args.quick:
        if rank == 0:
            print(json.dumps(line), flush=True)
        return
    extra = {}
    if world == 1 and args.extra_workloads:
        for wl in [x for x in args.extra_workloads.split(",") if x and x != args.workload]:
            # BASELINE.json configs[2] etc. in the same JSON line: a short run (frames are 10-100x heavier than the headline's)
            sub_args = argparse.Namespace(**vars(args))
            sub_args.sequences_per_gpu = 0
            sub_args.dump_outputs = None
            extra[wl] = measure(sub_args, wl, min(args.steps, 30), 5, ctx, not args.no_cpu_baseline, min(args.profile_frames, 10))
    if world > 1 and args.sharding == "sequence" and args.extra_workloads:
        # N > 1: the headline above is N independent sequences (replicas, no collective on the data path).  The two modes that share ONE
        # sequence over the GPUs are measured briefly into the same line: the spatially sharded map (NCCL broadcast of the frame, strong
        # scaling, on the workload where the per-voxel update dominates) and frame-per-GPU batches with the NCCL all-gather + delta merge.
        def guarded(fn):
            try:
                return fn()
            except Exception as e:          # a failing extra must not cost the headline line
                return {"error": f"{type(e).__name__}: {e}"}
        sub = argparse.Namespace(**vars(args))
        sub.sequences_per_gpu = 0
        sub.dump_outputs = None
        sub.sharding = "spatial"
        r1 = guarded(lambda: measure(sub, "merged2", 10, 3, ctx, False, 5))
        sub2 = argparse.Namespace(**vars(args))
        sub2.sharding = "frames"
        sub2.dump_outputs = None
        r2 = guarded(lambda: measure_frame_batches(sub2, args.workload, 10, 3, ctx))
        extra["merged2_spatial"] = r1
        extra[f"{args.workload}_frame_batches"] = r2
    if rank == 0:
        line["workloads"] = extra
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
