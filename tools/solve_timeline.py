"""Frame time of a `fast` workload timed and profiled, and the phase timeline of the persistent solve kernel.

    python tools/solve_timeline.py [--workload fast5] [--steps 100] [--warmup 10]

Runs the same frames twice on fresh maps: once back to back with profiling off (frames/s as bench.py's `value`), once with
profiling on (per-frame device span, clock64 phase marks and solver counters of the last frame).  The two frame times should
agree within a few per cent; where they do not, the probes move the phases they measure.  Prints one JSON object.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from kimera_semantics_b200.capi import Integrator  # noqa: E402


def gpu_name_and_power():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="fast5", choices=[k for k, v in bench.WORKLOADS.items() if k.startswith("fast")])
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()
    import torch

    _, w, h, _, _, _, _ = bench.WORKLOADS[args.workload]
    n = args.warmup + args.steps
    cam, frames = bench.gen_frames(args.workload, n)
    d_depth = [torch.from_numpy(f[0]).cuda() for f in frames]
    d_label = [torch.from_numpy(f[1]).cuda() for f in frames]
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    cfg = bench.make_cfg(args.workload)

    def run(integ, lo, hi, stats=False):
        for i in range(lo, hi):
            integ.integrate_depth_device(frames[i][2], d_depth[i].data_ptr(), d_label[i].data_ptr(), w, h, cam.K,
                                         stream.cuda_stream, want_stats=stats)

    integ = Integrator(cfg)
    run(integ, 0, args.warmup)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    run(integ, args.warmup, n)
    ev1.record(stream)
    torch.cuda.synchronize()
    timed_ms = ev0.elapsed_time(ev1) / args.steps
    integ.close()

    integ = Integrator(cfg)
    run(integ, 0, args.warmup)
    integ.set_profiling(True)
    run(integ, args.warmup, n, stats=True)
    prof = integ.get_profile()
    timeline = integ.fast_timeline()
    integ.close()
    profiled_ms = prof["frame"] / max(1, prof["frames"])
    print(json.dumps({"workload": args.workload, "gpu": gpu_name_and_power(), "steps": args.steps,
                      "timed_frame_ms": timed_ms, "timed_frames_per_s": 1e3 / timed_ms,
                      "profiled_frame_ms": profiled_ms, "profiled_over_timed": profiled_ms / timed_ms,
                      "profiled_phase_ms": {k: prof[k] / max(1, prof["frames"]) for k in Integrator.PHASES},
                      "solve_kernel_timeline_last_profiled_frame": timeline}, indent=1))


if __name__ == "__main__":
    main()
