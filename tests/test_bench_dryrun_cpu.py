"""bench.py's GPU arm cannot run in the build container, and a typo in it would cost the round its bench line.  This test runs
bench.main() end to end on the CPU with the device faked out: torch.cuda is stubbed, and the C-ABI Integrator is replaced by an
adapter around the CPU oracle (test infrastructure standing in for the device - nothing here is a measurement).  It checks
that every key of the contract's JSON line is produced and well-formed."""
import ctypes
import io
import json
import sys
import types
from contextlib import redirect_stdout

import numpy as np
import pytest
import torch

import bench
from kimera_semantics_b200 import capi
from oracle.oracle_py import OracleIntegrator


class FakeDeviceIntegrator:
    PHASES = capi.Integrator.PHASES

    def __init__(self, cfg):
        self.cfg = cfg
        self.o = OracleIntegrator(cfg, canonical_merged=(cfg.merged_bundle_order == 0))
        self.frames = 0

    @staticmethod
    def _view(ptr, n, ctype, dtype):
        return np.frombuffer((ctype * n).from_address(ptr), dtype=dtype)

    def integrate_depth_device(self, T, dptr, lptr, w, h, K, stream=0, want_stats=False):
        depth = self._view(dptr, w * h, ctypes.c_float, np.float32).reshape(h, w)
        label = self._view(lptr, w * h, ctypes.c_uint8, np.uint8).reshape(h, w)
        return self.integrate_depth(T, depth, label, K)

    def integrate_depth(self, T, depth, label, K):
        self.frames += 1
        st = self.o.integrate_depth(T, depth, label, K)
        st.fixpoint_iterations = 6
        return st

    def set_profiling(self, enable):
        self.frames = 0

    def get_profile(self):
        out = {name: 0.1 * (self.frames or 1) for name in self.PHASES}
        out.update(frames=self.frames, kernel_launches=35 * self.frames, library_calls=4 * self.frames)
        return out

    def num_blocks(self):
        return self.o.num_blocks()

    def integrate_depth_async(self, T, depth, label, K):
        self._pending = getattr(self, "_pending", [])
        self._pending.append(self.integrate_depth(T, depth, label, K))

    def wait_frame(self):
        return self._pending.pop(0)

    def fast_timeline(self):
        return {"sweeps": 6, "solve_kernel_us": 100.0}

    def sync(self):
        pass

    def export(self):
        return self.o.export()

    def close(self):
        self.o.close()


class FakeEvent:
    def __init__(self, enable_timing=True):
        self.t = 0.0

    def record(self, stream=None):
        import time
        self.t = time.perf_counter()

    def elapsed_time(self, other):
        return max(1e-3, (other.t - self.t) * 1e3)


def fake_device(monkeypatch):
    monkeypatch.setattr(capi, "Integrator", FakeDeviceIntegrator)
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "set_device", lambda d: None)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a: None)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a: types.SimpleNamespace(cuda_stream=0))
    monkeypatch.setattr(torch.cuda, "Event", FakeEvent)
    monkeypatch.setattr(torch.cuda, "Stream", lambda *a, **k: types.SimpleNamespace(cuda_stream=1))
    monkeypatch.setattr(torch.cuda, "set_stream", lambda s: None)
    monkeypatch.setattr(torch.Tensor, "cuda", lambda self, *a, **k: self)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **k: self)
    real_tensor = torch.tensor
    monkeypatch.setattr(torch, "tensor", lambda *a, **k: real_tensor(*a, **{kk: vv for kk, vv in k.items() if kk != "device"}))


@pytest.mark.parametrize("workload,extra", [("fast10", []), ("merged5", ["--merged-bundle-order", "libstdcxx", "--hot-voxels", "2"])])
def test_bench_main_dry_run_produces_a_complete_line(monkeypatch, workload, extra):
    if workload == "merged5":
        monkeypatch.setitem(bench.WORKLOADS, "merged5", (capi.KSG_INTEGRATOR_MERGED, 160, 120, 0.10, 21, 16 << 20, 8192))   # small frames
    fake_device(monkeypatch)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--workload", workload, "--steps", "4", "--warmup", "3", "--profile-frames", "2", "--sequences-per-gpu", "2", "--shim-e2e", "0",
                                      "--extra-workloads", "fast10" if workload != "fast10" else "merged5"] + extra)
    monkeypatch.setattr(bench, "best_cpu_arm", lambda wl, fr, cam: ("port", 1, {"port@1": 1.0}))
    buf = io.StringIO()
    with redirect_stdout(buf):
        bench.main()
    line = json.loads(buf.getvalue().strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
                "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert key in line, key
    assert line["steps"] == 4 and line["warmup"] == 3 and line["n_gpus"] == 1 and line["value"] > 0
    assert set(("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step")) <= set(line["e2e"]) and line["e2e"]["value"] > 0
    assert line["e2e"]["d2h_bytes_per_step"] == (152 + 568 if workload == "fast10" else 152 * 2)
    assert line["e2e"]["sync_value"] > 0 and line["e2e"]["mode"] == "pipelined"
    assert set(("frame_frac", "kernel", "phase", "tile_apply_frac")) <= set(line["roofline"])
    other = "merged5" if workload == "fast10" else "fast10"
    assert other in line["workloads"] and line["workloads"][other]["value"] > 0 and "roofline" in line["workloads"][other]
    if workload == "fast10":
        assert line["multi_sequence"]["sequences"] == 2 and line["multi_sequence"]["value"] > 0
    assert set(("bound", "achieved", "peak", "unit", "frac", "traffic")) <= set(line["roofline"]) and line["roofline"]["bound"] == "hbm"
    assert set(("value", "unit", "cores", "kind", "sample")) <= set(line["cpu_baseline"]) and line["cpu_baseline"]["value"] > 0
    assert line["config"]["merged_bundle_order"] == "libstdcxx"
    assert line["config"]["hot_voxel_mode"] == (2 if extra else 0)
    assert line["gpu_launches"] > 0


@pytest.mark.parametrize("limit", [None, 1 << 20])
def test_dump_outputs_is_the_map_after_exactly_the_timed_steps(monkeypatch, tmp_path, limit):
    """--dump-outputs writes the map of the timed integrator: warm-up + --steps frames, the same on every run, float32 / float64 only,
    within the byte budget (a seeded sample of the observed voxels when the map does not fit)."""
    fake_device(monkeypatch)
    if limit:
        monkeypatch.setattr(bench, "DUMP_BYTES", limit)
    dumps = []
    for run in range(2):
        out = tmp_path / f"run{run}"
        monkeypatch.setattr(sys, "argv", ["bench.py", "--workload", "fast10", "--steps", "5", "--warmup", "3", "--quick", "--dump-outputs", str(out)])
        with redirect_stdout(io.StringIO()):
            bench.main()
        dumps.append({p.stem: np.load(p) for p in sorted(out.iterdir())})
    a, b = dumps
    assert sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) for k in a)
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= bench.DUMP_BYTES
    cam, frames = bench.gen_frames("fast10", 3 + 5)
    ora = OracleIntegrator(bench.make_cfg("fast10"))
    for depth, label, T in frames:
        ora.integrate_depth(T, depth, label, cam.K)
    exp = ora.export()
    order = np.lexsort(exp["block_index"].T[::-1])
    assert np.array_equal(a["block_index"], exp["block_index"][order])
    observed = exp["tsdf_weight"][order] > 0
    assert a["observed_voxels"][0] == observed.sum()
    assert (len(a["voxel_index"]) < observed.sum()) == bool(limit)
    rows, vox = a["voxel_index"][:, 0].astype(int), a["voxel_index"][:, 1].astype(int)
    assert observed[rows, vox].all()
    for k in ("tsdf_distance", "tsdf_weight", "sem_priors", "sem_label"):
        assert np.array_equal(a[k], exp[k][order][rows, vox]), k
