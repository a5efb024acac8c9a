"""Generates tests/golden/ref_hybrid_golden.json from the REFERENCE'S OWN kimera_semantics sources
(semantic_tsdf_integrator_{fast,merged}.cpp, semantic_integrator_base.cpp, color.cpp, csv_iterator.cpp), compiled in the
build container by `make -C oracle ref` against the stand-in Eigen/glog/voxblox headers of oracle/ref_stubs/ (see
oracle/ref_hybrid.cpp for exactly which half is the real reference).  The fixtures are SHA-256 digests of the exported map
after small seeded sequences pushed through the reference boundary integratePointCloud(T_G_C, points_C, colors, freespace)
(fast.cpp:145-149, merged.cpp:65-69), at the reference's compile-time 21 labels.

They travel to the GPU box (where neither /root/reference nor, necessarily, the hybrid library exists) and anchor
  * the oracle            (tests/test_oracle_vs_ref_hybrid.py, CPU)  - every digest, bit for bit;
  * the CUDA path          (tests/test_gpu_ref_golden.py, GPU)        - `fast` and `merged`: every digest, bit for bit (the product's
    default bundle order for `merged` is the reference's libstdc++ hash-map order).

Given a reference checkout, `python tests/golden/make_ref_golden.py <checkout>` also records what the remaining comparisons with the
reference's own code need, so that they run without it: digests of the random fuzz cases, of a 10 012-frame run and of an 8-thread run,
the block counts of both layers, the outputs of the SemanticIntegratorBase helpers (ref_base_helpers.npz), the reference's label
tables (label_csv/) with the reference reader's parse of each, and its ros_params.cpp on a few parameter files
(ref_sources_golden.json).

Regenerate where the reference exists:   make -C oracle ref && python tests/golden/make_ref_golden.py <checkout>
"""
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

from kimera_semantics_b200 import capi, synth  # noqa: E402
from kimera_semantics_b200.capi import KSG_INTEGRATOR_FAST as FAST, KSG_INTEGRATOR_MERGED as MERGED  # noqa: E402
from parity_utils import frames, make_config  # noqa: E402

C21 = 21
# name: (integrator, width, height, voxel size, frames, config overrides, scenario)
#   scenario: freespace -> the cloud is integrated as freespace points; unknown_colors -> every 97th point carries a colour
#   that is not in the label table (color.cpp:75-80 maps it to label 0)
CASES = {
    "fast_default_3f": (FAST, 160, 120, 0.10, 3, {}, {}),
    "fast_5cm_2f": (FAST, 160, 120, 0.05, 2, {}, {}),
    "fast_vps8": (FAST, 128, 96, 0.10, 2, {"voxels_per_side": 8}, {}),
    "fast_sorted_order": (FAST, 128, 96, 0.10, 2, {"integration_order_mode": capi.KSG_ORDER_SORTED}, {}),
    "fast_color_mode_color": (FAST, 128, 96, 0.10, 2, {"color_mode": capi.KSG_COLOR_MODE_COLOR}, {}),
    "fast_color_mode_probability": (FAST, 128, 96, 0.10, 2, {"color_mode": capi.KSG_COLOR_MODE_SEMANTIC_PROBABILITY}, {}),
    "fast_const_weight_no_dropoff": (FAST, 128, 96, 0.10, 2, {"use_const_weight": 1, "use_weight_dropoff": 0}, {}),
    "fast_sparsity_compensation": (FAST, 128, 96, 0.10, 2, {"use_sparsity_compensation_factor": 1, "sparsity_compensation_factor": 10.0}, {}),
    "fast_no_collision_budget": (FAST, 128, 96, 0.10, 2, {"max_consecutive_ray_collisions": 0}, {}),
    "fast_subsampling_1": (FAST, 128, 96, 0.10, 2, {"start_voxel_subsampling_factor": 1.0}, {}),
    "fast_p08": (FAST, 128, 96, 0.10, 2, {"semantic_measurement_probability": 0.8}, {}),
    "fast_clearing_rays": (FAST, 128, 96, 0.10, 2, {"max_ray_length_m": 2.5}, {}),
    "fast_no_clearing": (FAST, 128, 96, 0.10, 2, {"max_ray_length_m": 2.5, "allow_clear": 0}, {}),
    "fast_no_carving": (FAST, 128, 96, 0.10, 2, {"voxel_carving_enabled": 0, "max_ray_length_m": 2.5}, {}),
    "fast_freespace_cloud": (FAST, 128, 96, 0.10, 2, {}, {"freespace": True}),
    "fast_freespace_no_carving": (FAST, 128, 96, 0.10, 2, {"voxel_carving_enabled": 0}, {"freespace": True}),
    "fast_unknown_colors": (FAST, 128, 96, 0.10, 2, {}, {"unknown_colors": True}),
    "fast_clear_sets_every_2nd_frame": (FAST, 128, 96, 0.10, 4, {"clear_checks_every_n_frames": 2}, {}),
    "fast_min_range_gate": (FAST, 128, 96, 0.10, 2, {"min_ray_length_m": 2.0}, {}),
    # kimera_semantics_ros/launch/kimera_semantics.launch:98-122: 5 cm, 32 voxels per side, p = 0.8, semantic colours, fast
    "fast_launch_file_config": (FAST, 320, 240, 0.05, 3, {"voxels_per_side": 32, "semantic_measurement_probability": 0.8, "max_blocks": 1024}, {}),
    "fast_fullsize_640x480_5cm_4f": (FAST, 640, 480, 0.05, 4, {}, {}),             # BASELINE.json configs[1] geometry
    "merged_default_2f": (MERGED, 160, 120, 0.10, 2, {}, {}),
    "merged_fullsize_640x480_5cm_1f": (MERGED, 640, 480, 0.05, 1, {}, {}),
    # BASELINE.json configs[2] at full size: 640x480, 2 cm, `merged` (31 M voxel updates in the frame)
    "merged_fullsize_640x480_2cm_1f": (MERGED, 640, 480, 0.02, 1, {"max_updates": 80 << 20, "max_blocks": 32768}, {}),
    "merged_5cm": (MERGED, 128, 96, 0.05, 2, {}, {}),
    "merged_antigrazing": (MERGED, 128, 96, 0.10, 2, {"enable_anti_grazing": 1}, {}),
    "merged_clearing_rays": (MERGED, 128, 96, 0.10, 2, {"max_ray_length_m": 2.5}, {}),
    "merged_clearing_antigrazing": (MERGED, 128, 96, 0.10, 2, {"max_ray_length_m": 2.5, "enable_anti_grazing": 1}, {}),
    "merged_no_carving": (MERGED, 128, 96, 0.10, 2, {"voxel_carving_enabled": 0, "max_ray_length_m": 2.5}, {}),
    "merged_const_weight": (MERGED, 128, 96, 0.10, 2, {"use_const_weight": 1}, {}),
    "merged_color_mode_probability": (MERGED, 128, 96, 0.10, 2, {"color_mode": capi.KSG_COLOR_MODE_SEMANTIC_PROBABILITY}, {}),
    "merged_freespace_cloud": (MERGED, 128, 96, 0.10, 2, {}, {"freespace": True}),
    "merged_unknown_colors": (MERGED, 128, 96, 0.10, 2, {}, {"unknown_colors": True}),
}
KEYS = ("block_index", "tsdf_distance", "tsdf_weight", "tsdf_rgba", "sem_label", "sem_priors", "sem_rgba")


def case_config(name):
    itype, w, h, vs, nf, kw, sc = CASES[name]
    return make_config(itype, vs, C21, max_points=w * h, **{"max_updates": 8 << 20, **kw})


def case_frames(name, cfg):
    """Yields (T_G_C, points_C, rgba, freespace) exactly as every arm of the comparison receives them."""
    itype, w, h, vs, nf, kw, sc = CASES[name]
    pal = np.array([[cfg.label_color[l][k] for k in range(4)] for l in range(256)], np.uint8)
    for cam, depth, label, T in frames(w, h, C21, nf):
        xyz, pix = synth.backproject(depth, cam)
        rgba = np.ascontiguousarray(pal[label.reshape(-1)[pix]])
        if sc.get("unknown_colors"):
            rgba[::97] = (1, 2, 3, 255)
        yield T, xyz, rgba, bool(sc.get("freespace", False))


def color_table(cfg):
    pal = np.array([[cfg.label_color[l][k] for k in range(3)] for l in range(C21)], np.uint8)
    return pal, np.arange(C21, dtype=np.uint8)


def order_insensitive(exp):
    """What survives a change of the per-voxel update order (bundle order in `merged`)."""
    w = exp["tsdf_weight"].astype(np.float64)
    touched = (exp["tsdf_weight"] > 0) | (exp["sem_priors"] != np.float32(-0.60205999132)).any(axis=-1)
    return {"block_index": hashlib.sha256(np.ascontiguousarray(exp["block_index"]).tobytes()).hexdigest(),
            "observed_mask": hashlib.sha256(np.packbits(exp["tsdf_weight"] > 0).tobytes()).hexdigest(),
            "touched_mask": hashlib.sha256(np.packbits(touched).tobytes()).hexdigest(),
            "observed_voxels": int((exp["tsdf_weight"] > 0).sum()), "touched_voxels": int(touched.sum()),
            "weight_sum": float(w.sum())}


def digest(exp):
    d = {k: hashlib.sha256(np.ascontiguousarray(exp[k]).tobytes()).hexdigest() for k in KEYS}
    d["order_insensitive"] = order_insensitive(exp)
    return d


def run_case(name, make_integrator):
    """make_integrator(cfg) -> object with set_color_to_label (optional), integrate_points(T, xyz, rgba=, freespace=), export()."""
    cfg = case_config(name)
    integ = make_integrator(cfg)
    if hasattr(integ, "set_color_to_label"):
        integ.set_color_to_label(*color_table(cfg))
    for T, xyz, rgba, freespace in case_frames(name, cfg):
        integ.integrate_points(T, xyz, rgba=rgba, freespace=freespace)
    return integ.export()


GOLDEN_DIR = os.path.dirname(os.path.abspath(__file__))
# the reference's label tables (kimera_semantics_ros/cfg), copied verbatim as data fixtures
LABEL_CSV_DIR = os.path.join(GOLDEN_DIR, "label_csv")
SOURCES_GOLDEN = os.path.join(GOLDEN_DIR, "ref_sources_golden.json")
HELPERS_GOLDEN = os.path.join(GOLDEN_DIR, "ref_base_helpers.npz")
CSV_PLACEHOLDER = "{csv}"      # stands for the label CSV path inside recorded ros_params output
THREADS_CASE = "fast_fullsize_640x480_5cm_4f"


def helper_inputs(n=200, seed=7):
    """Random prior / frequency rows for the SemanticIntegratorBase helpers, p = 0.8 (case fast_p08)."""
    rng = np.random.default_rng(seed)
    priors = (-rng.uniform(0.1, 40.0, (n, C21))).astype(np.float32)
    freqs = rng.integers(0, 6, (n, C21)).astype(np.float32)
    freqs[::5] = np.eye(C21, dtype=np.float32)[rng.integers(0, C21, len(freqs[::5]))]      # one-hot rows, as `fast` produces them
    return case_config("fast_p08"), priors, freqs


def full_reset_frames(n_frames=10012, points_per_frame=24, seed=5):
    """Many tiny clouds: drives the ApproxHashSet offset through its full-reset threshold (10 000 resets)."""
    rng = np.random.default_rng(seed)
    for f in range(n_frames):
        T = synth.pose(f % 300)
        xyz = np.stack([rng.uniform(-0.4, 0.4, points_per_frame), rng.uniform(-0.3, 0.3, points_per_frame),
                        rng.uniform(0.8, 1.6, points_per_frame)], axis=1).astype(np.float32)
        lab = rng.integers(0, 20, points_per_frame).astype(np.uint8)
        yield T, xyz, lab


def full_reset_config():
    return make_config(FAST, 0.10, C21, max_points=64)


def run_full_reset(integ, cfg):
    pal = np.array([[cfg.label_color[l][k] for k in range(4)] for l in range(256)], np.uint8)
    if hasattr(integ, "set_color_to_label"):
        integ.set_color_to_label(*color_table(cfg))
    for T, xyz, lab in full_reset_frames():
        integ.integrate_points(T, xyz, rgba=np.ascontiguousarray(pal[lab]))
    return integ.export()


ROS_PARAM_TEXTS = [
    "method: merged\nsemantic_color_mode: semantic_probability\nsemantic_measurement_probability: 0.75\ndynamic_semantic_labels: [20, 3, 7]\n",
    "dynamic_semantic_labels: []\n",                                  # every default: fast, colour mode "color", p = 0.9
    "semantic_color_mode: rainbow\ndynamic_semantic_labels: [1]\n",
    "method: fast\n",                                                 # CHECK(getParam("dynamic_semantic_labels")) ros_params.cpp:69
]
SMALL_LABEL_CSV = "name,red,green,blue,alpha,id\nfloor,10,20,30,255,1\nwall,40,50,60,255,2\n"


def _in_subprocess(expr, arg):
    """The reference aborts on malformed input (CHECK / LOG(FATAL)), so each call runs in its own process."""
    import subprocess
    r = subprocess.run([sys.executable, "-c", f"import sys; from oracle import ref_py; sys.stdout.write({expr}(sys.argv[1]))", arg],
                       capture_output=True, text=True, cwd=ROOT)
    # the last log line without its "F <source path>:<line>] " prefix
    last = r.stderr.strip().splitlines()[-1] if r.stderr.strip() else ""
    return {"ok": r.returncode == 0, "stdout": r.stdout, "error": last.split("] ", 1)[-1]}


def reference_records(ref_dir):
    """Everything else the tests compare with the reference's own code, recorded from oracle/_ref and the reference checkout."""
    import shutil
    import tempfile
    import fuzz_cases
    from oracle.ref_py import RefHybridIntegrator
    rec = {}
    fuzz = {}
    for seed in range(24):
        cfg, frames_ = fuzz_cases.make_case(seed)
        ref = RefHybridIntegrator(cfg)
        with fuzz_cases.quiet_stderr():
            for T, pts, rgba, freespace in frames_:
                ref.integrate_points(T, pts, rgba=rgba, freespace=freespace)
        fuzz[str(seed)] = digest(ref.export())
    rec["fuzz"] = fuzz
    cfg = case_config("fast_default_3f")
    ref = RefHybridIntegrator(cfg)
    for T, xyz, rgba, fs in case_frames("fast_default_3f", cfg):
        ref.integrate_points(T, xyz, rgba=rgba, freespace=fs)
    rec["block_counts_fast_default_3f"] = {"tsdf": ref.num_blocks(), "semantic": ref.num_semantic_blocks()}
    cfg = full_reset_config()
    rec["full_reset_10012_frames"] = digest(run_full_reset(RefHybridIntegrator(cfg), cfg))

    def threads(n):
        def make(cfg):
            cfg.integrator_threads = n
            return RefHybridIntegrator(cfg)
        return make
    rec["threads8_" + THREADS_CASE] = digest(run_case(THREADS_CASE, threads(8)))

    os.makedirs(LABEL_CSV_DIR, exist_ok=True)
    cfg_dir = os.path.join(ref_dir, "kimera_semantics_ros", "cfg")
    csv = {}
    for name in sorted(os.listdir(cfg_dir)):
        if name.endswith("_mapping.csv") or name == "simulation.csv":
            shutil.copyfile(os.path.join(cfg_dir, name), os.path.join(LABEL_CSV_DIR, name))
            csv[name] = _in_subprocess("ref_py.csv_dump", os.path.join(LABEL_CSV_DIR, name))
    rec["label_csv"] = csv
    params = []
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "labels.csv")
        open(path, "w").write(SMALL_LABEL_CSV)
        for text in ROS_PARAM_TEXTS:
            r = _in_subprocess("ref_py.ros_params", text + f"semantic_label_2_color_csv_filepath: {path}\n")
            r["stdout"] = r["stdout"].replace(path, CSV_PLACEHOLDER)
            params.append(dict(r, text=text))
    rec["ros_params"] = params
    return rec


def record_base_helpers():
    from oracle.ref_py import RefHybridIntegrator
    cfg, priors, freqs = helper_inputs()
    ref = RefHybridIntegrator(cfg)
    L, lm, ln = ref.log_likelihood()
    upd = np.stack([ref.update_probabilities(freqs[k], priors[k]) for k in range(len(priors))])
    np.savez_compressed(HELPERS_GOLDEN, log_likelihood=L, log_match=np.float32(lm), log_non_match=np.float32(ln), updated=upd,
                        label_rgba=np.stack([ref.label_color(l) for l in range(C21)]),
                        normalized=np.stack([ref.normalize_probabilities(u) for u in upd]))


if __name__ == "__main__":
    # usage: python tests/golden/make_ref_golden.py <reference checkout>   (after `make -C oracle ref REF=<checkout>/kimera_semantics ...`)
    from oracle.ref_py import RefHybridIntegrator, available
    assert available(), "build oracle/_ref first: make -C oracle ref"
    out = {name: digest(run_case(name, RefHybridIntegrator)) for name in CASES}
    path = os.path.join(GOLDEN_DIR, "ref_hybrid_golden.json")
    json.dump(out, open(path, "w"), indent=1, sort_keys=True)
    print("wrote", path, len(out), "cases")
    if len(sys.argv) > 1:
        json.dump(reference_records(sys.argv[1]), open(SOURCES_GOLDEN, "w"), indent=1, sort_keys=True)
        record_base_helpers()
        print("wrote", SOURCES_GOLDEN, HELPERS_GOLDEN, LABEL_CSV_DIR)
