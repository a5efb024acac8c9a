"""Pins the oracle against the reference's own code.

oracle/_ref/libks_ref_hybrid.so is built from the reference's kimera_semantics translation units (fast / merged integrators,
semantic_integrator_base, color, csv_iterator), compiled where they lie against stand-in Eigen / glog / voxblox headers
(oracle/ref_stubs; voxblox is un-vendored and none of the three is in the image).  tests/golden/ref_hybrid_golden.json holds
digests of its output for 32 seeded sequences covering every Config / SemanticConfig switch on the path.

  * test_oracle_matches_reference_golden     runs everywhere (GPU box included): oracle output == committed digests, bit for bit
    (`merged` in the oracle's faithful mode, which iterates bundles in libstdc++'s unordered_map order like merged.cpp:210-231);
  * test_live_reference_hybrid_*             run where the library exists: regenerate and diff field by field; elsewhere
    they hold the oracle to the same digests.
The remaining comparisons with the reference's own code use what make_ref_golden.py recorded from it (ref_sources_golden.json).
"""
import contextlib
import json
import os
import sys

import pytest

from oracle.oracle_py import OracleIntegrator
from oracle import ref_py
from parity_utils import compare_maps

import importlib.util
_spec = importlib.util.spec_from_file_location("make_ref_golden", os.path.join(os.path.dirname(__file__), "golden", "make_ref_golden.py"))
mrg = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(mrg)
GOLDEN = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ref_hybrid_golden.json")))
RECORDED = json.load(open(mrg.SOURCES_GOLDEN))

@contextlib.contextmanager
def quiet_stderr():
    """The reference logs every unknown colour (color.cpp:75-80); keep that out of the test report."""
    sys.stderr.flush()
    saved, devnull = os.dup(2), os.open(os.devnull, os.O_WRONLY)
    os.dup2(devnull, 2)
    try:
        yield
    finally:
        os.dup2(saved, 2)
        os.close(saved)
        os.close(devnull)


def faithful_oracle(cfg):
    return OracleIntegrator(cfg, canonical_merged=False)


def test_golden_covers_every_case():
    assert sorted(GOLDEN) == sorted(mrg.CASES)
    assert ref_py.available() or not os.path.isdir("/root/reference"), "in the build container the hybrid library must exist"


@pytest.mark.parametrize("name", sorted(mrg.CASES))
def test_oracle_matches_reference_golden(name):
    got = mrg.digest(mrg.run_case(name, faithful_oracle))
    want = GOLDEN[name]
    assert got["order_insensitive"]["observed_voxels"] > 0
    for k in mrg.KEYS:
        assert got[k] == want[k], f"{name}: {k} differs from the reference-hybrid golden"
    assert got["order_insensitive"] == want["order_insensitive"]


def assert_same_digest(got, want, what):
    for k in mrg.KEYS:
        assert got[k] == want[k], f"{what}: {k} differs from the reference's digest"
    assert got["order_insensitive"] == want["order_insensitive"], what


@pytest.mark.parametrize("name", sorted(mrg.CASES))
def test_live_reference_hybrid_equals_oracle_bit_for_bit(name):
    ora = mrg.run_case(name, faithful_oracle)
    if not ref_py.available():
        assert_same_digest(mrg.digest(ora), GOLDEN[name], name)
        return
    with quiet_stderr():
        ref = mrg.run_case(name, ref_py.RefHybridIntegrator)
    rep = compare_maps(ref, ora)
    assert rep["same_blocks"] == 1.0, rep
    bad = {k: v for k, v in rep.items() if k.endswith("mismatch") and v}
    assert not bad, f"{name}: {rep}"
    assert mrg.digest(ref) == GOLDEN[name], "committed golden is stale: python tests/golden/make_ref_golden.py"


def test_reference_allocates_tsdf_and_semantic_blocks_in_lock_step():
    """fast.cpp:125-132 / merged.cpp:315-321 touch both layers for every voxel; the product keeps ONE block table for both, with
    as many blocks as each of the reference's layers (counts recorded from the reference's sources)."""
    counts = RECORDED["block_counts_fast_default_3f"]
    assert counts["tsdf"] == counts["semantic"] > 0
    cfg = mrg.case_config("fast_default_3f")
    ora = faithful_oracle(cfg)
    ora.set_color_to_label(*mrg.color_table(cfg))
    for T, xyz, rgba, fs in mrg.case_frames("fast_default_3f", cfg):
        ora.integrate_points(T, xyz, rgba=rgba, freespace=fs)
    assert ora.num_blocks() == counts["tsdf"]


def test_canonical_bundle_order_keeps_the_order_insensitive_part_of_the_reference_result():
    """The CUDA path (and the oracle's default mode) apply `merged` bundles in first-insertion order instead of libstdc++'s
    hash-map order.  Same blocks, same touched voxels, same total weight (up to rounding); per-voxel values may differ."""
    for name in ("merged_default_2f", "merged_antigrazing", "merged_clearing_rays"):
        got = mrg.order_insensitive(mrg.run_case(name, lambda cfg: OracleIntegrator(cfg, canonical_merged=True)))
        want = GOLDEN[name]["order_insensitive"]
        for k in ("block_index", "observed_mask", "touched_mask", "observed_voxels", "touched_voxels"):
            assert got[k] == want[k], (name, k)
        assert abs(got["weight_sum"] - want["weight_sum"]) <= 1e-5 * want["weight_sum"]


tiny_frames = mrg.full_reset_frames      # the same clouds drive the CUDA path in test_gpu_more.py


def test_full_reset_of_the_approximate_sets_after_10000_frames_matches_the_reference():
    """fast.cpp:165-170 + ApproxHashSet::resetApproxSet: offset++ per frame, table wiped when it reaches 10 000."""
    cfg = mrg.full_reset_config()
    got = mrg.digest(mrg.run_full_reset(OracleIntegrator(cfg), cfg))
    assert_same_digest(got, RECORDED["full_reset_10012_frames"], "10 012 tiny frames")


def test_the_reference_itself_is_not_reproducible_with_several_threads():
    """Why parity is defined at integrator_threads = 1: the reference's own code (default: hardware_concurrency threads) races on
    the two approximate sets (`fast`) and on the per-voxel update order (both integrators), so its result changes from run to run.
    Reported here for the record; the assertion only requires that 8 threads do NOT reproduce the 1-thread map, which the oracle
    does reproduce.  Without the library, the 8-thread run is the one recorded from the reference's sources."""
    name = mrg.THREADS_CASE
    assert_same_digest(mrg.digest(mrg.run_case(name, faithful_oracle)), GOLDEN[name], name)
    recorded = RECORDED["threads8_" + name]
    assert any(recorded[k] != GOLDEN[name][k] for k in ("sem_priors", "tsdf_weight", "block_index"))
    if not ref_py.available():
        return

    def run(threads):
        def make(cfg):
            cfg.integrator_threads = threads
            return ref_py.RefHybridIntegrator(cfg)
        return mrg.run_case(name, make)
    one = run(1)
    assert mrg.digest(one) == GOLDEN[name]
    rep = compare_maps(run(8), one)
    observed = float((one["tsdf_weight"] > 0).sum())
    print(f"reference sources, 8 threads vs 1 thread ({name}): labels differ on {rep.get('label_mismatch', -1):.0f} of {observed:.0f} observed "
          f"voxels, distance bits on {rep.get('tsdf_distance_bit_mismatch', -1):.0f}, log-probability bits on {rep.get('sem_priors_bit_mismatch', -1):.0f}")
    assert rep["same_blocks"] != 1.0 or rep["sem_priors_bit_mismatch"] + rep["tsdf_weight_bit_mismatch"] > 0


@pytest.mark.skipif(not ref_py.available(fast_build=True), reason="oracle/_ref timing build not present")
@pytest.mark.parametrize("name", ["fast_default_3f", "merged_default_2f", "merged_clearing_antigrazing", "fast_color_mode_probability"])
def test_timing_build_of_the_reference_sources_gives_the_same_maps(name):
    """bench.py times the -O3 -march=x86-64-v3 build of the reference sources; it must compute exactly what the -O2 parity build does
    (no contraction, no reassociation: vectorisation alone does not change a float result)."""
    with quiet_stderr():
        fast = mrg.run_case(name, lambda cfg: ref_py.RefHybridIntegrator(cfg, fast_build=True))
    assert mrg.digest(fast) == GOLDEN[name]
