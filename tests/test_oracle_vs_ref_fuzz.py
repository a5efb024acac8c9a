"""Randomised differential test: the oracle against the reference's own sources (oracle/_ref) on random clouds, poses and
configuration switches - far/near/behind-the-camera points, |z| ~ 0 (zero weight), unknown colours, freespace clouds, every
Config flag.  Bit-exact in every exported field; `merged` in the oracle's faithful (libstdc++ bundle order) mode.  The reference's
maps are the digests tests/golden/make_ref_golden.py recorded from its sources on the same seeds.
The same generator (tests/fuzz_cases.py) drives the CUDA path in tests/test_gpu_fuzz.py."""
import importlib.util
import json
import os

import pytest

from oracle.oracle_py import OracleIntegrator
import fuzz_cases

_spec = importlib.util.spec_from_file_location("make_ref_golden", os.path.join(os.path.dirname(__file__), "golden", "make_ref_golden.py"))
mrg = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(mrg)
RECORDED = json.load(open(mrg.SOURCES_GOLDEN))["fuzz"]


@pytest.mark.parametrize("seed", range(24))
def test_random_case_oracle_equals_reference_sources(seed):
    cfg, frames = fuzz_cases.make_case(seed)
    ora = OracleIntegrator(cfg, canonical_merged=False)
    ora.set_color_to_label(*fuzz_cases.color_table(cfg))
    for T, pts, rgba, freespace in frames:
        ora.integrate_points(T, pts, rgba=rgba, freespace=freespace)
    got, want = mrg.digest(ora.export()), RECORDED[str(seed)]
    assert got["order_insensitive"] == want["order_insensitive"], (got["order_insensitive"], want["order_insensitive"])
    assert {k: got[k] == want[k] for k in mrg.KEYS} == {k: True for k in mrg.KEYS}
