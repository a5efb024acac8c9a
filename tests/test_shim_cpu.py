"""The C++ host shim (kimera_semantics_b200/cpp): builds without CUDA / Eigen / glog, mirrors the reference's factory
error convention (abort with a message) and never integrates on the CPU."""
import os
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CPP = os.path.join(ROOT, "kimera_semantics_b200", "cpp")


@pytest.fixture(scope="module")
def demo():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "kimera_semantics_b200", "csrc"), "libksg.so"], stdout=subprocess.DEVNULL)
    subprocess.check_call(["make", "-C", CPP], stdout=subprocess.DEVNULL)
    return os.path.join(CPP, "shim_demo")


def write_frames(path, frames_xyz_rgba, voxel_size, vps, palette, dynamic):
    import numpy as np
    with open(path, "wb") as f:
        f.write(np.int32(len(frames_xyz_rgba)).tobytes())
        f.write(np.float32(voxel_size).tobytes())
        f.write(np.int32(vps).tobytes())
        f.write(np.int32(len(palette)).tobytes())
        for l, c in enumerate(palette):
            f.write(bytes([int(c[0]), int(c[1]), int(c[2]), int(c[3]), l]))
        f.write(np.int32(len(dynamic)).tobytes())
        f.write(bytes(dynamic))
        for T, xyz, rgba in frames_xyz_rgba:
            f.write(np.int32(len(xyz)).tobytes())
            f.write(np.ascontiguousarray(T, np.float32).tobytes())
            f.write(np.ascontiguousarray(xyz, np.float32).tobytes())
            f.write(np.ascontiguousarray(rgba, np.uint8).tobytes())


def test_unknown_integrator_type_aborts_like_the_reference(demo, tmp_path):
    fr = tmp_path / "f.bin"
    write_frames(fr, [], 0.1, 16, [(255, 255, 255, 255)], [])
    r = subprocess.run([demo, "bogus", str(fr), str(tmp_path / "o.bin")], capture_output=True, text=True)
    assert r.returncode != 0
    assert "Unknown TSDF integrator type: bogus" in r.stderr       # LOG(FATAL) factory.cpp:61


@pytest.mark.skipif(torch.cuda.is_available(), reason="only meaningful on a box without a GPU")
def test_shim_has_no_cpu_fallback(demo, tmp_path):
    fr = tmp_path / "f.bin"
    write_frames(fr, [], 0.1, 16, [(255, 255, 255, 255)], [])
    r = subprocess.run([demo, "fast", str(fr), str(tmp_path / "o.bin")], capture_output=True, text=True)
    assert r.returncode != 0
    assert "ksg_create failed" in r.stderr and "no CPU fallback" in r.stderr


def test_shim_library_has_no_cuda_or_oracle_dependency():
    out = subprocess.run(["ldd", os.path.join(CPP, "libkimera_semantics_gpu.so")], capture_output=True, text=True).stdout
    assert "libksg.so" in out and "oracle" not in out
    syms = subprocess.run(["nm", "-D", "--defined-only", os.path.join(CPP, "libkimera_semantics_gpu.so")], capture_output=True, text=True).stdout
    for name in ("SemanticTsdfIntegratorFactory6create", "FastSemanticTsdfIntegrator19integratePointCloud",
                 "MergedSemanticTsdfIntegrator19integratePointCloud", "SemanticLabel2Color25getSemanticLabelFromColor"):
        assert name in syms, name


def test_label_colour_csv_loader_follows_reference_semantics(demo, tmp_path):
    """SemanticLabel2Color(filename): CSV rows name,red,green,blue,alpha,id (same shape as the reference's
    kimera_semantics_ros/cfg/*.csv); the header row parses to (0,0,0,0) -> 0 through atoi, later rows overwrite earlier ones,
    label 0 is forced to white and white to label 0 (color.cpp:42-67); lookup misses fall back to label 0 / colour (0,0,0,0)."""
    csv = tmp_path / "simulation.csv"
    csv.write_text("name,red,green,blue,alpha,id\nCube,255,0,127,255,0\nSphere,255,0,0,255,1\nPlane,0,255,0,255,2\nPlane,255,20,127,255,3\n")
    out = subprocess.run([os.path.join(CPP, "color_csv_test"), str(csv)], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    lines = out.stdout.strip().splitlines()
    assert lines[0] == "label 0 -> 255 255 255 255"          # forced white (color.cpp:64-65)
    assert lines[1] == "label 1 -> 255 0 0 255" and lines[2] == "label 2 -> 0 255 0 255" and lines[3] == "label 3 -> 255 20 127 255"
    assert lines[4] == "label 4 -> 0 0 0 0"                  # unknown label -> HashableColor() (color.cpp:92)
    assert "color 255 0 127 255 -> 0" in lines and "color 255 0 0 255 -> 1" in lines and "color 255 20 127 255 -> 3" in lines
    assert "color 255 255 255 255 -> 0" in lines and "color 0 0 0 0 -> 0" in lines and "color 1 2 3 255 -> 0" in lines
    bad = tmp_path / "bad.csv"
    bad.write_text("name,red,green\nA,1,2\n")
    r = subprocess.run([os.path.join(CPP, "color_csv_test"), str(bad)], capture_output=True, text=True)
    assert r.returncode != 0 and "Row 1 is invalid" in r.stderr      # CHECK_EQ(loop->size(), 6) color.cpp:51


def test_reference_call_patterns_compile_and_run_against_the_shim(demo):
    """cpp/test/api_compat_test.cpp: inheritance, enum values, Layer/Block accessors, factory overload signatures, default
    Config values - the call sites of the reference compile unchanged (SURVEY.md 7.3 item 7)."""
    out = subprocess.run([os.path.join(CPP, "api_compat_test")], capture_output=True, text=True)
    assert out.returncode == 0 and "api compat ok" in out.stdout, out.stdout + out.stderr


REF_FACTORY_DEMO = os.path.join(ROOT, "oracle", "_ref", "shim_demo_ref_factory")


@pytest.mark.skipif(not os.path.isdir("/root/reference"), reason="needs the reference sources (build container only)")
def test_reference_factory_source_compiles_and_links_against_the_shim(demo, tmp_path):
    """SURVEY.md 8b "Creation": the reference's own semantic_tsdf_integrator_factory.cpp builds unmodified against the shim's
    headers (constructor signatures, enum, type-name table, make_unique) and links in front of the shim library."""
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "ref"], stdout=subprocess.DEVNULL)
    assert os.path.exists(REF_FACTORY_DEMO)
    syms = subprocess.run(["nm", "-C", "--defined-only", REF_FACTORY_DEMO], capture_output=True, text=True).stdout
    assert "T kimera::SemanticTsdfIntegratorFactory::create(" in syms      # the reference's definition is the one in the binary
    fr = tmp_path / "f.bin"
    write_frames(fr, [], 0.1, 16, [(255, 255, 255, 255)], [])
    r = subprocess.run([REF_FACTORY_DEMO, "bogus", str(fr), str(tmp_path / "o.bin")], capture_output=True, text=True)
    assert r.returncode != 0 and "semantic_tsdf_integrator_factory.cpp:61] Unknown TSDF integrator type: bogus" in r.stderr
    if not torch.cuda.is_available():
        r = subprocess.run([REF_FACTORY_DEMO, "merged", str(fr), str(tmp_path / "o.bin")], capture_output=True, text=True)
        assert r.returncode != 0 and "no CPU fallback" in r.stderr       # the reference's factory reached OUR constructor


BINDING_CHECK = os.path.join(ROOT, "oracle", "_ref", "gpu_binding_check")


@pytest.mark.skipif(not os.path.isdir("/root/reference"), reason="needs the reference sources (build container only)")
def test_integration_md_binding_builds_against_the_reference_headers(demo, tmp_path):
    """INTEGRATION.md section B is real code: integration/kimera_semantics/semantic_tsdf_integrator_gpu.h compiles against the
    reference's own semantic_integrator_base.h / color.h / semantic_voxel.h, links with libksg.so, and reaches ksg_create."""
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "ref"], stdout=subprocess.DEVNULL)
    assert os.path.exists(BINDING_CHECK)
    out = subprocess.run(["ldd", BINDING_CHECK], capture_output=True, text=True).stdout
    assert "libksg.so" in out and "ks_oracle" not in out and "ks_ref_hybrid" not in out
    fr = tmp_path / "f.bin"
    write_frames(fr, [], 0.1, 16, [(255, 255, 255, 255)], [])
    if not torch.cuda.is_available():
        r = subprocess.run([BINDING_CHECK, "fast", str(fr), str(tmp_path / "o.bin")], capture_output=True, text=True)
        assert r.returncode != 0 and "semantic_tsdf_integrator_gpu.h" in r.stderr and "no CPU fallback" in r.stderr


def _make_ref_golden():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_ref_golden", os.path.join(ROOT, "tests", "golden", "make_ref_golden.py"))
    mrg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mrg)
    return mrg


def _recorded():
    import json
    return json.load(open(_make_ref_golden().SOURCES_GOLDEN))


def test_host_helpers_of_the_shim_equal_the_reference_implementations(demo, tmp_path):
    """SURVEY.md 8b "public surface": setSemanticProbabilities (the log-likelihood matrix), updateSemanticVoxelProbabilities,
    calculateMaximumLikelihoodLabel, updateSemanticVoxelColor, normalizeProbabilities of the shim's SemanticIntegratorBase against
    the reference's own compiled code on random vectors (its outputs recorded in tests/golden/ref_base_helpers.npz): bit-exact,
    except normalizeProbabilities whose L2 norm Eigen may accumulate in another order (1e-6 relative)."""
    import numpy as np
    mrg = _make_ref_golden()
    cfg, priors, freqs = mrg.helper_inputs()
    ref = np.load(mrg.HELPERS_GOLDEN)
    C, n = 21, len(priors)
    pal = [tuple(int(cfg.label_color[l][k]) for k in range(4)) for l in range(C)]
    fin, fout = tmp_path / "in.bin", tmp_path / "out.bin"
    with open(fin, "wb") as f:
        f.write(np.int32(n).tobytes() + np.int32(C).tobytes())
        for l, c in enumerate(pal):
            f.write(bytes([c[0], c[1], c[2], c[3], l]))
        f.write(np.float32(cfg.semantic_measurement_probability).tobytes())
        for k in range(n):
            f.write(priors[k].tobytes() + freqs[k].tobytes())
    r = subprocess.run([os.path.join(CPP, "base_helpers_test"), str(fin), str(fout)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    raw = open(fout, "rb").read()
    lm, ln = np.frombuffer(raw, "<f4", 2, 0)
    L = np.frombuffer(raw, "<f4", C * C, 8).reshape(C, C)
    assert np.array_equal(L, ref["log_likelihood"]) and lm == ref["log_match"] and ln == ref["log_non_match"]
    rec = np.dtype([("upd", "<f4", C), ("label", "u1"), ("rgba", "u1", 4), ("norm", "<f4", C)])
    got = np.frombuffer(raw, rec, n, 8 + 4 * C * C)
    for k in range(n):
        upd = ref["updated"][k]
        assert np.array_equal(got["upd"][k], upd), k
        assert got["label"][k] == int(np.argmax(upd))                                   # first maximum
        assert np.array_equal(got["rgba"][k], ref["label_rgba"][int(got["label"][k])])
        np.testing.assert_allclose(got["norm"][k], ref["normalized"][k], rtol=1e-6)


def test_label_csv_files_of_the_reference_parse_identically(demo):
    """The only data fixtures the reference ships are its label tables (kimera_semantics_ros/cfg/*.csv, SURVEY.md 8c, copied to
    tests/golden/label_csv): the shim's SemanticLabel2Color must build the same two tables from them as the reference's own reader
    (header row, duplicate colours, label 0 -> white override and all), whose parse of each file is recorded next to them."""
    mrg = _make_ref_golden()
    recorded = _recorded()["label_csv"]
    assert sorted(recorded) == sorted(os.listdir(mrg.LABEL_CSV_DIR)) and len(recorded) >= 4
    parsed = 0
    for name, want in sorted(recorded.items()):
        got = subprocess.run([os.path.join(CPP, "color_csv_test"), os.path.join(mrg.LABEL_CSV_DIR, name), "--dump"], capture_output=True, text=True)
        assert (got.returncode == 0) == want["ok"], (name, got.stderr, want["error"])
        if want["ok"]:
            assert got.stdout == want["stdout"], name
            parsed += 1
        else:   # one of the shipped files (mask_rcnn_mapping.csv) has two-column rows: both readers refuse it the same way
            assert "Row 2 is invalid" in got.stderr and "Row 2 is invalid" in want["error"], name
    assert parsed >= 4


def test_map_checkpoint_file_round_trip_on_the_host(demo, tmp_path):
    """map_io.h (SURVEY.md 8f NEXT-3 / checkpoint-resume): both layers -> one file -> fresh layers, every voxel bit-equal; foreign,
    mismatching and truncated files are refused."""
    r = subprocess.run([os.path.join(CPP, "map_io_test"), str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0 and "map io ok" in r.stdout, r.stderr
    raw = open(tmp_path / "map.ksgm", "rb").read()
    assert raw[:4] == b"KSGM" and len(raw) == 28 + 4 * (12 + 16 ** 3 * (4 + 4 + 4 + 1 + 4 * 21 + 4))
    _check_vxblx(tmp_path / "tsdf.vxblx")


def _check_vxblx(path):
    """The .vxblx file written by vxblx_io.h parses with google.protobuf against voxblox's schema (Layer.proto / Block.proto, restated in
    the header) in voxblox's framing: varint32 message count, then length-delimited LayerProto + BlockProto messages."""
    from google.protobuf import descriptor_pb2, descriptor_pool, message_factory
    fd = descriptor_pb2.FileDescriptorProto(name="vxblx_restated.proto", package="voxblox", syntax="proto2")
    T = descriptor_pb2.FieldDescriptorProto
    lay = fd.message_type.add(name="LayerProto")
    for name, num, typ in (("voxel_size", 1, T.TYPE_DOUBLE), ("voxels_per_side", 2, T.TYPE_UINT32), ("type", 3, T.TYPE_STRING)):
        lay.field.add(name=name, number=num, type=typ, label=T.LABEL_OPTIONAL)
    blk = fd.message_type.add(name="BlockProto")
    for name, num, typ in (("voxels_per_side", 1, T.TYPE_INT32), ("voxel_size", 2, T.TYPE_DOUBLE), ("origin_x", 3, T.TYPE_DOUBLE),
                           ("origin_y", 4, T.TYPE_DOUBLE), ("origin_z", 5, T.TYPE_DOUBLE), ("has_data", 6, T.TYPE_BOOL)):
        blk.field.add(name=name, number=num, type=typ, label=T.LABEL_OPTIONAL)
    f = blk.field.add(name="voxel_data", number=7, type=T.TYPE_UINT32, label=T.LABEL_REPEATED)
    f.options.packed = True
    pool = descriptor_pool.DescriptorPool()
    pool.Add(fd)
    Layer = message_factory.GetMessageClass(pool.FindMessageTypeByName("voxblox.LayerProto"))
    Block = message_factory.GetMessageClass(pool.FindMessageTypeByName("voxblox.BlockProto"))
    raw = open(path, "rb").read()

    def varint(pos):
        v = shift = 0
        while True:
            c = raw[pos]
            pos += 1
            v |= (c & 0x7F) << shift
            shift += 7
            if not c & 0x80:
                return v, pos
    n, pos = varint(0)
    assert n == 5                                    # layer header + the four blocks of the C++ test
    size, pos = varint(pos)
    layer = Layer()
    layer.ParseFromString(raw[pos:pos + size])
    pos += size
    assert layer.type == "tsdf" and layer.voxels_per_side == 16 and abs(layer.voxel_size - 0.05) < 1e-7
    origins = []
    for _ in range(n - 1):
        size, pos = varint(pos)
        b = Block()
        b.ParseFromString(raw[pos:pos + size])
        pos += size
        assert b.voxels_per_side == 16 and len(b.voxel_data) == 3 * 16 ** 3 and abs(b.voxel_size - 0.05) < 1e-7
        origins.append(tuple(round(o / (16 * 0.05)) for o in (b.origin_x, b.origin_y, b.origin_z)))
        if origins[-1] == (0, 0, 0):
            assert b.has_data
    assert pos == len(raw)
    assert sorted(origins) == sorted([(0, 0, 0), (-1, 2, 3), (5, -7, 1), (-100000, 99999, -3)])


LAUNCH_PARAMS = """# kimera_semantics_ros/launch/kimera_semantics.launch:98-122 as key: value lines
tsdf_voxel_size: 0.05
tsdf_voxels_per_side: 32
max_ray_length_m: 5
min_time_between_msgs_sec: 0.2
voxel_carving_enabled: true
use_const_weight: false
method: fast
semantic_color_mode: semantic
semantic_measurement_probability: 0.8
dynamic_semantic_labels: [20]
semantic_label_2_color_csv_filepath: {csv}
"""


def _write_small_csv(path):
    path.write_text(_make_ref_golden().SMALL_LABEL_CSV)


def test_params_reader_applies_the_launch_file_values(demo, tmp_path):
    csv = tmp_path / "labels.csv"
    _write_small_csv(csv)
    pf = tmp_path / "params.txt"
    pf.write_text(LAUNCH_PARAMS.format(csv=csv))
    out = subprocess.run([os.path.join(CPP, "params_test"), str(pf)], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert "method=fast" in out.stdout and "probability=0.800000012" in out.stdout and "color_mode=1" in out.stdout and "dynamic=20\n" in out.stdout
    assert "voxel_size=0.0500000007 vps=32 trunc=0.200000003 max_ray=5 carving=1 const_weight=0 throttle=0.2 order=mixed" in out.stdout


@pytest.mark.parametrize("text,fatal", [
    ("method: merged\nsemantic_color_mode: semantic_probability\nsemantic_measurement_probability: 0.75\ndynamic_semantic_labels: [20, 3, 7]\n", None),
    ("dynamic_semantic_labels: []\n", None),                                  # every default: fast, colour mode "color", p = 0.9
    ("semantic_color_mode: rainbow\ndynamic_semantic_labels: [1]\n", "Unknown semantic color mode: rainbow"),
    ("method: fast\n", "dynamic_semantic_labels"),                            # CHECK(getParam("dynamic_semantic_labels")) ros_params.cpp:69
])
def test_params_reader_equals_the_reference_ros_params(demo, tmp_path, text, fatal):
    """kimera_semantics/params.h against the reference's own kimera_semantics_ros/src/ros_params.cpp (compiled against a stand-in
    ros::NodeHandle; its output on the same parameter text is recorded in tests/golden): same values, same defaults, same fatal errors."""
    want = [r for r in _recorded()["ros_params"] if r["text"] == text]
    assert len(want) == 1
    want = want[0]
    csv = tmp_path / "labels.csv"
    _write_small_csv(csv)
    text = text + f"semantic_label_2_color_csv_filepath: {csv}\n"
    pf = tmp_path / "params.txt"
    pf.write_text(text)
    got = subprocess.run([os.path.join(CPP, "params_test"), str(pf)], capture_output=True, text=True)
    if fatal:
        assert got.returncode != 0 and not want["ok"]
        assert fatal in got.stderr and fatal in want["error"]
    else:
        assert got.returncode == 0 and want["ok"], (got.stderr, want["error"])
        want_stdout = want["stdout"].replace(_make_ref_golden().CSV_PLACEHOLDER, str(csv))
        assert got.stdout.startswith(want_stdout) and want_stdout.count("\n") == 6


@pytest.mark.skipif(not os.path.isdir("/root/reference"), reason="needs the reference sources (build container only)")
def test_api_compat_source_also_builds_against_the_reference_headers(demo):
    """cpp/test/api_compat_test.cpp uses only the reference's API; `make -C oracle ref` compiles the SAME file against the
    reference's real headers and sources (oracle/_ref/api_compat_ref).  Both binaries must pass: the client code the shim accepts
    is valid reference client code, and vice versa."""
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "ref"], stdout=subprocess.DEVNULL)
    for exe in (os.path.join(CPP, "api_compat_test"), os.path.join(ROOT, "oracle", "_ref", "api_compat_ref")):
        out = subprocess.run([exe], capture_output=True, text=True)
        assert out.returncode == 0 and "api compat ok" in out.stdout, (exe, out.stdout, out.stderr)
