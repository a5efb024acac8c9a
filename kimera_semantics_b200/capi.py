"""ctypes binding of the C-ABI in include/ksg.h (the drop-in boundary).

This is plumbing for tests and bench.py: it loads `csrc/libksg.so` (hand-written sm_100a CUDA behind
`extern "C"` entry points) and fails loudly when the library is missing — there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional

import numpy as np

KSG_ABI_VERSION = 1
KSG_INTEGRATOR_MERGED = 0
KSG_INTEGRATOR_FAST = 1
KSG_COLOR_MODE_COLOR = 0
KSG_COLOR_MODE_SEMANTIC = 1
KSG_COLOR_MODE_SEMANTIC_PROBABILITY = 2
KSG_ORDER_MIXED = 0
KSG_ORDER_SORTED = 1
KSG_BUNDLE_ORDER_CANONICAL = 0
KSG_BUNDLE_ORDER_LIBSTDCXX = 1

KSG_STATUS = {0: "OK", 1: "INVALID_ARGUMENT", 2: "CUDA", 3: "POOL_FULL", 4: "SCRATCH_FULL", 5: "INDEX_RANGE",
              6: "NO_DEVICE"}


class KsgConfig(C.Structure):
    """Mirror of `struct ksg_config` (include/ksg.h)."""
    _fields_ = [
        ("abi_version", C.c_int32),
        ("integrator_type", C.c_int32),
        ("voxel_size", C.c_float),
        ("voxels_per_side", C.c_int32),
        ("default_truncation_distance", C.c_float),
        ("max_weight", C.c_float),
        ("voxel_carving_enabled", C.c_int32),
        ("min_ray_length_m", C.c_float),
        ("max_ray_length_m", C.c_float),
        ("use_const_weight", C.c_int32),
        ("allow_clear", C.c_int32),
        ("use_weight_dropoff", C.c_int32),
        ("use_sparsity_compensation_factor", C.c_int32),
        ("sparsity_compensation_factor", C.c_float),
        ("integration_order_mode", C.c_int32),
        ("enable_anti_grazing", C.c_int32),
        ("start_voxel_subsampling_factor", C.c_float),
        ("max_consecutive_ray_collisions", C.c_int32),
        ("clear_checks_every_n_frames", C.c_int32),
        ("integrator_threads", C.c_int32),
        ("num_labels", C.c_int32),
        ("semantic_measurement_probability", C.c_float),
        ("color_mode", C.c_int32),
        ("label_color", (C.c_uint8 * 4) * 256),
        ("label_color_known", C.c_uint8 * 256),
        ("dynamic_label", C.c_uint8 * 256),
        ("device", C.c_int32),
        ("max_blocks", C.c_int32),
        ("max_points", C.c_int32),
        ("max_ray_steps", C.c_int64),
        ("max_updates", C.c_int64),
        ("apply_mode", C.c_int32),
        ("shard_rank", C.c_int32),
        ("shard_count", C.c_int32),
        ("merged_bundle_order", C.c_int32),
        ("hot_voxel_mode", C.c_int32),
        ("reserved", C.c_int32 * 3),
    ]


class KsgFrameStats(C.Structure):
    """Mirror of `struct ksg_frame_stats` (include/ksg.h)."""
    _fields_ = [
        ("points_in", C.c_int64),
        ("points_valid", C.c_int64),
        ("rays_cast", C.c_int64),
        ("ray_steps", C.c_int64),
        ("voxel_updates", C.c_int64),
        ("blocks_allocated", C.c_int64),
        ("blocks_touched", C.c_int64),
        ("tiles_touched", C.c_int64),
        ("fixpoint_iterations", C.c_int64),
        ("hot_voxels", C.c_int64),
        ("hot_fallback_chunks", C.c_int64),
        ("reserved", C.c_int64 * 5),
    ]

    def as_dict(self) -> Dict[str, int]:
        return {n: int(getattr(self, n)) for n, _ in self._fields_ if n != "reserved"}


def label_palette(num_labels: int) -> np.ndarray:
    """A deterministic label -> RGBA table (label 0 = white as color.cpp:64-66 forces)."""
    pal = np.zeros((256, 4), dtype=np.uint8)
    for l in range(256):
        pal[l] = ((l * 67 + 29) % 256, (l * 131 + 71) % 256, (l * 199 + 113) % 256, 255)
    pal[0] = (255, 255, 255, 255)
    return pal


def default_config(integrator_type: int = KSG_INTEGRATOR_FAST, voxel_size: float = 0.05, voxels_per_side: int = 16,
                   num_labels: int = 21) -> KsgConfig:
    """voxblox / kimera defaults (SURVEY.md A.6, base.h:77-86, 8d "Integrator config"). Must equal
    ksg_default_config() except for the palette / dynamic label which this helper also fills."""
    cfg = KsgConfig()
    cfg.abi_version = KSG_ABI_VERSION
    cfg.integrator_type = integrator_type
    cfg.voxel_size = voxel_size
    cfg.voxels_per_side = voxels_per_side
    cfg.default_truncation_distance = float(np.float32(4.0) * np.float32(voxel_size))
    cfg.max_weight = 10000.0
    cfg.voxel_carving_enabled = 1
    cfg.min_ray_length_m = 0.1
    cfg.max_ray_length_m = 5.0
    cfg.use_const_weight = 0
    cfg.allow_clear = 1
    cfg.use_weight_dropoff = 1
    cfg.use_sparsity_compensation_factor = 0
    cfg.sparsity_compensation_factor = 1.0
    cfg.integration_order_mode = KSG_ORDER_MIXED
    cfg.enable_anti_grazing = 0
    cfg.start_voxel_subsampling_factor = 2.0
    cfg.max_consecutive_ray_collisions = 2
    cfg.clear_checks_every_n_frames = 1
    cfg.integrator_threads = 1
    cfg.num_labels = num_labels
    cfg.semantic_measurement_probability = 0.9
    cfg.color_mode = KSG_COLOR_MODE_SEMANTIC
    pal = label_palette(num_labels)
    for l in range(256):
        for k in range(4):
            cfg.label_color[l][k] = int(pal[l, k])
        cfg.label_color_known[l] = 1 if l < num_labels else 0
        cfg.dynamic_label[l] = 0
    cfg.device = 0
    cfg.max_blocks = 8192
    cfg.max_points = 640 * 480
    cfg.max_ray_steps = 0   # 0 = let the library size it from max_points
    cfg.max_updates = 0
    cfg.apply_mode = 0
    cfg.shard_rank = 0
    cfg.shard_count = 1
    cfg.merged_bundle_order = KSG_BUNDLE_ORDER_LIBSTDCXX   # the reference's order (merged.cpp:210-231)
    cfg.hot_voxel_mode = 0   # opt-in: measured slower than the per-voxel kernels alone (profiles/r02/bench_merged2_hot.json)
    return cfg


def library_path() -> str:
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "libksg.so")


_LIB = None


def _ptr(a: Optional[np.ndarray], ctype):
    if a is None:
        return None
    return a.ctypes.data_as(C.POINTER(ctype))


def load_library(path: Optional[str] = None):
    """Load libksg.so and declare every symbol of include/ksg.h. Raises if the library is missing."""
    global _LIB
    if _LIB is not None and path is None:
        return _LIB
    p = path or library_path()
    if not os.path.exists(p):
        raise RuntimeError(f"{p} not found: build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()'). "
                           "There is no CPU fallback.")
    lib = C.CDLL(p)
    H = C.c_void_p
    fp, u8p, i32p = C.POINTER(C.c_float), C.POINTER(C.c_uint8), C.POINTER(C.c_int32)
    sp = C.POINTER(KsgFrameStats)
    lib.ksg_default_config.argtypes = [C.POINTER(KsgConfig), C.c_int32, C.c_float, C.c_int32, C.c_int32]
    lib.ksg_default_config.restype = None
    lib.ksg_create.argtypes = [C.POINTER(KsgConfig), C.POINTER(H)]
    lib.ksg_create.restype = C.c_int32
    lib.ksg_destroy.argtypes = [H]
    lib.ksg_destroy.restype = None
    lib.ksg_last_error.argtypes = [H]
    lib.ksg_last_error.restype = C.c_char_p
    lib.ksg_integrate_points.argtypes = [H, fp, fp, u8p, u8p, C.c_int64, C.c_int32, sp]
    lib.ksg_integrate_points.restype = C.c_int32
    lib.ksg_integrate_points_device.argtypes = [H, fp, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, sp]
    lib.ksg_integrate_points_device.restype = C.c_int32
    lib.ksg_integrate_depth.argtypes = [H, fp, fp, u8p, C.c_int32, C.c_int32, fp, sp]
    lib.ksg_integrate_depth.restype = C.c_int32
    lib.ksg_integrate_depth_device.argtypes = [H, fp, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, fp, C.c_void_p, sp]
    lib.ksg_integrate_depth_device.restype = C.c_int32
    lib.ksg_set_color_to_label.argtypes = [H, u8p, u8p, C.c_int32]
    lib.ksg_set_color_to_label.restype = C.c_int32
    lib.ksg_sync.argtypes = [H]
    lib.ksg_sync.restype = C.c_int32
    lib.ksg_num_blocks.argtypes = [H]
    lib.ksg_num_blocks.restype = C.c_int64
    lib.ksg_export_blocks.argtypes = [H, C.c_int64, i32p, fp, fp, u8p, u8p, fp, u8p]
    lib.ksg_export_blocks.restype = C.c_int32
    lib.ksg_export_blocks_by_index.argtypes = [H, C.c_int64, i32p, u8p, fp, fp, u8p, u8p, fp, u8p]
    lib.ksg_export_blocks_by_index.restype = C.c_int32
    lib.ksg_import_blocks.argtypes = [H, C.c_int64, i32p, fp, fp, u8p, u8p, fp, u8p]
    lib.ksg_import_blocks.restype = C.c_int32
    lib.ksg_last_updated_blocks.argtypes = [H, C.c_int64, i32p]
    lib.ksg_last_updated_blocks.restype = C.c_int64
    lib.ksg_reset.argtypes = [H]
    lib.ksg_reset.restype = C.c_int32
    lib.ksg_set_profiling.argtypes = [H, C.c_int32]
    lib.ksg_set_profiling.restype = C.c_int32
    lib.ksg_get_profile.argtypes = [H, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.ksg_get_profile.restype = C.c_int32
    lib.ksg_debug_tile_times.argtypes = [H, C.c_int32, C.c_int64, C.POINTER(C.c_int64)]
    lib.ksg_debug_tile_times.restype = C.c_int64
    lib.ksg_owner_mask.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int64, i32p, u8p]
    lib.ksg_owner_mask.restype = C.c_int32
    dp = C.POINTER(C.c_double)
    lib.ksg_integrate_depth_k64.argtypes = [H, fp, fp, u8p, C.c_int32, C.c_int32, dp, sp]
    lib.ksg_integrate_depth_k64.restype = C.c_int32
    lib.ksg_integrate_depth_device_k64.argtypes = [H, fp, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, dp, C.c_void_p, sp]
    lib.ksg_integrate_depth_device_k64.restype = C.c_int32
    lib.ksg_debug_chain_sum.argtypes = [fp, C.c_int64, C.c_float, fp]
    lib.ksg_debug_chain_sum.restype = C.c_int32
    lib.ksg_unordered_map_schedule.argtypes = [C.c_int64, C.POINTER(C.c_int64)]
    lib.ksg_unordered_map_schedule.restype = C.c_int64
    lib.ksg_debug_fast_timeline.argtypes = [H, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_double)]
    lib.ksg_debug_fast_timeline.restype = C.c_int64
    lib.ksg_integrate_depth_async.argtypes = [H, fp, fp, u8p, C.c_int32, C.c_int32, fp]
    lib.ksg_integrate_depth_async.restype = C.c_int32
    lib.ksg_wait_frame.argtypes = [H, sp]
    lib.ksg_wait_frame.restype = C.c_int32
    lib.ksg_device_map_view.argtypes = [H, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
    lib.ksg_device_map_view.restype = C.c_int32
    lib.ksg_merge_blocks_device.argtypes = [H, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ksg_merge_blocks_device.restype = C.c_int32
    lib.ksg_copy_map_device.argtypes = [H, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ksg_copy_map_device.restype = C.c_int32
    lib.ksg_integrate_image.argtypes = [H, fp, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, dp, sp]
    lib.ksg_integrate_image.restype = C.c_int32
    lib.ksg_set_update_log.argtypes = [H, C.c_int64]
    lib.ksg_set_update_log.restype = C.c_int32
    lib.ksg_fetch_update_log.argtypes = [H, C.POINTER(C.c_int64), C.POINTER(C.c_void_p), C.POINTER(C.POINTER(C.c_float))]
    lib.ksg_fetch_update_log.restype = C.c_int32
    lib.ksg_evaluate_labels.argtypes = [H, C.c_void_p, C.c_int32, C.c_float, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                        C.POINTER(C.c_int64)]
    lib.ksg_evaluate_labels.restype = C.c_int32
    lib.ksg_extract_mesh.argtypes = [H, C.c_float, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                     C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.ksg_extract_mesh.restype = C.c_int32
    lib.ksg_copy_update_log_device.argtypes = [H, C.POINTER(C.c_int64), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.ksg_copy_update_log_device.restype = C.c_int32
    lib.ksg_merge_voxels_device.argtypes = [H, C.c_int32, C.POINTER(C.c_int64), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ksg_merge_voxels_device.restype = C.c_int32
    lib.ksg_clear_map.argtypes = [H]
    lib.ksg_clear_map.restype = C.c_int32
    lib.ksg_build_info.argtypes = []
    lib.ksg_build_info.restype = C.c_char_p
    if path is None:
        _LIB = lib
    return lib


KSG_SYMBOLS = ["ksg_default_config", "ksg_create", "ksg_destroy", "ksg_last_error", "ksg_integrate_points",
               "ksg_integrate_points_device", "ksg_integrate_depth", "ksg_integrate_depth_device",
               "ksg_set_color_to_label", "ksg_sync", "ksg_num_blocks", "ksg_export_blocks", "ksg_export_blocks_by_index", "ksg_import_blocks",
               "ksg_last_updated_blocks", "ksg_reset", "ksg_build_info", "ksg_set_profiling", "ksg_get_profile", "ksg_debug_tile_times", "ksg_owner_mask",
               "ksg_unordered_map_schedule", "ksg_integrate_depth_k64", "ksg_integrate_depth_device_k64",
               "ksg_debug_chain_sum", "ksg_debug_fast_timeline", "ksg_integrate_depth_async", "ksg_wait_frame",
               "ksg_device_map_view", "ksg_merge_blocks_device", "ksg_copy_map_device", "ksg_integrate_image", "ksg_set_update_log", "ksg_fetch_update_log", "ksg_evaluate_labels", "ksg_extract_mesh", "ksg_clear_map", "ksg_copy_update_log_device", "ksg_merge_voxels_device"]


def debug_chain_sum(terms: np.ndarray, s0: float, lib=None) -> np.float32:
    """One warp's exact scan of the float32 chain s <- fl(s + terms[k]) (ksg_debug_chain_sum); needs a device."""
    lib = lib or load_library()
    t = np.ascontiguousarray(terms, np.float32)
    out = np.zeros(1, np.float32)
    rc = lib.ksg_debug_chain_sum(_ptr(t, C.c_float), len(t), C.c_float(float(s0)), _ptr(out, C.c_float))
    if rc != 0:
        raise KsgError(f"ksg_debug_chain_sum failed: {KSG_STATUS.get(rc, rc)}")
    return out[0]


def unordered_map_schedule(n: int, lib=None) -> np.ndarray:
    """bucket_count() of the platform's std::unordered_map after each of n insertions (host only; KSG_BUNDLE_ORDER_LIBSTDCXX)."""
    lib = lib or load_library()
    out = np.zeros(n, np.int64)
    if lib.ksg_unordered_map_schedule(n, _ptr(out, C.c_int64)) != n:
        raise KsgError("ksg_unordered_map_schedule failed")
    return out


def owner_mask(block_index: np.ndarray, vps: int, shard_rank: int, shard_count: int, lib=None) -> np.ndarray:
    """[nb, vps^3] uint8 mask of the voxels rank `shard_rank` owns (spatial sharding)."""
    lib = lib or load_library()
    bi = np.ascontiguousarray(block_index, np.int32)
    mask = np.zeros((len(bi), vps ** 3), np.uint8)
    rc = lib.ksg_owner_mask(vps, shard_rank, shard_count, len(bi), _ptr(bi, C.c_int32), _ptr(mask, C.c_uint8))
    if rc != 0:
        raise ValueError(f"ksg_owner_mask: {rc}")
    return mask


def merge_shard_exports(exports, vps: int, lib=None) -> Dict[str, np.ndarray]:
    """Assemble the full map from the per-rank exports of a spatially sharded run (every rank allocates every block)."""
    G = len(exports)
    out = {k: v.copy() for k, v in exports[0].items()}
    for r in range(G):
        assert np.array_equal(exports[r]["block_index"], exports[0]["block_index"]), "ranks disagree on the block set"
        m = owner_mask(exports[r]["block_index"], vps, r, G, lib).astype(bool)
        for k in ("tsdf_distance", "tsdf_weight", "sem_label"):
            out[k][m] = exports[r][k][m]
        for k in ("tsdf_rgba", "sem_rgba", "sem_priors"):
            out[k][m] = exports[r][k][m]
    return out


class KsgError(RuntimeError):
    pass


def export_arrays(lib, handle, prefix: str, vps: int, num_labels: int) -> Dict[str, np.ndarray]:
    """Shared by the product binding and the oracle binding (same export signature)."""
    nb = int(getattr(lib, prefix + "_num_blocks")(handle))
    V = vps ** 3
    out = {
        "block_index": np.zeros((nb, 3), np.int32),
        "tsdf_distance": np.zeros((nb, V), np.float32),
        "tsdf_weight": np.zeros((nb, V), np.float32),
        "tsdf_rgba": np.zeros((nb, V, 4), np.uint8),
        "sem_label": np.zeros((nb, V), np.uint8),
        "sem_priors": np.zeros((nb, V, num_labels), np.float32),
        "sem_rgba": np.zeros((nb, V, 4), np.uint8),
    }
    rc = getattr(lib, prefix + "_export_blocks")(
        handle, nb, _ptr(out["block_index"], C.c_int32), _ptr(out["tsdf_distance"], C.c_float),
        _ptr(out["tsdf_weight"], C.c_float), _ptr(out["tsdf_rgba"], C.c_uint8), _ptr(out["sem_label"], C.c_uint8),
        _ptr(out["sem_priors"], C.c_float), _ptr(out["sem_rgba"], C.c_uint8))
    if rc != 0:
        raise KsgError(f"{prefix}_export_blocks failed: {rc}")
    return out


class Integrator:
    """Host-buffer view of one ksg integrator handle (numpy in, numpy out)."""

    def __init__(self, cfg: KsgConfig, lib=None):
        self.lib = lib or load_library()
        self.cfg = cfg
        self.handle = C.c_void_p()
        rc = self.lib.ksg_create(C.byref(cfg), C.byref(self.handle))
        if rc != 0:
            msg = self.lib.ksg_last_error(None)
            raise KsgError(f"ksg_create failed: {KSG_STATUS.get(rc, rc)}: {msg.decode() if msg else ''}")

    def close(self):
        if self.handle:
            self.lib.ksg_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str):
        if rc != 0:
            msg = self.lib.ksg_last_error(self.handle)
            raise KsgError(f"{what} failed: {KSG_STATUS.get(rc, rc)}: {msg.decode() if msg else ''}")

    def set_color_to_label(self, rgb: np.ndarray, labels: np.ndarray):
        rgb = np.ascontiguousarray(rgb, np.uint8)
        labels = np.ascontiguousarray(labels, np.uint8)
        self._check(self.lib.ksg_set_color_to_label(self.handle, _ptr(rgb, C.c_uint8), _ptr(labels, C.c_uint8), len(labels)),
                    "ksg_set_color_to_label")

    def integrate_points(self, T_G_C, xyz, rgba=None, labels=None, freespace=False) -> KsgFrameStats:
        T = np.ascontiguousarray(T_G_C, np.float32)
        xyz = np.ascontiguousarray(xyz, np.float32)
        rgba = None if rgba is None else np.ascontiguousarray(rgba, np.uint8)
        labels = None if labels is None else np.ascontiguousarray(labels, np.uint8)
        st = KsgFrameStats()
        self._check(self.lib.ksg_integrate_points(self.handle, _ptr(T, C.c_float), _ptr(xyz, C.c_float), _ptr(rgba, C.c_uint8),
                                                  _ptr(labels, C.c_uint8), xyz.shape[0], int(freespace), C.byref(st)),
                    "ksg_integrate_points")
        return st

    def integrate_depth(self, T_G_C, depth, label, K) -> KsgFrameStats:
        T = np.ascontiguousarray(T_G_C, np.float32)
        depth = np.ascontiguousarray(depth, np.float32)
        label = np.ascontiguousarray(label, np.uint8)
        K = np.ascontiguousarray(K, np.float32)
        st = KsgFrameStats()
        h, w = depth.shape
        self._check(self.lib.ksg_integrate_depth(self.handle, _ptr(T, C.c_float), _ptr(depth, C.c_float), _ptr(label, C.c_uint8),
                                                 w, h, _ptr(K, C.c_float), C.byref(st)), "ksg_integrate_depth")
        return st

    def integrate_image(self, T_G_C, depth, semantic, K64) -> KsgFrameStats:
        """depth: float32 metres or uint16 millimetres [h, w]; semantic: uint8 labels [h, w] or RGB8 [h, w, 3] (ksg_integrate_image)."""
        T = np.ascontiguousarray(T_G_C, np.float32)
        K = np.ascontiguousarray(K64, np.float64)
        depth = np.ascontiguousarray(depth)
        semantic = np.ascontiguousarray(semantic, np.uint8)
        assert depth.dtype in (np.float32, np.uint16)
        h, w = depth.shape
        st = KsgFrameStats()
        self._check(self.lib.ksg_integrate_image(self.handle, _ptr(T, C.c_float), depth.ctypes.data_as(C.c_void_p), 1 if depth.dtype == np.uint16 else 0,
                                                 semantic.ctypes.data_as(C.c_void_p), 1 if semantic.ndim == 3 else 0, w, h, _ptr(K, C.c_double), C.byref(st)),
                    "ksg_integrate_image")
        return st

    def integrate_depth_async(self, T_G_C, depth, label, K):
        """Pipelined host-buffer entry: returns once the frame is enqueued; wait_frame() completes the oldest outstanding frame."""
        T = np.ascontiguousarray(T_G_C, np.float32)
        K = np.ascontiguousarray(K, np.float32)
        h, w = depth.shape
        self._check(self.lib.ksg_integrate_depth_async(self.handle, _ptr(T, C.c_float), _ptr(depth, C.c_float), _ptr(label, C.c_uint8),
                                                       w, h, _ptr(K, C.c_float)), "ksg_integrate_depth_async")

    def wait_frame(self) -> KsgFrameStats:
        st = KsgFrameStats()
        self._check(self.lib.ksg_wait_frame(self.handle, C.byref(st)), "ksg_wait_frame")
        return st

    def integrate_depth_k64(self, T_G_C, depth, label, K64) -> KsgFrameStats:
        """Depth entry with float64 intrinsics (fx fy cx cy), as sensor_msgs/CameraInfo holds them."""
        T = np.ascontiguousarray(T_G_C, np.float32)
        depth = np.ascontiguousarray(depth, np.float32)
        label = np.ascontiguousarray(label, np.uint8)
        K = np.ascontiguousarray(K64, np.float64)
        st = KsgFrameStats()
        h, w = depth.shape
        self._check(self.lib.ksg_integrate_depth_k64(self.handle, _ptr(T, C.c_float), _ptr(depth, C.c_float), _ptr(label, C.c_uint8),
                                                     w, h, _ptr(K, C.c_double), C.byref(st)), "ksg_integrate_depth_k64")
        return st

    def integrate_depth_device(self, T_G_C, d_depth_ptr: int, d_label_ptr: int, width: int, height: int, K,
                               stream: int = 0, want_stats: bool = False) -> Optional[KsgFrameStats]:
        T = np.ascontiguousarray(T_G_C, np.float32)
        K = np.ascontiguousarray(K, np.float32)
        st = KsgFrameStats() if want_stats else None
        self._check(self.lib.ksg_integrate_depth_device(self.handle, _ptr(T, C.c_float), C.c_void_p(d_depth_ptr),
                                                        C.c_void_p(d_label_ptr), width, height, _ptr(K, C.c_float),
                                                        C.c_void_p(stream), C.byref(st) if st is not None else None),
                    "ksg_integrate_depth_device")
        return st

    def integrate_points_device(self, T_G_C, d_xyz: int, d_rgba: int, d_labels: int, n: int, freespace=False,
                                stream: int = 0, want_stats: bool = False) -> Optional[KsgFrameStats]:
        T = np.ascontiguousarray(T_G_C, np.float32)
        st = KsgFrameStats() if want_stats else None
        self._check(self.lib.ksg_integrate_points_device(self.handle, _ptr(T, C.c_float), C.c_void_p(d_xyz),
                                                         C.c_void_p(d_rgba) if d_rgba else None,
                                                         C.c_void_p(d_labels) if d_labels else None, n, int(freespace),
                                                         C.c_void_p(stream), C.byref(st) if st is not None else None),
                    "ksg_integrate_points_device")
        return st

    PHASES = ("classify+start_set", "fixpoint|bundling", "ray_emit", "record_sort", "alloc+tile_heads", "tile_apply", "frame")

    def set_profiling(self, enable: bool):
        self._check(self.lib.ksg_set_profiling(self.handle, int(enable)), "ksg_set_profiling")

    def get_profile(self) -> Dict[str, float]:
        ms = (C.c_double * 7)()
        frames, launches, libcalls = C.c_int64(), C.c_int64(), C.c_int64()
        self._check(self.lib.ksg_get_profile(self.handle, ms, C.byref(frames), C.byref(launches), C.byref(libcalls)), "ksg_get_profile")
        out = {n: float(ms[i]) for i, n in enumerate(self.PHASES)}
        out["frames"] = int(frames.value)
        out["kernel_launches"] = int(launches.value)
        out["library_calls"] = int(libcalls.value)
        return out

    def fast_timeline(self) -> Dict[str, object]:
        """Phase boundaries of the last frame's persistent solve kernel in microseconds from its start (fast integrator, profiling on)."""
        out = (C.c_int64 * 112)()
        sweeps, khz = C.c_int64(), C.c_double()
        n = int(self.lib.ksg_debug_fast_timeline(self.handle, out, C.byref(sweeps), C.byref(khz)))
        if n == 0:
            return {}
        t = [int(v) for v in out]
        us = lambda a, b: (t[b] - t[a]) / (khz.value / 1e3)
        ns = int(sweeps.value)
        return {"sweeps": ns, "compact_us": us(0, 1), "ray_setup_us": us(1, 2),
                "sweep_us": [us(2 + i, 3 + i) for i in range(max(0, min(ns, 48)))],
                "commit_emit_us": us(52, 53), "tile_count_us": us(53, 54), "tile_alloc_block_init_us": us(54, 55), "scatter_us": us(55, 56),
                "solve_kernel_us": us(0, 56),
                "phase0_us": {"file_shared_slot_visitors": us(0, 57) if t[57] else None, "sort_shared_slots": us(57, 58) if t[58] else None,
                              "scan_cast_counts": us(58 if t[58] else 0, 59), "compaction": us(59, 1)},
                "debug": {"max_ray_setup_us": t[64] / (khz.value / 1e3), "max_ray_setup_insert_us": t[65] / (khz.value / 1e3),
                          "max_ray_eval_us": t[67] / (khz.value / 1e3), "ray_evals": t[68], "blocks_evaluated": t[69], "blocks_materialised": t[70],
                          "ray_evals_that_changed": t[71], "max_shared_slot_visitors": t[72], "shared_slot_visitors": t[73],
                          "shared_slots": t[74], "rays": t[75],
                          "max_setup_after_loads_us": t[76] / (khz.value / 1e3), "max_setup_after_init_us": t[77] / (khz.value / 1e3),
                          "max_setup_after_loop_us": t[78] / (khz.value / 1e3), "max_eval_first_block_loads_us": t[79] / (khz.value / 1e3),
                          "overflow_entries": t[80], "max_slot_count": t[81], "max_overflow_chain_walked": t[82],
                          "sweep_clean_rays": [t[84 + 2 * i] for i in range(max(0, min(ns, 14)))],
                          "sweep_ray_evals": [t[85 + 2 * i] for i in range(max(0, min(ns, 14)))]}}

    def sync(self):
        self._check(self.lib.ksg_sync(self.handle), "ksg_sync")

    def reset(self):
        self._check(self.lib.ksg_reset(self.handle), "ksg_reset")

    def num_blocks(self) -> int:
        return int(self.lib.ksg_num_blocks(self.handle))

    def export(self) -> Dict[str, np.ndarray]:
        return export_arrays(self.lib, self.handle, "ksg", self.cfg.voxels_per_side, self.cfg.num_labels)

    def import_blocks(self, exp: Dict[str, np.ndarray]):
        """Write an export (dict as returned by export()) into this integrator's map."""
        a = {k: np.ascontiguousarray(v) for k, v in exp.items()}
        self._check(self.lib.ksg_import_blocks(self.handle, len(a["block_index"]), _ptr(a["block_index"].astype(np.int32), C.c_int32),
                                               _ptr(a["tsdf_distance"], C.c_float), _ptr(a["tsdf_weight"], C.c_float),
                                               _ptr(a["tsdf_rgba"], C.c_uint8), _ptr(a["sem_label"], C.c_uint8),
                                               _ptr(a["sem_priors"], C.c_float), _ptr(a["sem_rgba"], C.c_uint8)), "ksg_import_blocks")

    def device_map_view(self):
        """(n_blocks, block_stride_bytes, pool pointer, block-key pointer) of the device-resident map (frame-per-GPU batch mode)."""
        nb, stride, pool, keys = C.c_int64(), C.c_int64(), C.c_void_p(), C.c_void_p()
        self._check(self.lib.ksg_device_map_view(self.handle, C.byref(nb), C.byref(stride), C.byref(pool), C.byref(keys)), "ksg_device_map_view")
        return int(nb.value), int(stride.value), int(pool.value or 0), int(keys.value or 0)

    def copy_map_device(self, d_pool: int, d_keys: int, stream: int = 0):
        self._check(self.lib.ksg_copy_map_device(self.handle, C.c_void_p(d_pool), C.c_void_p(d_keys), C.c_void_p(stream)), "ksg_copy_map_device")

    def merge_blocks_device(self, n_blocks: int, d_keys: int, d_pool: int, stream: int = 0):
        self._check(self.lib.ksg_merge_blocks_device(self.handle, n_blocks, C.c_void_p(d_keys), C.c_void_p(d_pool), C.c_void_p(stream)),
                    "ksg_merge_blocks_device")

    def set_update_log(self, capacity_voxels: int):
        self._check(self.lib.ksg_set_update_log(self.handle, capacity_voxels), "ksg_set_update_log")

    def fetch_update_log(self):
        """(heads structured array [n], priors [n, C]) of the voxels the last frame updated (copies)."""
        n, heads, pri = C.c_int64(), C.c_void_p(), C.POINTER(C.c_float)()
        self._check(self.lib.ksg_fetch_update_log(self.handle, C.byref(n), C.byref(heads), C.byref(pri)), "ksg_fetch_update_log")
        dt = np.dtype([("block_index", np.int32, 3), ("lin_label", np.uint32), ("tsdf_distance", np.float32), ("tsdf_weight", np.float32),
                       ("tsdf_rgba", np.uint8, 4), ("sem_rgba", np.uint8, 4)])
        k = int(n.value)
        if k == 0:
            return np.zeros(0, dt), np.zeros((0, self.cfg.num_labels), np.float32)
        h = np.frombuffer((C.c_uint8 * (k * dt.itemsize)).from_address(heads.value), dtype=dt).copy()
        p = np.ctypeslib.as_array(pri, shape=(k, self.cfg.num_labels)).copy()
        return h, p

    WORLD_DTYPE = np.dtype([("type", np.int32), ("a", np.float32, 3), ("b", np.float32, 3), ("label", np.int32)])

    def evaluate_labels(self, objects: np.ndarray, max_dist: float, band: float, checker_size: float = 0.0, checker_margin: float = 0.0):
        """(evaluated, correct, observed) voxel counts of the map's labels against an analytic world (ksg_evaluate_labels)."""
        objs = np.ascontiguousarray(objects, self.WORLD_DTYPE)
        ev, ok, ob = C.c_int64(), C.c_int64(), C.c_int64()
        self._check(self.lib.ksg_evaluate_labels(self.handle, objs.ctypes.data_as(C.c_void_p), len(objs), max_dist, band, checker_size, checker_margin,
                                                 C.byref(ev), C.byref(ok), C.byref(ob)), "ksg_evaluate_labels")
        return int(ev.value), int(ok.value), int(ob.value)

    def update_log_size(self) -> int:
        n = C.c_int64()
        self._check(self.lib.ksg_copy_update_log_device(self.handle, C.byref(n), None, None, 0, None), "ksg_copy_update_log_device")
        return int(n.value)

    def copy_update_log_device(self, d_updates: int, d_priors: int, capacity: int, stream: int = 0) -> int:
        """Copy the last frame's update log (32-byte entries, num_labels floats each) into device buffers; returns the entry count."""
        n = C.c_int64()
        self._check(self.lib.ksg_copy_update_log_device(self.handle, C.byref(n), C.c_void_p(d_updates), C.c_void_p(d_priors), capacity, C.c_void_p(stream)),
                    "ksg_copy_update_log_device")
        return int(n.value)

    def merge_voxels_device(self, counts, stride: int, d_updates: int, d_priors: int, stream: int = 0):
        """Merge len(counts) voxel-granular deltas (delta g at entry offset g * stride) into this map, in order (ksg_merge_voxels_device)."""
        arr = (C.c_int64 * len(counts))(*[int(c) for c in counts])
        self._check(self.lib.ksg_merge_voxels_device(self.handle, len(counts), arr, stride, C.c_void_p(d_updates), C.c_void_p(d_priors), C.c_void_p(stream)),
                    "ksg_merge_voxels_device")

    def clear_map(self):
        """Remove every block, keep the integrator state (ksg_clear_map)."""
        self._check(self.lib.ksg_clear_map(self.handle), "ksg_clear_map")

    def extract_mesh(self, min_weight: float = 1e-4):
        """Semantic mesh of the map (ksg_extract_mesh): dict(vertices [n, 3] f32 - three consecutive vertices per triangle, rgba [n, 4] u8,
        labels [n] u8, block_index [nb, 3] i32 in (z, y, x) order, block_first [nb + 1] i64)."""
        nv, nb = C.c_int64(), C.c_int64()
        self._check(self.lib.ksg_extract_mesh(self.handle, min_weight, 0, None, None, None, 0, None, None, C.byref(nv), C.byref(nb)), "ksg_extract_mesh")
        n, b = int(nv.value), int(nb.value)
        vtx = np.zeros((n, 3), np.float32); rgba = np.zeros((n, 4), np.uint8); lab = np.zeros(n, np.uint8)
        bidx = np.zeros((b, 3), np.int32); first = np.zeros(b + 1, np.int64)
        self._check(self.lib.ksg_extract_mesh(self.handle, min_weight, n, vtx.ctypes.data_as(C.c_void_p), rgba.ctypes.data_as(C.c_void_p),
                                              lab.ctypes.data_as(C.c_void_p), b, bidx.ctypes.data_as(C.c_void_p), first.ctypes.data_as(C.c_void_p),
                                              C.byref(nv), C.byref(nb)), "ksg_extract_mesh")
        return {"vertices": vtx, "rgba": rgba, "labels": lab, "block_index": bidx, "block_first": first}

    def last_updated_blocks(self) -> np.ndarray:
        n = int(self.lib.ksg_last_updated_blocks(self.handle, 0, None))
        out = np.zeros((n, 3), np.int32)
        if n:
            self.lib.ksg_last_updated_blocks(self.handle, n, _ptr(out, C.c_int32))
        return out
