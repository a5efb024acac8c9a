/*
 * ksg.h — C-ABI of the B200-native semantic TSDF integrator ("ksg" = Kimera-Semantics on GPU).
 *
 * This header is the drop-in boundary. Everything above it (the C++ classes in
 * kimera_semantics_b200/cpp that mirror kimera::FastSemanticTsdfIntegrator /
 * kimera::MergedSemanticTsdfIntegrator / kimera::SemanticTsdfIntegratorFactory) is a thin
 * host shim; everything below it is hand-written sm_100a CUDA.  Signatures use plain
 * pointers and sizes only (no torch / Eigen / voxblox types).
 *
 * Each entry point cites the reference interface it replaces (paths relative to the
 * reference checkout, see SURVEY.md for the abbreviations):
 *   fast.cpp   = kimera_semantics/src/semantic_tsdf_integrator_fast.cpp
 *   merged.cpp = kimera_semantics/src/semantic_tsdf_integrator_merged.cpp
 *   base.cpp/h = kimera_semantics/{src,include/kimera_semantics}/semantic_integrator_base.*
 *   factory.*  = kimera_semantics/{src,include/kimera_semantics}/semantic_tsdf_integrator_factory.*
 */
#ifndef KSG_H_
#define KSG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KSG_ABI_VERSION 1

/* status codes (the reference aborts through glog CHECK; the C++ shim turns non-zero
 * codes back into aborts, the C-ABI itself never throws / aborts) */
enum {
  KSG_OK = 0,
  KSG_ERR_INVALID_ARGUMENT = 1, /* reference: CHECK failures base.cpp:74,80,98-107; factory.cpp:61,83 */
  KSG_ERR_CUDA = 2,
  KSG_ERR_POOL_FULL = 3,       /* device block pool / hash table exhausted */
  KSG_ERR_SCRATCH_FULL = 4,    /* per-frame scratch exhausted (grow max_* in the config) */
  KSG_ERR_INDEX_RANGE = 5,     /* a voxel index left the packed-key range (|idx| >= 2^20 blocks) */
  KSG_ERR_NO_DEVICE = 6
};

/* integrator types: factory.h:49-54 (kMerged = 0, kFast = 1) */
enum { KSG_INTEGRATOR_MERGED = 0, KSG_INTEGRATOR_FAST = 1 };
/* colour modes: base.h:54-58 */
enum { KSG_COLOR_MODE_COLOR = 0, KSG_COLOR_MODE_SEMANTIC = 1, KSG_COLOR_MODE_SEMANTIC_PROBABILITY = 2 };
/* integration order: voxblox ThreadSafeIndexFactory ("mixed" | "sorted"), fast.cpp:172-174 */
enum { KSG_ORDER_MIXED = 0, KSG_ORDER_SORTED = 1 };
/* ksg_config.merged_bundle_order */
enum { KSG_BUNDLE_ORDER_CANONICAL = 0, KSG_BUNDLE_ORDER_LIBSTDCXX = 1 };

/*
 * One POD that carries vxb::TsdfIntegratorBase::Config (voxblox tsdf_integrator.h, defaults in
 * SURVEY.md A.6), kimera::SemanticIntegratorBase::SemanticConfig (base.h:68-87), the layer
 * geometry (vxb::Layer ctor: voxel_size, voxels_per_side; ros/src/semantic_tsdf_server.cpp:68-69)
 * and the run-time class count that replaces the compile-time kTotalNumberOfLabels (common.h:26).
 */
typedef struct ksg_config {
  int32_t abi_version;                 /* must be KSG_ABI_VERSION */
  int32_t integrator_type;             /* KSG_INTEGRATOR_* (factory.h:49-54) */
  /* layer geometry */
  float voxel_size;                    /* metres */
  int32_t voxels_per_side;             /* power of two */
  /* vxb::TsdfIntegratorBase::Config */
  float default_truncation_distance;
  float max_weight;
  int32_t voxel_carving_enabled;
  float min_ray_length_m;
  float max_ray_length_m;
  int32_t use_const_weight;
  int32_t allow_clear;
  int32_t use_weight_dropoff;
  int32_t use_sparsity_compensation_factor;
  float sparsity_compensation_factor;
  int32_t integration_order_mode;      /* KSG_ORDER_* */
  int32_t enable_anti_grazing;         /* merged only (merged.cpp:306-313) */
  float start_voxel_subsampling_factor;      /* fast only (fast.cpp:87-92) */
  int32_t max_consecutive_ray_collisions;    /* fast only (fast.cpp:115-122) */
  int32_t clear_checks_every_n_frames;       /* fast only (fast.cpp:165-170) */
  int32_t integrator_threads;          /* CPU oracle only; the GPU path ignores it */
  /* kimera SemanticConfig */
  int32_t num_labels;                  /* C, 2..256 (reference: constexpr 21) */
  float semantic_measurement_probability;    /* base.h:77 */
  int32_t color_mode;                  /* KSG_COLOR_MODE_* */
  uint8_t label_color[256][4];         /* SemanticLabel2Color label -> RGBA (color.cpp:84-94) */
  uint8_t label_color_known[256];      /* 0 -> lookup miss: colour (0,0,0,0), color.cpp:92 */
  uint8_t dynamic_label[256];          /* 1 -> label is dynamic; fast skips it (base.h:170-175) */
  /* device side sizing (GPU path only) */
  int32_t device;                      /* CUDA device ordinal */
  int32_t max_blocks;                  /* block pool capacity (blocks of voxels_per_side^3) */
  int32_t max_points;                  /* largest cloud / frame (pixels) accepted */
  int64_t max_ray_steps;               /* scratch: upper bound on ray-step candidates per frame */
  int64_t max_updates;                 /* scratch: upper bound on voxel updates per frame */
  int32_t apply_mode;                  /* 0 = TMA-staged tile apply (default), 1 = cooperative-copy staging */
  /* spatial hash-block sharding of ONE map over several GPUs (SURVEY.md 8e): every rank receives every frame and casts every
   * ray, but applies only the 8^3 tiles it owns (owner = f(block index, tile)); results per voxel are identical to the
   * unsharded run. shard_count <= 1: off. */
  int32_t shard_rank;
  int32_t shard_count;
  /* merged only: the order in which the bundles of a frame are applied (per-voxel results depend on it, updateTsdfVoxel clamps
   * after averaging).  KSG_BUNDLE_ORDER_CANONICAL (0): first-insertion order of bundleRays.
   * KSG_BUNDLE_ORDER_LIBSTDCXX (1, default since round 2): the iteration order of the std::unordered_map<LongIndex, ..., LongIndexHash> the reference
   * fills in bundleRays and walks in integrateVoxels (merged.cpp:110-124, 210-231) - i.e. the reference's result with
   * integrator_threads = 1 on a platform whose libstdc++ has this library's rehash policy. */
  int32_t merged_bundle_order;
  /* merged only, C <= 32, apply_mode 0.  1 = the semantic log-probability rows of the few voxels that receive thousands of updates in
   * one frame (the voxels next to the camera) are computed by a parallel pre-pass (an exact scan of the float addition chain,
   * csrc/ksg_hot.cuh) instead of one warp's sequential loop; results are bit-identical.  2 = additionally, a hot voxel that sits at
   * (distance, weight) = (+truncation, max_weight) is CHECKED in parallel to be left untouched by every record of the frame, and
   * its sequential TSDF recurrence is then skipped.  0 (default) = off.  Experimental: written at the end of round 1, not yet
   * measured. */
  int32_t hot_voxel_mode;
  int32_t reserved[3];
} ksg_config;

/* per-frame counters (the oracle reports the same numbers; SURVEY.md 8d: one voxel update =
 * one {updateTsdfVoxel; updateSemanticVoxel} pair, fast.cpp:124-140 / merged.cpp:315-327) */
typedef struct ksg_frame_stats {
  int64_t points_in;          /* points handed to integratePointCloud */
  int64_t points_valid;       /* passed isPointValid (+ dynamic-label filter for fast) */
  int64_t rays_cast;          /* fast: rays surviving the start-voxel set; merged: bundles (both passes) */
  int64_t ray_steps;          /* candidate ray steps enumerated */
  int64_t voxel_updates;      /* executed per-voxel update bodies */
  int64_t blocks_allocated;   /* blocks in the map after this frame */
  int64_t blocks_touched;     /* blocks that received >= 1 update this frame */
  int64_t tiles_touched;      /* 8^3 tiles staged by the apply kernel */
  int64_t fixpoint_iterations;/* fast: iterations of the observed-set solver */
  int64_t hot_voxels;         /* merged, hot_voxel_mode = 1: voxels whose semantic row was finished by the pre-pass this frame */
  int64_t hot_fallback_chunks;/* ... and how many of their 1024-record chunks had to be re-evaluated sequentially (cumulative) */
  int64_t reserved[5];
} ksg_frame_stats;

typedef struct ksg_integrator ksg_integrator; /* opaque */

/* Fill *cfg with the voxblox / kimera defaults (SURVEY.md A.6, base.h:77-86) for the given
 * geometry: truncation 4*voxel_size as voxblox_ros sets it, p = 0.9, colour mode kSemantic,
 * label colours = grey for every label (known), no dynamic labels. */
void ksg_default_config(ksg_config* cfg, int32_t integrator_type, float voxel_size,
                        int32_t voxels_per_side, int32_t num_labels);

/* Replaces SemanticTsdfIntegratorFactory::create (factory.h:71-93, factory.cpp:43-88) together with
 * the Fast/Merged constructors (fast.cpp:49-55, merged.cpp:56-62) and SemanticIntegratorBase's
 * ctor (base.cpp:57-76: layer geometry cache + setSemanticProbabilities base.cpp:93-128).
 * The map (both layers) lives in device memory owned by the returned object. */
int32_t ksg_create(const ksg_config* cfg, ksg_integrator** out);
void ksg_destroy(ksg_integrator* h);

/* Human-readable description of the last non-OK status on this handle (NULL handle: global). */
const char* ksg_last_error(const ksg_integrator* h);

/* Replaces  virtual void integratePointCloud(const Transformation& T_G_C, const Pointcloud& points_C,
 *           const Colors& colors, const bool freespace_points)       fast.h:82-86, merged.h:70-73
 * (bodies fast.cpp:145-199, merged.cpp:65-149).
 *   T_G_C      : 7 floats  qw qx qy qz tx ty tz  (minkindr QuatTransformation<float>)
 *   xyz        : n*3 floats, camera frame
 *   rgba       : n*4 bytes or NULL. When labels == NULL the label of a point is looked up from its
 *                colour through the table set with ksg_set_color_to_label (fast.cpp:152-158).
 *   labels     : n bytes or NULL. merged.h:82-86 label-explicit overload.  With rgba AND labels the merged integrator keeps the colours out
 *                of the TSDF layer (they are blended per bundle in the reference, merged.cpp:262-274): exact in ColorMode kSemantic /
 *                kSemanticProbability, where the TSDF colour is overwritten anyway; in ColorMode::kColor that combination is rejected with
 *                KSG_ERR_INVALID_ARGUMENT.
 * Host buffers; the call copies them to the device, integrates and returns after the device
 * finished (the reference call is synchronous, SURVEY.md 8b "Threading"). */
int32_t ksg_integrate_points(ksg_integrator* h, const float* T_G_C, const float* xyz,
                             const uint8_t* rgba, const uint8_t* labels, int64_t n,
                             int32_t freespace_points, ksg_frame_stats* stats);

/* Same call with DEVICE buffers, enqueued on `cuda_stream` (a cudaStream_t passed as void*).  `fast`: the frame has no host read-back, the
 * call returns as soon as it is enqueued unless stats != NULL (then it waits for the frame); a device-side error surfaces at the next call
 * that completes a frame (ksg_sync, ksg_wait_frame, an export, ...).  `merged`: the call reads the record count back once and returns when
 * the frame is enqueued behind it.  Used by bench.py's device-resident leg. */
int32_t ksg_integrate_points_device(ksg_integrator* h, const float* T_G_C_host, const float* d_xyz,
                                    const uint8_t* d_rgba, const uint8_t* d_labels, int64_t n,
                                    int32_t freespace_points, void* cuda_stream, ksg_frame_stats* stats);

/* Depth + label frame entry (SURVEY.md 8f NEXT-1): fuses PointCloudFromDepth::convert<float>
 * (kimera_semantics_ros/include/kimera_semantics_ros/depth_map_to_pointcloud.h:222-266; x=(u-cx)*d*(1/fx),
 * y=(v-cy)*d*(1/fy), z=d, non-finite depth -> dropped point as voxblox_ros convertPointcloud does)
 * with integratePointCloud.  depth: h*w float32 metres, label: h*w uint8, K = fx fy cx cy.
 * Precision note: the reference derives constant_x = float(1.0 / fx) from the DOUBLE fx of sensor_msgs/CameraInfo and
 * center_x = float(cx) (depth_map_to_pointcloud.h:222-230).  The *_k64 variants below take the intrinsics as double and
 * reproduce that exactly; the float-K entries are the same call with K widened, i.e. bit-identical to the reference when the
 * intrinsics are representable in float (integral / half-integral values) and up to one float ulp off in 1/fx otherwise
 * (e.g. fx = 415.69219381653056 of a 60-degree, 480-line simulator camera). */
int32_t ksg_integrate_depth(ksg_integrator* h, const float* T_G_C, const float* depth,
                            const uint8_t* label, int32_t width, int32_t height, const float* K,
                            ksg_frame_stats* stats);
int32_t ksg_integrate_depth_device(ksg_integrator* h, const float* T_G_C_host, const float* d_depth,
                                   const uint8_t* d_label, int32_t width, int32_t height,
                                   const float* K_host, void* cuda_stream, ksg_frame_stats* stats);
/* The same two calls with double intrinsics (K = fx fy cx cy as float64, the type of sensor_msgs/CameraInfo::K). */
int32_t ksg_integrate_depth_k64(ksg_integrator* h, const float* T_G_C, const float* depth,
                                const uint8_t* label, int32_t width, int32_t height, const double* K,
                                ksg_frame_stats* stats);
int32_t ksg_integrate_depth_device_k64(ksg_integrator* h, const float* T_G_C_host, const float* d_depth,
                                       const uint8_t* d_label, int32_t width, int32_t height,
                                       const double* K_host, void* cuda_stream, ksg_frame_stats* stats);

/* Generic image entry (host buffers): the two depth encodings and the two semantic encodings the reference's front end accepts
 * (kimera_semantics_ros/include/kimera_semantics_ros/depth_map_to_pointcloud.h:183-193: TYPE_32FC1 / TYPE_16UC1; semantic image = RGB8 colour
 * image whose colours name the labels, fast.cpp:152-158).  uint16 depth follows depth_image_proc::DepthTraits<uint16_t>: 0 = invalid,
 * metres = depth * 0.001f, x = (u - cx) * depth * float(double(0.001f) / fx) (depth_map_to_pointcloud.h:222-230,259-265).  With an RGB
 * semantic image every pixel's label comes from the table of ksg_set_color_to_label (unknown colour -> label 0) and the point carries the
 * image colour, exactly as integratePointCloud(points_C, colors) receives it.  K = fx fy cx cy (float64). */
enum { KSG_DEPTH_F32_METRES = 0, KSG_DEPTH_U16_MILLIMETRES = 1 };
enum { KSG_SEMANTIC_LABEL_U8 = 0, KSG_SEMANTIC_RGB8 = 1 };
int32_t ksg_integrate_image(ksg_integrator* h, const float* T_G_C, const void* depth, int32_t depth_type, const void* semantic,
                            int32_t semantic_type, int32_t width, int32_t height, const double* K, ksg_frame_stats* stats);

/* Pipelined variant of ksg_integrate_depth for a camera stream: enqueues the host->device copy of THIS frame on a copy stream (so it
 * overlaps the kernels of the previous frame) and the frame's kernels behind it, and returns without waiting; at most two frames are in
 * flight.  ksg_wait_frame completes the OLDEST outstanding frame and returns its statistics / status (the reference call is synchronous:
 * a caller that needs those semantics calls ksg_wait_frame right after, or uses ksg_integrate_depth).  Page-locked caller buffers are read
 * asynchronously and must stay unchanged until the frame's ksg_wait_frame returns; pageable buffers are staged before the call returns. */
int32_t ksg_integrate_depth_async(ksg_integrator* h, const float* T_G_C, const float* depth, const uint8_t* label,
                                  int32_t width, int32_t height, const float* K);
int32_t ksg_wait_frame(ksg_integrator* h, ksg_frame_stats* stats);

/* Colour -> label table: SemanticLabel2Color::getSemanticLabelFromColor (color.cpp:69-82). n entries
 * of (r,g,b) -> label (alpha is forced to 255 by the callers fast.cpp:157, merged.cpp:87). A colour
 * that is not in the table maps to label 0 (color.cpp:80). */
int32_t ksg_set_color_to_label(ksg_integrator* h, const uint8_t* rgb, const uint8_t* labels, int32_t n);

/* Wait for all enqueued work of this integrator; returns a deferred device-side error if any. */
int32_t ksg_sync(ksg_integrator* h);

/* Map read-back: replaces the direct host reads of Layer<TsdfVoxel> / Layer<SemanticVoxel> that
 * callers perform after integratePointCloud returns (SURVEY.md 8b "Ownership"; base.cpp:257-265
 * merges the blocks into the host layer).  Blocks come out sorted by (z, y, x) block index; voxels in
 * voxblox linear order x + vps*(y + vps*z).  Any output pointer may be NULL.
 *   block_index  nb*3 int32
 *   tsdf_distance, tsdf_weight  nb*V float ;  tsdf_rgba nb*V*4 uint8           (vxb::TsdfVoxel)
 *   sem_label nb*V uint8 ; sem_priors nb*V*C float ; sem_rgba nb*V*4 uint8     (semantic_voxel.h:14-27)
 */
int64_t ksg_num_blocks(ksg_integrator* h);
int32_t ksg_export_blocks(ksg_integrator* h, int64_t capacity_blocks, int32_t* block_index,
                          float* tsdf_distance, float* tsdf_weight, uint8_t* tsdf_rgba,
                          uint8_t* sem_label, float* sem_priors, uint8_t* sem_rgba);
/* Same outputs for an explicit list of n block indices (n*3 int32), in list order; found[i] = 0 and the
 * outputs of block i are left untouched when the block is not allocated.  Used by the C++ shim to refresh
 * only the blocks an integrate call updated (SURVEY.md 8f NEXT-3). */
int32_t ksg_export_blocks_by_index(ksg_integrator* h, int64_t n, const int32_t* block_index, uint8_t* found,
                                   float* tsdf_distance, float* tsdf_weight, uint8_t* tsdf_rgba,
                                   uint8_t* sem_label, float* sem_priors, uint8_t* sem_rgba);
/* Inverse of ksg_export_blocks_by_index: writes n blocks (same layouts) into the device map, allocating the blocks that do not
 * exist yet (a NULL array leaves that field untouched / default-constructed for new blocks).  Restores a saved map the way the
 * reference reloads a TSDF layer (kimera_semantics_ros/src/semantic_simulation_server.cpp:57-88); SURVEY.md 8f NEXT-3.  The
 * fast integrator's two approximate sets are not part of a map and start empty, exactly as in a freshly constructed reference
 * integrator. */
int32_t ksg_import_blocks(ksg_integrator* h, int64_t n, const int32_t* block_index, const float* tsdf_distance,
                          const float* tsdf_weight, const uint8_t* tsdf_rgba, const uint8_t* sem_label,
                          const float* sem_priors, const uint8_t* sem_rgba);
/* Frame-per-GPU batch mode (SURVEY.md 8e row 1; DESIGN.md section 8).  ksg_device_map_view exposes this integrator's map as device
 * memory without a copy: its n_blocks blocks in pool layout (block_stride_bytes each, tiles of [distance | weight | rgba | sem rgba | label |
 * log-probabilities]) and one packed 64-bit block key per block - the payload a rank sends to its peers.  ksg_merge_blocks_device merges such a
 * payload (device memory of THIS device, e.g. the receive buffer of an all-gather) into this integrator's map voxel by voxel: TSDF by
 * voxblox's mergeVoxelAIntoVoxelB (weighted mean, blended colour, weight capped at max_weight), labels by adding the payload's accumulated
 * log-likelihoods (base.cpp:283-314) followed by arg-max and the colour hand-off; blocks the map does not hold yet are created.  Payloads are
 * merged in the order of the calls.  Both integrators must share voxel size, voxels_per_side and num_labels. */
int32_t ksg_device_map_view(ksg_integrator* h, int64_t* n_blocks, int64_t* block_stride_bytes, void** d_pool, void** d_block_keys);
int32_t ksg_merge_blocks_device(ksg_integrator* h, int64_t n_blocks, const void* d_block_keys, const void* d_pool_src, void* cuda_stream);
/* Copies the payload of ksg_device_map_view (n_blocks * block_stride_bytes, n_blocks keys) into caller-owned device buffers on `cuda_stream`
 * (e.g. the send buffer of the all-gather). */
int32_t ksg_copy_map_device(ksg_integrator* h, void* d_dst_pool, void* d_dst_keys, void* cuda_stream);

/* Update log: the cheap way to keep HOST layers in step with the device map after every call (the reference's contract, base.cpp:257-265:
 * on return the caller reads the host Layer<> objects).  With a log of `capacity_voxels` entries switched on, every integrate call of the
 * `fast` integrator leaves one entry per voxel it updated (final distance, weight, colours, label and log-probabilities): kilobytes to a
 * few megabytes per frame instead of whole blocks.  ksg_fetch_update_log completes the last frame, copies its entries to page-locked host
 * memory owned by the library (two DMA transfers) and returns pointers that stay valid until the next call on this handle; *n = -1 and
 * KSG_ERR_SCRATCH_FULL when the frame updated more voxels than the log holds (use the block export then).  capacity 0 switches it off. */
typedef struct ksg_voxel_update {
  int32_t block_index[3];
  uint32_t lin_label;       /* voxblox linear voxel index x + vps*(y + vps*z) in bits 0..23, semantic label in bits 24..31 */
  float tsdf_distance, tsdf_weight;
  uint8_t tsdf_rgba[4], sem_rgba[4];
} ksg_voxel_update;
int32_t ksg_set_update_log(ksg_integrator* h, int64_t capacity_voxels);
int32_t ksg_fetch_update_log(ksg_integrator* h, int64_t* n, const ksg_voxel_update** updates, const float** sem_priors /* n * num_labels */);

/* Voxel-granular deltas for the frame-per-GPU batch mode (DESIGN.md 8): the update log of a frame integrated into EMPTIED layers
 * (ksg_clear_map) lists exactly the voxels of that delta map with their final state.  ksg_copy_update_log_device copies the last frame's
 * log (n entries of ksg_voxel_update + n * num_labels floats) into caller-owned device buffers - the payload of an ncclAllGather; both
 * destinations NULL = size query.  ksg_merge_voxels_device merges n_deltas (<= 16) such logs, delta g at entry offset g * stride with
 * counts[g] valid entries (counts on the host), into this map in delta order with the arithmetic of ksg_merge_blocks_device: the two
 * give identical maps (tests/test_gpu_delta_merge.py).  One synchronisation per call. */
int32_t ksg_copy_update_log_device(ksg_integrator* h, int64_t* n, void* d_dst_updates, void* d_dst_priors, int64_t capacity_entries, void* stream);
int32_t ksg_merge_voxels_device(ksg_integrator* h, int32_t n_deltas, const int64_t* counts, int64_t stride_entries, const void* d_updates,
                                const void* d_priors, void* stream);

/* Indices (nb*3 int32, sorted as above) of the blocks updated by the most recent integrate call:
 * the blocks whose updated() flag the reference sets (base.cpp:248). Returns the count. */
int64_t ksg_last_updated_blocks(ksg_integrator* h, int64_t capacity_blocks, int32_t* block_index);

/* Ground-truth label accuracy of the map against an analytic world (SURVEY.md 8f NEXT-4), computed on the device.  The ground truth
 * follows SemanticSimulationWorld::generateSemanticSdfFromWorld (kimera_semantics/src/simulation/semantic_simulation_world.cpp:35-97): the
 * label of a voxel is the label of the world object closest to its centre (voxblox simulation objects; distances below max_dist only).
 * Evaluated over the voxels with weight > 0 and |distance| <= band.  checker_size > 0 selects the labelling of the synthetic benchmark
 * scene instead: label = 1 + ((floor(x/s) + floor(y/s) + floor(z/s) + object label) mod (num_labels - 1)), leaving out voxels closer than
 * checker_margin to a checker boundary.  Outputs: voxels evaluated, voxels whose stored label equals the ground truth, observed voxels. */
typedef struct ksg_world_object {
  int32_t type;      /* 0 sphere: a = centre, b[0] = radius;  1 plane: a = point, b = normal;  2 axis-aligned cube: a = centre, b = size */
  float a[3], b[3];
  int32_t label;
} ksg_world_object;
int32_t ksg_evaluate_labels(ksg_integrator* h, const ksg_world_object* objects, int32_t n_objects, float max_dist, float band,
                            float checker_size, float checker_margin, int64_t* evaluated, int64_t* correct, int64_t* observed);

/* Semantic mesh of the map (SURVEY.md 8f NEXT-4), extracted on the device: marching cubes over the TSDF, every vertex carrying
 * TsdfVoxel.color (which the semantic integrators overwrite with the label colour, semantic_integrator_base.cpp:172-191 - the mesh the
 * reference displays, launch/kimera_semantics.launch:130-132) and the semantic label of the voxel that contains it.  Restates voxblox's
 * MeshIntegrator / MarchingCubes (not under the reference tree: unpinned; csrc/ksg_mesh.cuh lists the conventions and the two deliberate
 * differences).  min_weight: voxels with weight <= min_weight are unobserved (voxblox default 1e-4).  Triangles are 3 consecutive vertices.
 * Blocks are listed in (z, y, x) order like ksg_export_blocks; block_first_vertex (block_capacity + 1 entries) holds the first vertex of
 * every block and, last, the total.  A call with vertices = rgba = labels = NULL only counts (n_vertices, n_blocks, block tables);
 * KSG_ERR_INVALID_ARGUMENT if a capacity is too small (n_vertices / n_blocks still report the need). */
int32_t ksg_extract_mesh(ksg_integrator* h, float min_weight, int64_t vertex_capacity, float* vertices /* 3 per vertex */,
                         uint8_t* rgba /* 4 per vertex */, uint8_t* labels /* 1 per vertex */, int64_t block_capacity,
                         int32_t* block_index /* 3 per block */, int64_t* block_first_vertex, int64_t* n_vertices, int64_t* n_blocks);

/* Remove every block but keep the integrator: what Layer::removeAllBlocks() on both layers does to a live reference integrator.  The
 * fast integrator's two per-scan approximate sets (members of the integrator, fast.h:114-130) keep their contents and offsets, so the
 * next frame is integrated exactly as the reference integrator object would integrate it into its emptied layers.  Used by the
 * frame-per-GPU batch mode (the per-GPU "delta" map is emptied between batches; DESIGN.md 8). */
int32_t ksg_clear_map(ksg_integrator* h);

/* Remove every block and reset the fast integrator's two approximate sets. */
int32_t ksg_reset(ksg_integrator* h);

/* Spatial sharding helper (pure function, no device): mask[b*V + lin] = 1 where rank `shard_rank` of `shard_count` owns voxel
 * `lin` (voxblox linear order) of block b.  The masks of all ranks partition every block; a caller assembles the full map
 * from the per-rank exports with them. */
int32_t ksg_owner_mask(int32_t voxels_per_side, int32_t shard_rank, int32_t shard_count, int64_t n,
                       const int32_t* block_index, uint8_t* mask);

/* Host-only helper behind KSG_BUNDLE_ORDER_LIBSTDCXX (no device needed): bucket_count() of a std::unordered_map after each of
 * n successive insertions of distinct keys into an empty map, probed from the C++ runtime this library is linked with.
 * Writes n values; returns n, or -1 for bad arguments. */
int64_t ksg_unordered_map_schedule(int64_t n, int64_t* bucket_count_after_insert);

/* Optional per-phase device timing (CUDA events on the launching stream) and kernel-launch counting.
 * Phases: 0 classify+start-set, 1 observed-set fixpoint (fast) / bundling (merged), 2 ray emit,
 * 3 record sort, 4 block alloc + tile heads, 5 tile apply, 6 whole frame.  ksg_get_profile returns the
 * accumulated milliseconds per phase since the last ksg_set_profiling call and the number of frames. */
#define KSG_NUM_PHASES 7
int32_t ksg_set_profiling(ksg_integrator* h, int32_t enable);
int32_t ksg_get_profile(ksg_integrator* h, double* phase_ms /* KSG_NUM_PHASES */, int64_t* frames,
                        int64_t* kernel_launches /* own kernels */, int64_t* library_calls /* CUB sort/select calls */);

/* Debug aid: enable = 1 makes the tile kernel record (records, SM cycles) per processed tile; the call returns the
 * number of tiles of the last frame and copies 2 int64 per tile when records_and_cycles has room. */
int64_t ksg_debug_tile_times(ksg_integrator* h, int32_t enable, int64_t capacity, int64_t* records_and_cycles);

/* Debug aid (fast integrator, profiling enabled): SM-clock stamps that block 0 of the frame's persistent solve kernel took at its phase
 * boundaries during the LAST frame: out[0] kernel start, out[1] rays compacted, out[2] rays set up, out[3 .. 2+sweeps] end of each
 * observed-set sweep, out[52] sweeps done, out[53] table commit + ray emit done, out[54] records counted per tile, out[55] tile
 * segments allocated + new blocks constructed, out[56] records scattered (kernel end); out[64..79]: maxima / counts gathered inside the
 * kernel (longest single ray set-up / evaluation in clocks, rays evaluated, blocks evaluated / materialised, ...); *sweeps = sweeps of that
 * frame, *clock_khz = SM clock the stamps count in.  Returns the number of slots written (80) or 0. */
int64_t ksg_debug_fast_timeline(ksg_integrator* h, int64_t* out112 /* 64 time marks + 16 debug maxima / counts + 32 solver counters */, int64_t* sweeps, double* clock_khz);

/* Debug aid for the next optimisation (not on the integration path): evaluates  s <- fl(s + terms[k]), k = 0..n-1  (s0 < 0, terms <= 0,
 * float32, round to nearest even) with ONE warp as an exact associative scan (lanes = records, csrc/ksg_chain.cuh) and returns the
 * final s, which must equal the sequential loop bit for bit.  This is the per-voxel, per-class log-probability recurrence of the
 * `merged` integrator (base.cpp:306-307).  Host buffers. */
int32_t ksg_debug_chain_sum(const float* terms, int64_t n, float s0, float* result);

/* Build information: "sm_100a" etc. */
const char* ksg_build_info(void);

#ifdef __cplusplus
}
#endif
#endif /* KSG_H_ */
